// Classification head: mean over spectral blocks -> LN(D) -> Linear(D -> nc*p1*p1) -> 'b h w (p1 p2 nc) -> b nc (h p1)(w p2)'
// (reference src/vit_spatial_spectral.py:550-562 and :481-493), forward + backward, and the finetune loss
// nn.CrossEntropyLoss(ignore_index=-1) (finetune.py:136, src/utils.py:646) as one fused fwd+bwd kernel.
// One warp per (sample, spatial position); D/32 features per lane.
#include "common.cuh"

namespace msst {

constexpr int HT = 256;

struct HeadGeom { int B, C, G, p1, D, nc, S, T, NO, Wout; };

template <int NJ>
__device__ __forceinline__ void pool_ln(const HeadGeom& g, const float* __restrict__ x, int b, int s, int lane,
                                        const float (&lw)[NJ], const float (&lb)[NJ], float (&zh)[NJ], float (&zl)[NJ], float& rstd) {
    float z[NJ];
#pragma unroll
    for (int j = 0; j < NJ; ++j) z[j] = 0.f;
    for (int c = 0; c < g.C; ++c) {
        const float* p = x + ((int64_t)b * g.T + (int64_t)c * g.S + s) * g.D;
#pragma unroll
        for (int j = 0; j < NJ; ++j) z[j] += p[lane + 32 * j];
    }
    float sum = 0.f;
#pragma unroll
    for (int j = 0; j < NJ; ++j) { z[j] /= g.C; sum += z[j]; }
    const float mean = warp_sum(sum) / g.D;
    float sq = 0.f;
#pragma unroll
    for (int j = 0; j < NJ; ++j) { z[j] -= mean; sq += z[j] * z[j]; }
    rstd = rsqrtf(warp_sum(sq) / g.D + 1e-5f);
#pragma unroll
    for (int j = 0; j < NJ; ++j) { zh[j] = z[j] * rstd; zl[j] = zh[j] * lw[j] + lb[j]; }
}

__device__ __forceinline__ int64_t logit_index(const HeadGeom& g, int b, int s, int o) {
    // linear output o = (pi*p1 + pj)*nc + n  ->  logits[b, n, h*p1+pi, w*p1+pj]
    const int n = o % g.nc, pp = o / g.nc, pi = pp / g.p1, pj = pp % g.p1, h = s / g.G, w = s % g.G;
    return (((int64_t)b * g.nc + n) * g.Wout + (h * g.p1 + pi)) * g.Wout + (w * g.p1 + pj);
}

template <int NJ>
__global__ void __launch_bounds__(HT) head_fwd_kernel(HeadGeom g, const float* __restrict__ x, const float* __restrict__ ln_w,
                                                      const float* __restrict__ ln_b, const float* __restrict__ W,
                                                      const float* __restrict__ bias, float* __restrict__ logits) {
    extern __shared__ float Ws[];   // [NO][D]
    for (int i = threadIdx.x; i < g.NO * g.D; i += HT) Ws[i] = W[i];
    __syncthreads();
    const int lane = threadIdx.x & 31;
    float lw[NJ], lb[NJ];
#pragma unroll
    for (int j = 0; j < NJ; ++j) { lw[j] = ln_w[lane + 32 * j]; lb[j] = ln_b[lane + 32 * j]; }
    const int64_t total = (int64_t)g.B * g.S;
    for (int64_t it = (int64_t)blockIdx.x * (HT / 32) + (threadIdx.x >> 5); it < total; it += (int64_t)gridDim.x * (HT / 32)) {
        const int b = (int)(it / g.S), s = (int)(it % g.S);
        float zh[NJ], zl[NJ], rstd;
        pool_ln<NJ>(g, x, b, s, lane, lw, lb, zh, zl, rstd);
        for (int o = 0; o < g.NO; ++o) {
            float a = 0.f;
#pragma unroll
            for (int j = 0; j < NJ; ++j) a = fmaf(zl[j], Ws[o * g.D + lane + 32 * j], a);
            a = warp_sum(a);
            if (lane == 0) logits[logit_index(g, b, s, o)] = a + bias[o];
        }
    }
}

template <int NJ>
__global__ void __launch_bounds__(HT) head_bwd_kernel(HeadGeom g, const float* __restrict__ x, const float* __restrict__ ln_w,
                                                      const float* __restrict__ ln_b, const float* __restrict__ W,
                                                      const float* __restrict__ d_logits, float* __restrict__ d_x,
                                                      float* __restrict__ d_ln_w, float* __restrict__ d_ln_b,
                                                      float* __restrict__ d_W, float* __restrict__ d_bias) {
    extern __shared__ float sm[];
    float* Ws = sm;                         // [NO][D]
    float* dWs = Ws + g.NO * g.D;           // [NO][D] accumulators
    float* dbs = dWs + g.NO * g.D;          // [NO]
    float* dl = dbs + g.NO;                 // [8 warps][NO]
    float* red = dl + 8 * g.NO;             // [2][8][D]
    for (int i = threadIdx.x; i < g.NO * g.D; i += HT) { Ws[i] = W[i]; dWs[i] = 0.f; }
    for (int i = threadIdx.x; i < g.NO; i += HT) dbs[i] = 0.f;
    __syncthreads();
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    float lw[NJ], lb[NJ], a_w[NJ], a_b[NJ];
#pragma unroll
    for (int j = 0; j < NJ; ++j) { lw[j] = ln_w[lane + 32 * j]; lb[j] = ln_b[lane + 32 * j]; a_w[j] = a_b[j] = 0.f; }
    const int64_t total = (int64_t)g.B * g.S;
    for (int64_t it = (int64_t)blockIdx.x * (HT / 32) + warp; it < total; it += (int64_t)gridDim.x * (HT / 32)) {
        const int b = (int)(it / g.S), s = (int)(it % g.S);
        float zh[NJ], zl[NJ], rstd;
        pool_ln<NJ>(g, x, b, s, lane, lw, lb, zh, zl, rstd);
        for (int o = lane; o < g.NO; o += 32) dl[warp * g.NO + o] = d_logits[logit_index(g, b, s, o)];
        __syncwarp();
        float dz[NJ];
#pragma unroll
        for (int j = 0; j < NJ; ++j) dz[j] = 0.f;
        for (int o = 0; o < g.NO; ++o) {
            const float dlo = dl[warp * g.NO + o];
            if (lane == 0) atomicAdd(dbs + o, dlo);
#pragma unroll
            for (int j = 0; j < NJ; ++j) {
                atomicAdd(dWs + o * g.D + lane + 32 * j, dlo * zl[j]);
                dz[j] = fmaf(dlo, Ws[o * g.D + lane + 32 * j], dz[j]);
            }
        }
        __syncwarp();
        float c1 = 0.f, c2 = 0.f, gj[NJ];
#pragma unroll
        for (int j = 0; j < NJ; ++j) {
            a_w[j] += dz[j] * zh[j]; a_b[j] += dz[j];
            gj[j] = dz[j] * lw[j];
            c1 += gj[j]; c2 += gj[j] * zh[j];
        }
        c1 = warp_sum(c1) / g.D; c2 = warp_sum(c2) / g.D;
        const float invC = 1.f / g.C;
#pragma unroll
        for (int j = 0; j < NJ; ++j) gj[j] = rstd * (gj[j] - c1 - zh[j] * c2) * invC;
        for (int c = 0; c < g.C; ++c) {
            float* p = d_x + ((int64_t)b * g.T + (int64_t)c * g.S + s) * g.D;
#pragma unroll
            for (int j = 0; j < NJ; ++j) p[lane + 32 * j] = gj[j];
        }
    }
#pragma unroll
    for (int j = 0; j < NJ; ++j) { red[warp * g.D + lane + 32 * j] = a_w[j]; red[(8 + warp) * g.D + lane + 32 * j] = a_b[j]; }
    __syncthreads();
    for (int f = threadIdx.x; f < g.D; f += HT) {
        float sw = 0.f, sb = 0.f;
        for (int k = 0; k < 8; ++k) { sw += red[k * g.D + f]; sb += red[(8 + k) * g.D + f]; }
        atomicAdd(d_ln_w + f, sw); atomicAdd(d_ln_b + f, sb);
    }
    for (int i = threadIdx.x; i < g.NO * g.D; i += HT) atomicAdd(d_W + i, dWs[i]);
    for (int i = threadIdx.x; i < g.NO; i += HT) atomicAdd(d_bias + i, dbs[i]);
}

// one thread per pixel; classes strided by HW (coalesced across the warp)
__global__ void ce_kernel(const float* __restrict__ logits, const int64_t* __restrict__ labels, int B, int nc, int HW,
                          int ignore_index, float* __restrict__ loss_sum_count, float* __restrict__ d_logits) {
    __shared__ float red[2][32];
    const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    float nll = 0.f, cnt = 0.f;
    if (i < (int64_t)B * HW) {
        const int b = (int)(i / HW), px = (int)(i % HW);
        const float* p = logits + (int64_t)b * nc * HW + px;
        const int64_t lab = labels[i];
        const bool valid = lab != ignore_index && lab >= 0 && lab < nc;
        float mx = -INFINITY;
        for (int c = 0; c < nc; ++c) mx = fmaxf(mx, p[(int64_t)c * HW]);
        float se = 0.f;
        for (int c = 0; c < nc; ++c) se += expf(p[(int64_t)c * HW] - mx);
        // log-sum-exp is kept relative to the max: with large logits (|x| ~ 1e4, fp32 spacing ~1e-3) rounding mx + log(se) to
        // fp32 would put an error of ~5e-4 into every probability that is not saturated
        const float lse_rel = logf(se);
        if (valid) { nll = (mx - p[lab * HW]) + lse_rel; cnt = 1.f; }
        if (d_logits) {
            float* dp = d_logits + (int64_t)b * nc * HW + px;
            for (int c = 0; c < nc; ++c)
                dp[(int64_t)c * HW] = valid ? expf((p[(int64_t)c * HW] - mx) - lse_rel) - (c == lab ? 1.f : 0.f) : 0.f;
        }
    }
    nll = warp_sum(nll); cnt = warp_sum(cnt);
    if ((threadIdx.x & 31) == 0) { red[0][threadIdx.x >> 5] = nll; red[1][threadIdx.x >> 5] = cnt; }
    __syncthreads();
    if (threadIdx.x < 32) {
        const int nw = blockDim.x >> 5;
        float a = threadIdx.x < nw ? red[0][threadIdx.x] : 0.f, c = threadIdx.x < nw ? red[1][threadIdx.x] : 0.f;
        a = warp_sum(a); c = warp_sum(c);
        if (threadIdx.x == 0) { atomicAdd(loss_sum_count, a); atomicAdd(loss_sum_count + 1, c); }
    }
}

static int make_geom(const msst_head_dims* d, HeadGeom& g) {
    MSST_REQUIRE(d && d->B > 0 && d->C > 0 && d->G > 0 && d->p1 > 0 && d->nc > 0, "head: bad dims");
    MSST_REQUIRE(d->D % 32 == 0 && d->D >= 32 && d->D <= 256, "head: D=%d must be a multiple of 32 in [32,256]", d->D);
    g.B = d->B; g.C = d->C; g.G = d->G; g.p1 = d->p1; g.D = d->D; g.nc = d->nc;
    g.S = d->G * d->G; g.T = g.C * g.S; g.NO = d->nc * d->p1 * d->p1; g.Wout = d->G * d->p1;
    MSST_REQUIRE((size_t)g.NO * g.D * 8 + 4096 * 4 < 200 * 1024, "head: num_classes*p1*p1*D too large for the fused head");
    return MSST_OK;
}

}  // namespace msst
using namespace msst;

extern "C" int msst_head_fwd(const msst_head_dims* d, const float* x, const float* ln_w, const float* ln_b, const float* W,
                             const float* bias, float* logits, msst_stream_t stream) {
    HeadGeom g;
    if (int rc = make_geom(d, g)) return rc;
    const size_t smem = sizeof(float) * (size_t)g.NO * g.D;
    int64_t grid = ceil_div((int64_t)g.B * g.S, HT / 32);
    if (grid > 8 * kNumSMs) grid = 8 * kNumSMs;
    cudaStream_t st = (cudaStream_t)stream;
#define MSST_H(NJ)                                                                                                    \
    case NJ:                                                                                                          \
        MSST_CUDA(cudaFuncSetAttribute(head_fwd_kernel<NJ>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem)); \
        head_fwd_kernel<NJ><<<(int)grid, HT, smem, st>>>(g, x, ln_w, ln_b, W, bias, logits);                           \
        break;
    switch (g.D / 32) { MSST_H(1) MSST_H(2) MSST_H(3) MSST_H(4) MSST_H(6) MSST_H(8) default: set_error("head: D unsupported"); return MSST_ERR_ARG; }
#undef MSST_H
    MSST_LAUNCH_CHECK();
    return MSST_OK;
}

extern "C" int msst_head_bwd(const msst_head_dims* d, const float* x, const float* ln_w, const float* ln_b, const float* W,
                             const float* d_logits, float* d_x, float* d_ln_w, float* d_ln_b, float* d_W, float* d_bias,
                             msst_stream_t stream) {
    HeadGeom g;
    if (int rc = make_geom(d, g)) return rc;
    const size_t smem = sizeof(float) * ((size_t)2 * g.NO * g.D + g.NO + 8 * g.NO + 16 * g.D);
    int64_t grid = ceil_div((int64_t)g.B * g.S, HT / 32);
    if (grid > kNumSMs) grid = kNumSMs;
    cudaStream_t st = (cudaStream_t)stream;
#define MSST_H(NJ)                                                                                                    \
    case NJ:                                                                                                          \
        MSST_CUDA(cudaFuncSetAttribute(head_bwd_kernel<NJ>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem)); \
        head_bwd_kernel<NJ><<<(int)grid, HT, smem, st>>>(g, x, ln_w, ln_b, W, d_logits, d_x, d_ln_w, d_ln_b, d_W, d_bias); \
        break;
    switch (g.D / 32) { MSST_H(1) MSST_H(2) MSST_H(3) MSST_H(4) MSST_H(6) MSST_H(8) default: set_error("head: D unsupported"); return MSST_ERR_ARG; }
#undef MSST_H
    MSST_LAUNCH_CHECK();
    return MSST_OK;
}

extern "C" int msst_cross_entropy_fwd_bwd(const float* logits, const int64_t* labels, int B, int nc, int HW, int ignore_index,
                                          float* loss_sum_count, float* d_logits, msst_stream_t stream) {
    MSST_REQUIRE(B > 0 && nc > 0 && HW > 0, "cross_entropy: bad dims");
    cudaStream_t st = (cudaStream_t)stream;
    MSST_CUDA(cudaMemsetAsync(loss_sum_count, 0, 2 * sizeof(float), st));
    const int64_t n = (int64_t)B * HW;
    ce_kernel<<<(int)ceil_div(n, 256), 256, 0, st>>>(logits, labels, B, nc, HW, ignore_index, loss_sum_count, d_logits);
    MSST_LAUNCH_CHECK();
    return MSST_OK;
}
