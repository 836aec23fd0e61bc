// Kernel (1): fused gather + LN(P) + per-spectral-block Linear(P->D) + LN(D) + pos-embed add
// + SimMIM mask-token select + emb-dropout, forward and backward.
// Reference arithmetic: src/vit_spatial_spectral.py:197-229 (to_patch/embed), :522-530,
// src/vit_simmim_original.py:236-249,285.  HBM-bound: per token it reads P fp32 pixels and writes D fp32.
//
// Work decomposition: one CTA per (sample b, spectral block c, chunk of 64 spatial positions).  With
// spatial patch size 1 the chunk's pixels are P runs of 64 contiguous floats (256 B each) -> coalesced.
#include "common.cuh"
#include "pixel_source.cuh"

namespace msst {

constexpr int kTok = 64;       // tokens per CTA chunk
constexpr int kThreads = 256;  // 8 warps, 8 tokens each

struct EmbedGeom {
    int B, C, G, p0, p1, D, P, S, T, HW, Wimg, nb;
    PixelSource src;
};

__device__ __forceinline__ float load_pixel(const EmbedGeom& g, int b, int c, int s, int p) {
    // element p = (p0i, p1i, p2i) of the patch at spatial position s = (h, w) of spectral block c
    if (g.p1 == 1) return g.src.load(b, c * g.p0 + p, s / g.Wimg, s % g.Wimg);
    const int pp = g.p1 * g.p1;
    const int p0i = p / pp, r = p % pp, p1i = r / g.p1, p2i = r % g.p1;
    const int h = s / g.G, w = s % g.G;
    return g.src.load(b, c * g.p0 + p0i, h * g.p1 + p1i, w * g.p1 + p2i);
}

// loads the chunk's raw patches into xs[tok][P+1] and pre-normalises: xs <- xhat, hs <- xhat*w+b
__device__ __forceinline__ void load_and_prenorm(const EmbedGeom& g, int b, int c, int s0,
                                                 const float* __restrict__ pre_w, const float* __restrict__ pre_b,
                                                 float* xs, float* hs, float* rstd_s) {
    const int P = g.P, ld = P + 1;
    for (int i = threadIdx.x; i < kTok * P; i += kThreads) {
        const int tok = i % kTok, p = i / kTok;
        const int s = s0 + tok;
        xs[tok * ld + p] = s < g.S ? load_pixel(g, b, c, s, p) : 0.f;
    }
    __syncthreads();
    if (threadIdx.x < kTok) {
        const int tok = threadIdx.x;
        float mean = 0.f;
        for (int p = 0; p < P; ++p) mean += xs[tok * ld + p];
        mean /= P;
        float var = 0.f;
        for (int p = 0; p < P; ++p) { const float dlt = xs[tok * ld + p] - mean; var += dlt * dlt; }
        const float rstd = rsqrtf(var / P + 1e-5f);
        rstd_s[tok] = rstd;
        for (int p = 0; p < P; ++p) {
            const float xh = (xs[tok * ld + p] - mean) * rstd;
            xs[tok * ld + p] = xh;
            hs[tok * ld + p] = xh * pre_w[p] + pre_b[p];
        }
    }
    __syncthreads();
}

template <int NJ>
__global__ void __launch_bounds__(kThreads)
patch_embed_fwd_kernel(EmbedGeom g, int n_wb, const float* __restrict__ img, const float* __restrict__ pre_w,
                       const float* __restrict__ pre_b, const float* __restrict__ W, const float* __restrict__ bias,
                       const float* __restrict__ post_w, const float* __restrict__ post_b, const float* __restrict__ pos,
                       const uint8_t* __restrict__ mask, const float* __restrict__ mask_token, float* __restrict__ tokens,
                       float* __restrict__ patches_ln, Drop drop) {
    extern __shared__ float smem[];
    const int P = g.P, ld = P + 1, D = g.D;
    float* xs = smem;                    // [64][P+1]
    float* hs = xs + kTok * ld;          // [64][P+1]
    float* Ws = hs + kTok * ld;          // [D][P+1]
    float* rstd_s = Ws + D * ld;         // [64]
    const int chunks = (g.S + kTok - 1) / kTok;
    const int chunk = blockIdx.x % chunks, c = (blockIdx.x / chunks) % g.C, b = blockIdx.x / (chunks * g.C);
    const int s0 = chunk * kTok;
    const int wb = n_wb == 1 ? 0 : c;
    for (int i = threadIdx.x; i < D * P; i += kThreads) Ws[(i / P) * ld + (i % P)] = __ldg(W + (int64_t)wb * D * P + i);
    load_and_prenorm(g, b, c, s0, pre_w, pre_b, xs, hs, rstd_s);

    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    float bj[NJ], pw[NJ], pb[NJ], mt[NJ];
#pragma unroll
    for (int j = 0; j < NJ; ++j) {
        const int f = lane + 32 * j;
        bj[j] = bias[wb * D + f]; pw[j] = post_w[f]; pb[j] = post_b[f];
        mt[j] = mask_token ? mask_token[f] : 0.f;
    }
    for (int k = 0; k < kTok / 8; ++k) {
        const int tok = warp * (kTok / 8) + k, s = s0 + tok;
        if (s >= g.S) break;
        const int t = c * g.S + s;
        float y[NJ];
        float sum = 0.f;
#pragma unroll
        for (int j = 0; j < NJ; ++j) {
            const int f = lane + 32 * j;
            float acc = bj[j];
            for (int p = 0; p < P; ++p) acc = fmaf(Ws[f * ld + p], hs[tok * ld + p], acc);
            y[j] = acc; sum += acc;
        }
        const float mean = warp_sum(sum) / D;
        float sq = 0.f;
#pragma unroll
        for (int j = 0; j < NJ; ++j) { const float dlt = y[j] - mean; sq += dlt * dlt; }
        const float rstd = rsqrtf(warp_sum(sq) / D + 1e-5f);
        const bool masked = mask && mask[(int64_t)b * g.T + t];
        const int64_t row = (int64_t)b * g.T + t;
#pragma unroll
        for (int j = 0; j < NJ; ++j) {
            const int f = lane + 32 * j;
            float o = (y[j] - mean) * rstd * pw[j] + pb[j];
            if (masked) o = mt[j];
            o += pos[(int64_t)t * D + f];
            if (drop.on()) o *= drop_factor(drop, (uint64_t)row * D + f);
            tokens[row * D + f] = o;
        }
        if (patches_ln) for (int p = lane; p < P; p += 32) patches_ln[row * P + p] = hs[tok * ld + p];
    }
}

// Backward.  grid = (C * chunks, nb): CTA (c, chunk, z) loops over samples b = z, z+nb, ... so the token set
// it touches is fixed -> d_pos / parameter gradients accumulate in registers, one atomic flush at the end.
template <int NJ, int PMAX>
__global__ void __launch_bounds__(kThreads, 2)      // <= 128 registers: two CTAs per SM (three: spills, 381 vs 288 us) (the token loop is a chain of warp reductions: latency, not issue, bound)
patch_embed_bwd_kernel(EmbedGeom g, int n_wb, const float* __restrict__ img, const float* __restrict__ pre_w,
                       const float* __restrict__ pre_b, const float* __restrict__ W, const float* __restrict__ bias,
                       const float* __restrict__ post_w, const float* __restrict__ post_b, const uint8_t* __restrict__ mask,
                       const float* __restrict__ d_tokens, const float* __restrict__ d_patches_ln, float* __restrict__ d_pre_w,
                       float* __restrict__ d_pre_b, float* __restrict__ d_W, float* __restrict__ d_bias,
                       float* __restrict__ d_post_w, float* __restrict__ d_post_b, float* __restrict__ d_pos,
                       float* __restrict__ d_mask_token, Drop drop) {
    extern __shared__ float smem[];
    const int P = g.P, ld = P + 1, D = g.D;
    float* xs = smem;
    float* hs = xs + kTok * ld;
    float* Ws = hs + kTok * ld;
    float* rstd_s = Ws + D * ld;
    float* red = rstd_s + kTok;          // [8 warps][D] reduction scratch
    const int chunks = (g.S + kTok - 1) / kTok;
    const int chunk = blockIdx.x % chunks, c = blockIdx.x / chunks;
    const int s0 = chunk * kTok;
    const int wb = n_wb == 1 ? 0 : c;
    for (int i = threadIdx.x; i < D * P; i += kThreads) Ws[(i / P) * ld + (i % P)] = __ldg(W + (int64_t)wb * D * P + i);
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    constexpr int TPW = kTok / 8;

    float bj[NJ], pw[NJ];
    // a_G[f][p] = sum_tok dy[tok,f] * xhat[tok,p].  Everything downstream of dy is linear in it, so the per-token work stops here:
    //   dW[f,p]   = pre_w[p] * G[f,p] + pre_b[p] * dbias[f]            (h = xhat * pre_w + pre_b)
    //   dpre_w[p] = sum_f W[f,p] * G[f,p],   dpre_b[p] = sum_f W[f,p] * dbias[f]
    // are formed once per CTA at the flush (no dh = W^T dy GEMV + 10 warp reductions per token).  Only the PatchEmbed/SimMIM
    // target gradient d_patches_ln enters the pre-norm gradients directly: lane p accumulates it (a_plw / a_plb).
    float a_postw[NJ], a_postb[NJ], a_bias[NJ], a_mt[NJ], a_pos[TPW][NJ], a_G[NJ][PMAX];
    float a_plw = 0.f, a_plb = 0.f;
#pragma unroll
    for (int j = 0; j < NJ; ++j) {
        const int f = lane + 32 * j;
        bj[j] = bias[wb * D + f]; pw[j] = post_w[f];
        a_postw[j] = a_postb[j] = a_bias[j] = a_mt[j] = 0.f;
#pragma unroll
        for (int k = 0; k < TPW; ++k) a_pos[k][j] = 0.f;
#pragma unroll
        for (int p = 0; p < PMAX; ++p) a_G[j][p] = 0.f;
    }

    for (int b = blockIdx.y; b < g.B; b += gridDim.y) {
        // this warp's 8 token gradients + mask bytes are fetched up front: their DRAM latency overlaps the slab load / pre-norm
        float dt_all[TPW][NJ];
        bool masked_all[TPW];
#pragma unroll
        for (int k = 0; k < TPW; ++k) {
            const int s = s0 + warp * TPW + k;
            const int64_t row = (int64_t)b * g.T + c * g.S + s;
            masked_all[k] = s < g.S && mask && mask[row];
#pragma unroll
            for (int j = 0; j < NJ; ++j) dt_all[k][j] = s < g.S ? d_tokens[row * D + lane + 32 * j] : 0.f;
        }
        __syncthreads();
        load_and_prenorm(g, b, c, s0, pre_w, pre_b, xs, hs, rstd_s);
#pragma unroll
        for (int k = 0; k < TPW; ++k) {
            const int tok = warp * TPW + k, s = s0 + tok;
            if (s >= g.S) continue;
            const int t = c * g.S + s;
            const int64_t row = (int64_t)b * g.T + t;
            float dt[NJ];
#pragma unroll
            for (int j = 0; j < NJ; ++j) {
                const int f = lane + 32 * j;
                dt[j] = dt_all[k][j];
                if (drop.on()) dt[j] *= drop_factor(drop, (uint64_t)row * D + f);
                a_pos[k][j] += dt[j];
            }
            const bool masked = masked_all[k];
            if (d_patches_ln && lane < P) {   // gradient that reaches the LayerNormed patches directly (PatchEmbed SimMIM target)
                const float dl = d_patches_ln[row * P + lane];
                a_plw = fmaf(dl, xs[tok * ld + lane], a_plw);
                a_plb += dl;
            }
            if (masked) {
#pragma unroll
                for (int j = 0; j < NJ; ++j) a_mt[j] += dt[j];
                continue;                                   // embedding path gets no token gradient
            }
            float y[NJ], sum = 0.f;
#pragma unroll
            for (int j = 0; j < NJ; ++j) {
                const int f = lane + 32 * j;
                float acc = bj[j];
                for (int p = 0; p < P; ++p) acc = fmaf(Ws[f * ld + p], hs[tok * ld + p], acc);
                y[j] = acc; sum += acc;
            }
            const float mean = warp_sum(sum) / D;
            float sq = 0.f;
#pragma unroll
            for (int j = 0; j < NJ; ++j) { y[j] -= mean; sq += y[j] * y[j]; }
            const float rstd = rsqrtf(warp_sum(sq) / D + 1e-5f);
            float c1 = 0.f, c2 = 0.f, dyh[NJ];
#pragma unroll
            for (int j = 0; j < NJ; ++j) {
                y[j] *= rstd;                         // yhat
                a_postw[j] += dt[j] * y[j];
                a_postb[j] += dt[j];
                dyh[j] = dt[j] * pw[j];
                c1 += dyh[j]; c2 += dyh[j] * y[j];
            }
            c1 = warp_sum(c1) / D; c2 = warp_sum(c2) / D;
            float dy[NJ];
#pragma unroll
            for (int j = 0; j < NJ; ++j) {
                dy[j] = rstd * (dyh[j] - c1 - y[j] * c2);
                a_bias[j] += dy[j];
            }
#pragma unroll
            for (int p = 0; p < PMAX; ++p) {
                if (p < P) {
                    const float xh = xs[tok * ld + p];
#pragma unroll
                    for (int j = 0; j < NJ; ++j) a_G[j][p] = fmaf(dy[j], xh, a_G[j][p]);
                }
            }
        }
    }
    // ---- flush: d_pos rows are owned by this warp (other CTAs along y add to the same rows) ----
#pragma unroll
    for (int k = 0; k < TPW; ++k) {
        const int s = s0 + warp * TPW + k;
        if (s < g.S) {
#pragma unroll
            for (int j = 0; j < NJ; ++j) atomicAdd(d_pos + (int64_t)(c * g.S + s) * D + lane + 32 * j, a_pos[k][j]);
        }
    }
    // cross-warp reduction of the per-feature accumulators through smem, then one atomic per value per CTA
    auto flush_feat = [&](float (&acc)[NJ], float* dst) {
        __syncthreads();
#pragma unroll
        for (int j = 0; j < NJ; ++j) red[warp * D + lane + 32 * j] = acc[j];
        __syncthreads();
        for (int f = threadIdx.x; f < D; f += kThreads) {
            float s = 0.f;
            for (int w = 0; w < 8; ++w) s += red[w * D + f];
            atomicAdd(dst + f, s);
        }
    };
    flush_feat(a_postw, d_post_w);
    flush_feat(a_postb, d_post_b);
    flush_feat(a_bias, d_bias + wb * D);
    if (d_mask_token) flush_feat(a_mt, d_mask_token);
    // dW, dpre_w, dpre_b from G and dbias (see the accumulator comment); per column p: cross-warp sum of G[:,p] and dbias, then
    // each feature thread adds its dW entry and its term of the two pre-norm sums (block-reduced, one atomic per CTA and p)
    float prew_part[PMAX], preb_part[PMAX];
#pragma unroll
    for (int p = 0; p < PMAX; ++p) prew_part[p] = preb_part[p] = 0.f;
    __syncthreads();
#pragma unroll
    for (int j = 0; j < NJ; ++j) red[warp * D + lane + 32 * j] = a_bias[j];
    __syncthreads();
    float dbias_f = 0.f;     // CTA-wide dbias of feature f = threadIdx.x (threads >= D idle)
    if (threadIdx.x < D) for (int w = 0; w < 8; ++w) dbias_f += red[w * D + threadIdx.x];
#pragma unroll
    for (int p = 0; p < PMAX; ++p) {
        if (p < P) {
            __syncthreads();
#pragma unroll
            for (int j = 0; j < NJ; ++j) red[warp * D + lane + 32 * j] = a_G[j][p];
            __syncthreads();
            if (threadIdx.x < D) {
                const int f = threadIdx.x;
                float G = 0.f;
                for (int w = 0; w < 8; ++w) G += red[w * D + f];
                atomicAdd(d_W + ((int64_t)wb * D + f) * P + p, fmaf(pre_w[p], G, pre_b[p] * dbias_f));
                const float wfp = Ws[f * ld + p];
                prew_part[p] = wfp * G;
                preb_part[p] = wfp * dbias_f;
            }
        }
    }
    // block-reduce the per-feature terms (D <= 128 <= kThreads features live in threads 0..D-1) + the direct d_patches_ln part
#pragma unroll
    for (int p = 0; p < PMAX; ++p) {
        if (p < P) {
            float sw = warp_sum(prew_part[p]), sb = warp_sum(preb_part[p]);
            __syncthreads();
            if (lane == 0) { red[warp] = sw; red[8 + warp] = sb; }
            __syncthreads();
            if (threadIdx.x == 0) {
                float tw = 0.f, tb = 0.f;
                for (int w = 0; w < 8; ++w) { tw += red[w]; tb += red[8 + w]; }
                atomicAdd(d_pre_w + p, tw);
                atomicAdd(d_pre_b + p, tb);
            }
        }
    }
    if (d_patches_ln && lane < P) { atomicAdd(d_pre_w + lane, a_plw); atomicAdd(d_pre_b + lane, a_plb); }
}

static int make_geom(const msst_embed_dims* d, const float* img, EmbedGeom& g) {
    MSST_REQUIRE(d && d->B > 0 && d->C > 0 && d->G > 0 && d->p0 > 0 && d->p1 > 0, "patch_embed: bad dims");
    MSST_REQUIRE(d->D % 32 == 0 && d->D >= 32 && d->D <= 256, "patch_embed: D=%d must be a multiple of 32 in [32,256]", d->D);
    MSST_REQUIRE(d->n_weight_blocks == 1 || d->n_weight_blocks == d->C, "patch_embed: n_weight_blocks must be 1 or C");
    MSST_REQUIRE(drop_p_ok(d->drop_p), "patch_embed: drop_p=%g outside [0, 1]", (double)d->drop_p);
    g.B = d->B; g.C = d->C; g.G = d->G; g.p0 = d->p0; g.p1 = d->p1; g.D = d->D;
    g.P = d->p0 * d->p1 * d->p1; g.S = d->G * d->G; g.T = g.C * g.S;
    g.Wimg = d->G * d->p1; g.HW = g.Wimg * g.Wimg; g.nb = 1;
    MSST_REQUIRE(g.P <= 64, "patch_embed: pixels per patch %d > 64 unsupported", g.P);
    if (const char* e = make_pixel_source(g.src, img, d->raw, g.C * g.p0, g.Wimg, g.Wimg)) { set_error("patch_embed: %s", e); return MSST_ERR_ARG; }
    return MSST_OK;
}

template <int NJ>
static int launch_fwd(const EmbedGeom& g, int n_wb, size_t smem, cudaStream_t st, const float* img, const float* pre_w,
                      const float* pre_b, const float* W, const float* bias, const float* post_w, const float* post_b,
                      const float* pos, const uint8_t* mask, const float* mask_token, float* tokens, float* patches_ln, Drop drop) {
    const int chunks = (g.S + kTok - 1) / kTok;
    MSST_CUDA(cudaFuncSetAttribute(patch_embed_fwd_kernel<NJ>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    patch_embed_fwd_kernel<NJ><<<g.B * g.C * chunks, kThreads, smem, st>>>(g, n_wb, img, pre_w, pre_b, W, bias, post_w, post_b,
                                                                           pos, mask, mask_token, tokens, patches_ln, drop);
    MSST_LAUNCH_CHECK();
    return MSST_OK;
}

template <int NJ, int PMAX>
static int launch_bwd(const EmbedGeom& g, int n_wb, size_t smem, cudaStream_t st, const float* img, const float* pre_w,
                      const float* pre_b, const float* W, const float* bias, const float* post_w, const float* post_b,
                      const uint8_t* mask, const float* d_tokens, const float* d_pln, float* d_pre_w, float* d_pre_b,
                      float* d_W, float* d_bias, float* d_post_w, float* d_post_b, float* d_pos, float* d_mt, Drop drop) {
    const int chunks = (g.S + kTok - 1) / kTok;
    int nb = (int)((4 * kNumSMs) / ((int64_t)g.C * chunks));   // floor: at most two full waves of two CTAs per SM (no tail wave)
    nb = nb < 1 ? 1 : (nb > g.B ? g.B : nb);
    MSST_CUDA(cudaFuncSetAttribute(patch_embed_bwd_kernel<NJ, PMAX>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    patch_embed_bwd_kernel<NJ, PMAX><<<dim3(g.C * chunks, nb), kThreads, smem, st>>>(
        g, n_wb, img, pre_w, pre_b, W, bias, post_w, post_b, mask, d_tokens, d_pln, d_pre_w, d_pre_b, d_W, d_bias, d_post_w,
        d_post_b, d_pos, d_mt, drop);
    MSST_LAUNCH_CHECK();
    return MSST_OK;
}

}  // namespace msst

using namespace msst;

extern "C" int msst_patch_embed_fwd(const msst_embed_dims* d, const float* img, const float* pre_w, const float* pre_b,
                                    const float* W, const float* bias, const float* post_w, const float* post_b,
                                    const float* pos, const uint8_t* mask, const float* mask_token, float* tokens,
                                    float* patches_ln, msst_stream_t stream) {
    EmbedGeom g;
    if (int rc = make_geom(d, img, g)) return rc;
    MSST_REQUIRE(!mask || mask_token, "patch_embed: mask given without mask_token");
    const size_t smem = sizeof(float) * ((size_t)2 * kTok * (g.P + 1) + (size_t)g.D * (g.P + 1) + kTok);
    const Drop drop = make_drop(d->drop_p, d->seed, kSiteEmb, d->seed_dev);
    cudaStream_t st = (cudaStream_t)stream;
#define MSST_FWD(NJ) return launch_fwd<NJ>(g, d->n_weight_blocks, smem, st, img, pre_w, pre_b, W, bias, post_w, post_b, pos, mask, mask_token, tokens, patches_ln, drop)
    switch (g.D / 32) {
        case 1: MSST_FWD(1); case 2: MSST_FWD(2); case 3: MSST_FWD(3); case 4: MSST_FWD(4);
    }
#undef MSST_FWD
    set_error("patch_embed: D=%d unsupported (32,64,96,128)", g.D);
    return MSST_ERR_ARG;
}

extern "C" int msst_patch_embed_bwd(const msst_embed_dims* d, const float* img, const float* pre_w, const float* pre_b,
                                    const float* W, const float* bias, const float* post_w, const float* post_b,
                                    const uint8_t* mask, const float* d_tokens, const float* d_patches_ln, float* d_pre_w,
                                    float* d_pre_b, float* d_W, float* d_bias, float* d_post_w, float* d_post_b,
                                    float* d_pos, float* d_mask_token, msst_stream_t stream) {
    EmbedGeom g;
    if (int rc = make_geom(d, img, g)) return rc;
    MSST_REQUIRE(g.P <= 16, "patch_embed_bwd: pixels per patch %d > 16 unsupported in backward", g.P);
    const int pmax = g.P <= 10 ? 10 : 16;   // the per-lane G accumulators are [D/32][pmax] registers
    size_t red = (size_t)8 * g.D;
    if (red < (size_t)8 * 2 * pmax) red = (size_t)8 * 2 * pmax;
    const size_t smem = sizeof(float) * ((size_t)2 * kTok * (g.P + 1) + (size_t)g.D * (g.P + 1) + kTok + red);
    const Drop drop = make_drop(d->drop_p, d->seed, kSiteEmb, d->seed_dev);
    cudaStream_t st = (cudaStream_t)stream;
#define MSST_BWD(NJ, PM) return launch_bwd<NJ, PM>(g, d->n_weight_blocks, smem, st, img, pre_w, pre_b, W, bias, post_w, post_b, mask, d_tokens, d_patches_ln, d_pre_w, d_pre_b, d_W, d_bias, d_post_w, d_post_b, d_pos, d_mask_token, drop)
    if (pmax == 16) {
        switch (g.D / 32) {
            case 1: MSST_BWD(1, 16); case 2: MSST_BWD(2, 16); case 3: MSST_BWD(3, 16); case 4: MSST_BWD(4, 16);
        }
    } else {
        switch (g.D / 32) {
            case 1: MSST_BWD(1, 10); case 2: MSST_BWD(2, 10); case 3: MSST_BWD(3, 10); case 4: MSST_BWD(4, 10);
        }
    }
#undef MSST_BWD
    set_error("patch_embed_bwd: (D=%d, P=%d) unsupported", g.D, g.P);
    return MSST_ERR_ARG;
}
