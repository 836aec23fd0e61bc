// Kernel (4a): warp-shuffle LayerNorm forward/backward (nn.LayerNorm semantics: biased variance, eps in sqrt).
// Reference: PreNorm, src/vit_spatial_spectral.py:22-29 (16 calls per forward).  HBM-bound:
// fwd reads rows*D*4 B and writes rows*D*(4|2) B; one warp per row, D/32 values per lane in registers.
#include "common.cuh"
#include "kernels.h"

namespace msst {

constexpr int kLnThreads = 256;

constexpr int kLnRows = 4;   // rows per warp per iteration: 4 x NJ independent loads in flight hide the DRAM latency

template <int NJ, bool BF16>
__global__ void __launch_bounds__(kLnThreads)
ln_fwd_kernel(const float* __restrict__ x, const float* __restrict__ w, const float* __restrict__ b, void* __restrict__ y,
              float* __restrict__ stats, int64_t rows, int D, float eps) {
    const int lane = threadIdx.x & 31;
    const int64_t warp0 = (int64_t)blockIdx.x * (kLnThreads / 32) + (threadIdx.x >> 5);
    const int64_t nwarps = (int64_t)gridDim.x * (kLnThreads / 32);
    float wj[NJ], bj[NJ];
#pragma unroll
    for (int j = 0; j < NJ; ++j) { const int f = lane + 32 * j; wj[j] = f < D ? w[f] : 0.f; bj[j] = f < D ? b[f] : 0.f; }
    for (int64_t r0 = warp0 * kLnRows; r0 < rows; r0 += nwarps * kLnRows) {
        float v[kLnRows][NJ];
#pragma unroll
        for (int k = 0; k < kLnRows; ++k)
#pragma unroll
            for (int j = 0; j < NJ; ++j) { const int f = lane + 32 * j; v[k][j] = (r0 + k < rows && f < D) ? x[(r0 + k) * D + f] : 0.f; }
#pragma unroll
        for (int k = 0; k < kLnRows; ++k) {
            const int64_t r = r0 + k;
            if (r >= rows) break;
            float s = 0.f;
#pragma unroll
            for (int j = 0; j < NJ; ++j) s += v[k][j];
            const float mean = warp_sum(s) / D;
            float sq = 0.f;
#pragma unroll
            for (int j = 0; j < NJ; ++j) { const int f = lane + 32 * j; const float dl = f < D ? v[k][j] - mean : 0.f; sq += dl * dl; }
            const float rstd = rsqrtf(warp_sum(sq) / D + eps);
            if (stats && lane == 0) { stats[2 * r] = mean; stats[2 * r + 1] = rstd; }
#pragma unroll
            for (int j = 0; j < NJ; ++j) {
                const int f = lane + 32 * j;
                if (f < D) {
                    const float o = (v[k][j] - mean) * rstd * wj[j] + bj[j];
                    if (BF16) reinterpret_cast<__nv_bfloat16*>(y)[r * D + f] = __float2bfloat16(o);
                    else reinterpret_cast<float*>(y)[r * D + f] = o;
                }
            }
        }
    }
}

// dx = dx_add + rstd * (dy*w - mean(dy*w) - xhat * mean(dy*w*xhat)); dw += sum dy*xhat; db += sum dy
template <int NJ>
__global__ void __launch_bounds__(kLnThreads)
ln_bwd_kernel(const float* __restrict__ x, const float* __restrict__ w, const float* __restrict__ stats,
              const float* __restrict__ dy, const float* __restrict__ dx_add, float* __restrict__ dx,
              float* __restrict__ dw, float* __restrict__ db, int64_t rows, int D) {
    __shared__ float red[2][kLnThreads / 32][NJ * 32];
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const int64_t warp0 = (int64_t)blockIdx.x * (kLnThreads / 32) + warp;
    const int64_t nwarps = (int64_t)gridDim.x * (kLnThreads / 32);
    float wj[NJ], aw[NJ], ab[NJ];
#pragma unroll
    for (int j = 0; j < NJ; ++j) { const int f = lane + 32 * j; wj[j] = f < D ? w[f] : 0.f; aw[j] = ab[j] = 0.f; }
    for (int64_t r0 = warp0 * kLnRows; r0 < rows; r0 += nwarps * kLnRows) {
        float xv[kLnRows][NJ], dv[kLnRows][NJ], av[kLnRows][NJ], mean[kLnRows], rstd[kLnRows];
#pragma unroll
        for (int k = 0; k < kLnRows; ++k) {
            const bool ok = r0 + k < rows;
            mean[k] = ok ? stats[2 * (r0 + k)] : 0.f; rstd[k] = ok ? stats[2 * (r0 + k) + 1] : 0.f;
#pragma unroll
            for (int j = 0; j < NJ; ++j) {
                const int f = lane + 32 * j;
                const bool in = ok && f < D;
                const int64_t o = (r0 + k) * D + f;
                xv[k][j] = in ? x[o] : 0.f; dv[k][j] = in ? dy[o] : 0.f; av[k][j] = (in && dx_add) ? dx_add[o] : 0.f;
            }
        }
#pragma unroll
        for (int k = 0; k < kLnRows; ++k) {
            const int64_t r = r0 + k;
            if (r >= rows) break;
            float xh[NJ], g[NJ], c1 = 0.f, c2 = 0.f;
#pragma unroll
            for (int j = 0; j < NJ; ++j) {
                const int f = lane + 32 * j;
                xh[j] = f < D ? (xv[k][j] - mean[k]) * rstd[k] : 0.f;
                aw[j] += dv[k][j] * xh[j]; ab[j] += dv[k][j];
                g[j] = dv[k][j] * wj[j];
                c1 += g[j]; c2 += g[j] * xh[j];
            }
            c1 = warp_sum(c1) / D; c2 = warp_sum(c2) / D;
#pragma unroll
            for (int j = 0; j < NJ; ++j) {
                const int f = lane + 32 * j;
                if (f < D) dx[r * D + f] = rstd[k] * (g[j] - c1 - xh[j] * c2) + av[k][j];
            }
        }
    }
#pragma unroll
    for (int j = 0; j < NJ; ++j) { red[0][warp][lane + 32 * j] = aw[j]; red[1][warp][lane + 32 * j] = ab[j]; }
    __syncthreads();
    for (int f = threadIdx.x; f < D; f += kLnThreads) {
        float sw = 0.f, sb = 0.f;
        for (int k = 0; k < kLnThreads / 32; ++k) { sw += red[0][k][f]; sb += red[1][k][f]; }
        atomicAdd(dw + f, sw);
        atomicAdd(db + f, sb);
    }
}

// ---- D % 4 == 0, D <= 128 (the model's D = 96): lane owns 4 consecutive columns (float4 loads/stores, 24 of 32 lanes active
// at D = 96).  The quad alignment lets the backward kernel also emit, for free, what the NEXT GEMMs need from the gradient
// stream: a bf16 copy with the consumer's output-dropout mask applied and its column sums (the bias gradient) --
// i.e. the separate cast_rows pass is fused away. ----
template <bool BF16>
__global__ void __launch_bounds__(kLnThreads)
ln_fwd4_kernel(const float* __restrict__ x, const float* __restrict__ w, const float* __restrict__ b, void* __restrict__ y,
               float* __restrict__ stats, int64_t rows, int D, float eps) {
    const int lane = threadIdx.x & 31, c = lane * 4;
    const bool act = c < D;
    const int64_t warp0 = (int64_t)blockIdx.x * (kLnThreads / 32) + (threadIdx.x >> 5);
    const int64_t nwarps = (int64_t)gridDim.x * (kLnThreads / 32);
    const float4 w4 = act ? *reinterpret_cast<const float4*>(w + c) : make_float4(0.f, 0.f, 0.f, 0.f);
    const float4 b4 = act ? *reinterpret_cast<const float4*>(b + c) : make_float4(0.f, 0.f, 0.f, 0.f);
    for (int64_t r0 = warp0 * kLnRows; r0 < rows; r0 += nwarps * kLnRows) {
        float4 v[kLnRows];
#pragma unroll
        for (int k = 0; k < kLnRows; ++k)
            v[k] = (act && r0 + k < rows) ? *reinterpret_cast<const float4*>(x + (r0 + k) * D + c) : make_float4(0.f, 0.f, 0.f, 0.f);
#pragma unroll
        for (int k = 0; k < kLnRows; ++k) {
            const int64_t r = r0 + k;
            if (r >= rows) break;
            const float mean = warp_sum(v[k].x + v[k].y + v[k].z + v[k].w) / D;
            const float d0 = v[k].x - mean, d1 = v[k].y - mean, d2 = v[k].z - mean, d3 = v[k].w - mean;
            const float rstd = rsqrtf(warp_sum(act ? d0 * d0 + d1 * d1 + d2 * d2 + d3 * d3 : 0.f) / D + eps);
            if (stats && lane == 0) { stats[2 * r] = mean; stats[2 * r + 1] = rstd; }
            if (act) {
                const float o0 = d0 * rstd * w4.x + b4.x, o1 = d1 * rstd * w4.y + b4.y, o2 = d2 * rstd * w4.z + b4.z, o3 = d3 * rstd * w4.w + b4.w;
                if (BF16) {
                    __nv_bfloat162 lo = __floats2bfloat162_rn(o0, o1), hi = __floats2bfloat162_rn(o2, o3);
                    uint2 t; t.x = *reinterpret_cast<uint32_t*>(&lo); t.y = *reinterpret_cast<uint32_t*>(&hi);
                    *reinterpret_cast<uint2*>(reinterpret_cast<__nv_bfloat16*>(y) + r * D + c) = t;
                } else {
                    *reinterpret_cast<float4*>(reinterpret_cast<float*>(y) + r * D + c) = make_float4(o0, o1, o2, o3);
                }
            }
        }
    }
}

__global__ void __launch_bounds__(kLnThreads)
ln_bwd4_kernel(const float* __restrict__ x, const float* __restrict__ w, const float* __restrict__ stats,
               const float* __restrict__ dy, const float* __restrict__ dx_add, float* __restrict__ dx,
               float* __restrict__ dw, float* __restrict__ db, int64_t rows, int D,
               __nv_bfloat16* __restrict__ cast_out, Drop cast_drop, float* __restrict__ cast_colsum) {
    __shared__ float red[3][kLnThreads / 32][128];
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5, c = lane * 4;
    const bool act = c < D;
    const int64_t warp0 = (int64_t)blockIdx.x * (kLnThreads / 32) + warp;
    const int64_t nwarps = (int64_t)gridDim.x * (kLnThreads / 32);
    const float4 w4 = act ? *reinterpret_cast<const float4*>(w + c) : make_float4(0.f, 0.f, 0.f, 0.f);
    float aw[4] = {0.f, 0.f, 0.f, 0.f}, ab[4] = {0.f, 0.f, 0.f, 0.f}, ac[4] = {0.f, 0.f, 0.f, 0.f};
    const float4 z4 = make_float4(0.f, 0.f, 0.f, 0.f);
    for (int64_t r0 = warp0 * kLnRows; r0 < rows; r0 += nwarps * kLnRows) {
        float4 xv[kLnRows], dv[kLnRows], av[kLnRows];
        float mean[kLnRows], rstd[kLnRows];
#pragma unroll
        for (int k = 0; k < kLnRows; ++k) {
            const bool ok = r0 + k < rows;
            mean[k] = ok ? stats[2 * (r0 + k)] : 0.f; rstd[k] = ok ? stats[2 * (r0 + k) + 1] : 0.f;
            const int64_t o = (r0 + k) * D + c;
            xv[k] = (ok && act) ? *reinterpret_cast<const float4*>(x + o) : z4;
            dv[k] = (ok && act) ? *reinterpret_cast<const float4*>(dy + o) : z4;
            av[k] = (ok && act && dx_add) ? *reinterpret_cast<const float4*>(dx_add + o) : z4;
        }
#pragma unroll
        for (int k = 0; k < kLnRows; ++k) {
            const int64_t r = r0 + k;
            if (r >= rows) break;
            const float xs[4] = {xv[k].x, xv[k].y, xv[k].z, xv[k].w}, ds[4] = {dv[k].x, dv[k].y, dv[k].z, dv[k].w};
            const float ws[4] = {w4.x, w4.y, w4.z, w4.w}, as[4] = {av[k].x, av[k].y, av[k].z, av[k].w};
            float xh[4], g[4], c1 = 0.f, c2 = 0.f;
#pragma unroll
            for (int t = 0; t < 4; ++t) {
                xh[t] = act ? (xs[t] - mean[k]) * rstd[k] : 0.f;
                aw[t] += ds[t] * xh[t]; ab[t] += ds[t];
                g[t] = ds[t] * ws[t];
                c1 += g[t]; c2 += g[t] * xh[t];
            }
            c1 = warp_sum(c1) / D; c2 = warp_sum(c2) / D;
            if (act) {
                float o[4];
#pragma unroll
                for (int t = 0; t < 4; ++t) o[t] = rstd[k] * (g[t] - c1 - xh[t] * c2) + as[t];
                const int64_t off = r * D + c;
                *reinterpret_cast<float4*>(dx + off) = make_float4(o[0], o[1], o[2], o[3]);
                if (cast_out) {
                    if (cast_drop.on()) {
                        float f[4];
                        drop_factor4(cast_drop, (uint64_t)off >> 2, f);
#pragma unroll
                        for (int t = 0; t < 4; ++t) o[t] *= f[t];
                    }
                    __nv_bfloat162 lo = __floats2bfloat162_rn(o[0], o[1]), hi = __floats2bfloat162_rn(o[2], o[3]);
                    uint2 t2; t2.x = *reinterpret_cast<uint32_t*>(&lo); t2.y = *reinterpret_cast<uint32_t*>(&hi);
                    *reinterpret_cast<uint2*>(cast_out + off) = t2;
#pragma unroll
                    for (int t = 0; t < 4; ++t) ac[t] += o[t];
                }
            }
        }
    }
    if (act) {
#pragma unroll
        for (int t = 0; t < 4; ++t) { red[0][warp][c + t] = aw[t]; red[1][warp][c + t] = ab[t]; red[2][warp][c + t] = ac[t]; }
    }
    __syncthreads();
    for (int f = threadIdx.x; f < D; f += kLnThreads) {
        float sw = 0.f, sb = 0.f, sc = 0.f;
        for (int k = 0; k < kLnThreads / 32; ++k) { sw += red[0][k][f]; sb += red[1][k][f]; sc += red[2][k][f]; }
        atomicAdd(dw + f, sw);
        atomicAdd(db + f, sb);
        if (cast_colsum) atomicAdd(cast_colsum + f, sc);
    }
}

// ---- generic row width (D > 256, e.g. the spectral-MLP head's LayerNorm(D*C)): lanes stride over the row, re-reading it
// from L1/L2 instead of caching it in registers ----
template <bool BF16>
__global__ void __launch_bounds__(kLnThreads)
ln_fwd_wide_kernel(const float* __restrict__ x, const float* __restrict__ w, const float* __restrict__ b, void* __restrict__ y,
                   float* __restrict__ stats, int64_t rows, int D, float eps) {
    const int lane = threadIdx.x & 31;
    const int64_t warp0 = (int64_t)blockIdx.x * (kLnThreads / 32) + (threadIdx.x >> 5);
    const int64_t nwarps = (int64_t)gridDim.x * (kLnThreads / 32);
    for (int64_t r = warp0; r < rows; r += nwarps) {
        const float* xr = x + r * D;
        float s = 0.f;
        for (int f = lane; f < D; f += 32) s += xr[f];
        const float mean = warp_sum(s) / D;
        float sq = 0.f;
        for (int f = lane; f < D; f += 32) { const float dl = xr[f] - mean; sq += dl * dl; }
        const float rstd = rsqrtf(warp_sum(sq) / D + eps);
        if (stats && lane == 0) { stats[2 * r] = mean; stats[2 * r + 1] = rstd; }
        for (int f = lane; f < D; f += 32) {
            const float o = (xr[f] - mean) * rstd * w[f] + b[f];
            if (BF16) reinterpret_cast<__nv_bfloat16*>(y)[r * D + f] = __float2bfloat16(o);
            else reinterpret_cast<float*>(y)[r * D + f] = o;
        }
    }
}

__global__ void __launch_bounds__(kLnThreads)
ln_bwd_wide_kernel(const float* __restrict__ x, const float* __restrict__ w, const float* __restrict__ stats,
                   const float* __restrict__ dy, const float* __restrict__ dx_add, float* __restrict__ dx,
                   float* __restrict__ dw, float* __restrict__ db, int64_t rows, int D) {
    const int lane = threadIdx.x & 31;
    const int64_t warp0 = (int64_t)blockIdx.x * (kLnThreads / 32) + (threadIdx.x >> 5);
    const int64_t nwarps = (int64_t)gridDim.x * (kLnThreads / 32);
    for (int64_t r = warp0; r < rows; r += nwarps) {
        const float mean = stats[2 * r], rstd = stats[2 * r + 1];
        const float* xr = x + r * D; const float* dr = dy + r * D;
        float c1 = 0.f, c2 = 0.f;
        for (int f = lane; f < D; f += 32) {
            const float xh = (xr[f] - mean) * rstd, g = dr[f] * w[f];
            c1 += g; c2 += g * xh;
            atomicAdd(dw + f, dr[f] * xh);     // wide rows are a rarely used head variant: plain atomics
            atomicAdd(db + f, dr[f]);
        }
        c1 = warp_sum(c1) / D; c2 = warp_sum(c2) / D;
        for (int f = lane; f < D; f += 32) {
            const float xh = (xr[f] - mean) * rstd;
            float o = rstd * (dr[f] * w[f] - c1 - xh * c2);
            if (dx_add) o += dx_add[r * D + f];
            dx[r * D + f] = o;
        }
    }
}

static inline int ln_grid(int64_t rows) {
    int64_t blocks = ceil_div(rows, (kLnThreads / 32) * kLnRows);
    const int64_t cap = (int64_t)kNumSMs * 8;   // 8 resident CTAs of 256 threads per SM
    return (int)(blocks < cap ? blocks : cap);
}

int layernorm_fwd(const float* x, const float* w, const float* b, void* y, int y_bf16, float* stats, int64_t rows, int D,
                  float eps, cudaStream_t st) {
    MSST_REQUIRE(D >= 1, "layernorm: D=%d out of range", D);
    if (rows == 0) return MSST_OK;
    const int nj = (D + 31) / 32, grid = ln_grid(rows);
    if (D % 4 == 0 && D <= 128 && (reinterpret_cast<uintptr_t>(x) & 15) == 0 && (reinterpret_cast<uintptr_t>(y) & 15) == 0 &&
        (reinterpret_cast<uintptr_t>(w) & 15) == 0 && (reinterpret_cast<uintptr_t>(b) & 15) == 0) {
        if (y_bf16) ln_fwd4_kernel<true><<<grid, kLnThreads, 0, st>>>(x, w, b, y, stats, rows, D, eps);
        else ln_fwd4_kernel<false><<<grid, kLnThreads, 0, st>>>(x, w, b, y, stats, rows, D, eps);
        MSST_LAUNCH_CHECK();
        return MSST_OK;
    }
    if (D > 256) {
        if (y_bf16) ln_fwd_wide_kernel<true><<<grid, kLnThreads, 0, st>>>(x, w, b, y, stats, rows, D, eps);
        else ln_fwd_wide_kernel<false><<<grid, kLnThreads, 0, st>>>(x, w, b, y, stats, rows, D, eps);
        MSST_LAUNCH_CHECK();
        return MSST_OK;
    }
#define MSST_LN(NJ)                                                                                            \
    if (nj <= NJ) {                                                                                            \
        if (y_bf16) ln_fwd_kernel<NJ, true><<<grid, kLnThreads, 0, st>>>(x, w, b, y, stats, rows, D, eps);      \
        else ln_fwd_kernel<NJ, false><<<grid, kLnThreads, 0, st>>>(x, w, b, y, stats, rows, D, eps);            \
        MSST_LAUNCH_CHECK();                                                                                   \
        return MSST_OK;                                                                                        \
    }
    MSST_LN(1) MSST_LN(2) MSST_LN(3) MSST_LN(4) MSST_LN(8)
#undef MSST_LN
    return MSST_ERR_ARG;
}

int layernorm_bwd(const float* x, const float* w, const float* stats, const float* dy, const float* dx_add, float* dx,
                  float* dw, float* db, int64_t rows, int D, cudaStream_t st, __nv_bfloat16* cast_out, Drop cast_drop,
                  float* cast_colsum) {
    MSST_REQUIRE(D >= 1, "layernorm: D=%d out of range", D);
    if (rows == 0) return MSST_OK;
    const int nj = (D + 31) / 32;
    auto al16 = [](const void* q) { return (reinterpret_cast<uintptr_t>(q) & 15) == 0; };
    if (D % 4 == 0 && D <= 128 && al16(x) && al16(w) && al16(dy) && al16(dx) && (!dx_add || al16(dx_add))) {
        ln_bwd4_kernel<<<ln_grid(rows), kLnThreads, 0, st>>>(x, w, stats, dy, dx_add, dx, dw, db, rows, D, cast_out, cast_drop, cast_colsum);
        MSST_LAUNCH_CHECK();
        return MSST_OK;
    }
    // Otherwise (D > 128 in the bf16 transformer stack) the cast is a second pass over dx: cast_rows draws the same dropout mask
    // (drop_factor4 of the element index / 4).  Its requirements are checked here, before anything is launched.
    MSST_REQUIRE(cast_out == nullptr || (D % 4 == 0 && D <= 4096 && al16(dx) && (reinterpret_cast<uintptr_t>(cast_out) & 7) == 0),
                 "layernorm_bwd: the bf16 cast of dx needs D %% 4 == 0, D <= 4096 and aligned rows");
    const int grid = ln_grid(rows);   // up to 8 CTAs/SM: the row loop is a dependent chain, memory-level parallelism comes from warps
    if (D > 256) ln_bwd_wide_kernel<<<grid, kLnThreads, 0, st>>>(x, w, stats, dy, dx_add, dx, dw, db, rows, D);
    else if (nj <= 1) ln_bwd_kernel<1><<<grid, kLnThreads, 0, st>>>(x, w, stats, dy, dx_add, dx, dw, db, rows, D);
    else if (nj <= 2) ln_bwd_kernel<2><<<grid, kLnThreads, 0, st>>>(x, w, stats, dy, dx_add, dx, dw, db, rows, D);
    else if (nj <= 3) ln_bwd_kernel<3><<<grid, kLnThreads, 0, st>>>(x, w, stats, dy, dx_add, dx, dw, db, rows, D);
    else if (nj <= 4) ln_bwd_kernel<4><<<grid, kLnThreads, 0, st>>>(x, w, stats, dy, dx_add, dx, dw, db, rows, D);
    else ln_bwd_kernel<8><<<grid, kLnThreads, 0, st>>>(x, w, stats, dy, dx_add, dx, dw, db, rows, D);
    MSST_LAUNCH_CHECK();
    if (cast_out) return cast_rows_f32(dx, cast_out, cast_colsum, rows, D, cast_drop, st);
    return MSST_OK;
}

}  // namespace msst

extern "C" int msst_layernorm_fwd(const float* x, const float* w, const float* b, void* y, int y_bf16, float* stats,
                                  int64_t rows, int D, float eps, msst_stream_t stream) {
    return msst::layernorm_fwd(x, w, b, y, y_bf16, stats, rows, D, eps, (cudaStream_t)stream);
}
extern "C" int msst_layernorm_bwd(const float* x, const float* w, const float* stats, const float* dy, const float* dx_add,
                                  float* dx, float* dw, float* db, int64_t rows, int D, msst_stream_t stream) {
    return msst::layernorm_bwd(x, w, stats, dy, dx_add, dx, dw, db, rows, D, (cudaStream_t)stream, nullptr, msst::make_drop(0.f, 0, 0), nullptr);
}
