// Shared device/host helpers for the MaskedSST B200 kernels (sm_100a only).
#pragma once
#include <cuda_runtime.h>
#include <cuda_bf16.h>
#include <stdint.h>
#include <stdio.h>
#include <math.h>

#include "../../include/msst.h"

namespace msst {

// ---- error plumbing: no exception crosses the C boundary (SURVEY.md §8(b) "Errors") ----
void set_error(const char* fmt, ...);
inline int cuda_fail(cudaError_t e, const char* what, const char* file, int line) {
    set_error("%s failed at %s:%d: %s", what, file, line, cudaGetErrorString(e));
    return MSST_ERR_CUDA;
}
#define MSST_CUDA(call)                                                        \
    do {                                                                       \
        cudaError_t e__ = (call);                                              \
        if (e__ != cudaSuccess) return ::msst::cuda_fail(e__, #call, __FILE__, __LINE__); \
    } while (0)
void count_launch();
#define MSST_LAUNCH_CHECK() do { ::msst::count_launch(); MSST_CUDA(cudaPeekAtLastError()); } while (0)
#define MSST_REQUIRE(cond, ...)                                                \
    do {                                                                       \
        if (!(cond)) { ::msst::set_error(__VA_ARGS__); return MSST_ERR_ARG; }  \
    } while (0)

constexpr int kNumSMs = 148;  // B200: 2 dies x 74 SMs

// cudaFuncSetAttribute is per device: one-time setup guards are kept per device ordinal (one process may drive several GPUs)
struct PerDeviceOnce {
    unsigned long long done = 0ull;
    bool first() {
        int dev = 0;
        cudaGetDevice(&dev);
        const unsigned long long bit = 1ull << (dev & 63);
        if (done & bit) return false;
        done |= bit;
        return true;
    }
};

__host__ __device__ inline int64_t ceil_div(int64_t a, int64_t b) { return (a + b - 1) / b; }

// ---- warp helpers ----
__device__ __forceinline__ float warp_sum(float v) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
    return v;
}
__device__ __forceinline__ float warp_max(float v) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v = fmaxf(v, __shfl_xor_sync(0xffffffffu, v, o));
    return v;
}

// exact (erf) GELU and its derivative: nn.GELU() default, reference src/vit_spatial_spectral.py:37
__device__ __forceinline__ float gelu_erf(float x) { return 0.5f * x * (1.0f + erff(x * 0.70710678118654752440f)); }
__device__ __forceinline__ float gelu_erf_grad(float x) {
    const float cdf = 0.5f * (1.0f + erff(x * 0.70710678118654752440f));
    const float pdf = 0.39894228040143267794f * expf(-0.5f * x * x);
    return cdf + x * pdf;
}

// bf16-mode variants: erf by Abramowitz-Stegun 7.1.26 (|err| <= 1.5e-7, far below bf16 resolution), ~3x fewer instructions
__device__ __forceinline__ float erf_as(float x) {
    const float ax = fabsf(x);
    const float t = __fdividef(1.0f, fmaf(0.3275911f, ax, 1.0f));   // rcp.approx (1 ulp): far inside the formula's own 1.5e-7
    float p = fmaf(1.061405429f, t, -1.453152027f);
    p = fmaf(p, t, 1.421413741f); p = fmaf(p, t, -0.284496736f); p = fmaf(p, t, 0.254829592f);
    const float r = 1.0f - p * t * __expf(-ax * ax);
    return copysignf(r, x);
}
__device__ __forceinline__ float gelu_fast(float x) { return 0.5f * x * (1.0f + erf_as(x * 0.70710678118654752440f)); }
__device__ __forceinline__ float gelu_fast_grad(float x) {
    const float cdf = 0.5f * (1.0f + erf_as(x * 0.70710678118654752440f));
    return fmaf(x * 0.39894228040143267794f, __expf(-0.5f * x * x), cdf);
}

// same function with the work shared between the two terms: e = exp(-x^2/2) serves the erf tail AND the density, the 0.5 of the cdf is
// folded into the polynomial, and the sign is resolved by one select (~17 FP32 + 2 MUFU instead of ~30): the fused FeedForward backward
// (mlp_block_tc.cu) is issue-bound on this epilogue
__device__ __forceinline__ float gelu_fast_grad2(float x) {
    const float ax = fabsf(x);
    const float t = __fdividef(1.0f, fmaf(0.3275911f * 0.70710678118654752440f, ax, 1.0f));
    float p = fmaf(0.5f * 1.061405429f, t, 0.5f * -1.453152027f);
    p = fmaf(p, t, 0.5f * 1.421413741f); p = fmaf(p, t, 0.5f * -0.284496736f); p = fmaf(p, t, 0.5f * 0.254829592f);
    float e;
    asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(e) : "f"(x * x * -0.72134752044448170368f));   // exp(-x^2 / 2)
    const float q = p * t * e;                                   // 0.5 * erfc(|x| / sqrt 2)
    const float cdf = x >= 0.f ? 1.0f - q : q;
    return fmaf(x * 0.39894228040143267794f, e, cdf);
}

// ---- counter-based dropout RNG ----
// Masks are never stored: forward and backward regenerate them from (seed, site, element index).  One call yields 64 random
// bits = four 16-bit lanes for elements 4q..4q+3 of site `site`: the counter is folded to 32 bits and passed through the
// "lowbias32" integer finaliser (two multiply-xorshift rounds, full avalanche), the second word by one more chained round.
// (Round 1 used Philox4x32-7 here: ~19 instructions per element, which made the dropout-carrying GEMM / LayerNorm epilogues
// issue-bound; this is ~6.  Keep decision: lane >= thresh >> 16, i.e. p is resolved to 2^-16.)
__host__ __device__ inline uint32_t mix32(uint32_t x) {
    x ^= x >> 16; x *= 0x7feb352du; x ^= x >> 15; x *= 0x846ca68bu; x ^= x >> 16;
    return x;
}
__host__ __device__ inline void drop_bits64(uint64_t seed, uint32_t site, uint64_t quad, uint32_t& a, uint32_t& b) {
    const uint32_t x = ((uint32_t)quad + (uint32_t)(seed >> 32)) * 0x9E3779B1u ^ ((uint32_t)(quad >> 32) * 0x85EBCA77u) ^ (uint32_t)seed ^
                       (site * 0xC2B2AE3Du);
    a = mix32(x);
    b = mix32(a + 0x9E3779B9u);
}

// Inverted-dropout descriptor. keep element iff rand16 >= thresh >> 16, thresh = p * 2^32.
struct Drop {
    uint64_t seed;
    const uint64_t* seed_dev;   // optional device-resident seed offset (lets a captured CUDA graph draw fresh masks per replay)
    uint32_t site;
    uint32_t thresh;   // 0 => dropout disabled
    float scale;       // 1/(1-p); 0 for p = 1 (a lane of 0xFFFF still passes the compare, and must yield 0, not inf)
    __host__ __device__ bool on() const { return thresh != 0u; }
};
// p must lie in [0, 1] (nn.Dropout's range; NaN fails): every entry point that takes a dropout probability checks it first
inline bool drop_p_ok(float p) { return p >= 0.f && p <= 1.f; }
inline Drop make_drop(float p, uint64_t seed, uint32_t site, const uint64_t* seed_dev = nullptr) {
    Drop d; d.seed = seed; d.site = site; d.seed_dev = seed_dev;
    if (p <= 0.f) { d.thresh = 0u; d.scale = 1.f; }
    else {
        double t = (double)p * 4294967296.0;
        d.thresh = t >= 4294967295.0 ? 4294967295u : (uint32_t)t;
        if (d.thresh == 0u) d.thresh = 1u;
        d.scale = p >= 1.f ? 0.f : 1.f / (1.f - p);
    }
    return d;
}
// factor (0 or scale) for a single element index e of the site
__device__ __forceinline__ float drop_factor(const Drop& d, uint64_t e) {
    uint32_t a, b;
    drop_bits64(d.seed + (d.seed_dev ? __ldg(d.seed_dev) : 0ull), d.site, e >> 2, a, b);
    const uint32_t w = (e & 2) ? b : a;
    return (((e & 1) ? (w >> 16) : (w & 0xFFFFu)) >= (d.thresh >> 16)) ? d.scale : 0.f;
}
// factors for the aligned quad 4q..4q+3
__device__ __forceinline__ void drop_factor4(const Drop& d, uint64_t quad, float (&f)[4]) {
    uint32_t a, b;
    drop_bits64(d.seed + (d.seed_dev ? __ldg(d.seed_dev) : 0ull), d.site, quad, a, b);
    const uint32_t t16 = d.thresh >> 16;
    f[0] = (a & 0xFFFFu) >= t16 ? d.scale : 0.f; f[1] = (a >> 16) >= t16 ? d.scale : 0.f;
    f[2] = (b & 0xFFFFu) >= t16 ? d.scale : 0.f; f[3] = (b >> 16) >= t16 ? d.scale : 0.f;
}

// dropout site ids (distinct RNG streams); per transformer layer: site = base + layer*8 + k
enum DropSite : uint32_t { kSiteEmb = 1, kSiteLayerBase = 16, kSiteAttnProb = 0, kSiteAttnOut = 1, kSiteMlpHidden = 2, kSiteMlpOut = 3 };

}  // namespace msst
