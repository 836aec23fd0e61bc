// Kernel (5): fused Adam / AdamW over a flat fp32 arena segment, with the reference's elementwise gradient clamp
// (pretrain.py:71-73, SURVEY C9) and the data-parallel 1/world scale folded in, optionally emitting the bf16 copy
// of the updated weights that the tcgen05 GEMMs consume.  Update rules: torch.optim.AdamW / Adam as configured by
// src/utils.py:36-44 and finetune.py:133-135.  HBM-bound: 28 B/param (read g,p,m,v; write p,m,v) [+2 B bf16].
#include "adam.cuh"

namespace msst {

__global__ void __launch_bounds__(256) adam_kernel(AdamK a, float* __restrict__ p, const float* __restrict__ g, float* __restrict__ m,
                                                   float* __restrict__ v, __nv_bfloat16* __restrict__ bf, int64_t n, int vec) {
    const int64_t tid = (int64_t)blockIdx.x * blockDim.x + threadIdx.x, nth = (int64_t)gridDim.x * blockDim.x;
    if (a.step_dev) {   // graph-capturable mode: bias corrections from the device-resident step counter
        const float t = (float)__ldg(a.step_dev);
        a.inv_bc1 = 1.f / (-expm1f(t * log1pf(a.b1 - 1.f)));          // 1 - b^t without cancellation
        a.inv_sqrt_bc2 = rsqrtf(-expm1f(t * log1pf(a.b2 - 1.f)));
    }
    if (vec) {
        const int64_t n4 = n >> 2;
        for (int64_t q = tid; q < n4; q += nth) {
            float4 P = reinterpret_cast<float4*>(p)[q], M = reinterpret_cast<float4*>(m)[q], V = reinterpret_cast<float4*>(v)[q];
            const float4 G = reinterpret_cast<const float4*>(g)[q];
            adam_one(a, P.x, G.x, M.x, V.x); adam_one(a, P.y, G.y, M.y, V.y);
            adam_one(a, P.z, G.z, M.z, V.z); adam_one(a, P.w, G.w, M.w, V.w);
            reinterpret_cast<float4*>(p)[q] = P; reinterpret_cast<float4*>(m)[q] = M; reinterpret_cast<float4*>(v)[q] = V;
            if (bf) {
                __nv_bfloat162 lo = __floats2bfloat162_rn(P.x, P.y), hi = __floats2bfloat162_rn(P.z, P.w);
                reinterpret_cast<__nv_bfloat162*>(bf)[2 * q] = lo; reinterpret_cast<__nv_bfloat162*>(bf)[2 * q + 1] = hi;
            }
        }
        for (int64_t i = (n4 << 2) + tid; i < n; i += nth) {
            float P = p[i], M = m[i], V = v[i];
            adam_one(a, P, g[i], M, V);
            p[i] = P; m[i] = M; v[i] = V;
            if (bf) bf[i] = __float2bfloat16(P);
        }
    } else {
        for (int64_t i = tid; i < n; i += nth) {
            float P = p[i], M = m[i], V = v[i];
            adam_one(a, P, g[i], M, V);
            p[i] = P; m[i] = M; v[i] = V;
            if (bf) bf[i] = __float2bfloat16(P);
        }
    }
}

}  // namespace msst
using namespace msst;

extern "C" int msst_adam_step(const msst_adam_args* a, float* p, const float* g, float* m, float* v, void* bf16_out, int64_t n,
                              msst_stream_t stream) {
    MSST_REQUIRE(a && (a->step >= 1 || a->step_dev), "adam_step: step must be >= 1");
    if (n == 0) return MSST_OK;
    AdamK k;
    k.lr = a->lr; k.b1 = a->beta1; k.b2 = a->beta2; k.eps = a->eps; k.wd = a->weight_decay; k.clamp = a->clamp;
    k.gscale = a->grad_scale; k.decoupled = a->decoupled;
    k.omb1 = 1.f - k.b1; k.omb2 = 1.f - k.b2;
    const int st = a->step >= 1 ? a->step : 1;
    k.inv_bc1 = (float)(1.0 / (1.0 - pow((double)a->beta1, (double)st)));
    k.inv_sqrt_bc2 = (float)(1.0 / sqrt(1.0 - pow((double)a->beta2, (double)st)));
    k.step_dev = a->step_dev;
    auto al = [](const void* q) { return (reinterpret_cast<uintptr_t>(q) & 15u) == 0; };
    const int vec = al(p) && al(g) && al(m) && al(v) && (!bf16_out || (reinterpret_cast<uintptr_t>(bf16_out) & 7u) == 0);
    int64_t blocks = ceil_div(vec ? n / 4 + 1 : n, 256);
    if (blocks > 8 * kNumSMs) blocks = 8 * kNumSMs;
    adam_kernel<<<(int)blocks, 256, 0, (cudaStream_t)stream>>>(k, p, g, m, v, (__nv_bfloat16*)bf16_out, n, vec);
    MSST_LAUNCH_CHECK();
    return MSST_OK;
}
