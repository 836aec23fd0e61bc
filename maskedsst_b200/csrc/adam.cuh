// The Adam / AdamW update of one parameter, shared by the optimiser arena kernel (adamw.cu) and the fused linear-probe update
// (linprobe.cu), so both follow torch.optim.AdamW / Adam with the same arithmetic.
#pragma once
#include "common.cuh"

namespace msst {

// omb1 / omb2 = 1 - beta1 / 1 - beta2 as the caller rounds them to fp32: msst_adam_step keeps the fp32 difference 1.f - beta it has
// always used; the linear probe rounds 1 - beta from double, as torch.optim.AdamW does (1.f - 0.999f is 1.3e-5 off 0.001)
struct AdamK { float lr, b1, b2, eps, wd, clamp, gscale, inv_bc1, inv_sqrt_bc2, omb1, omb2; int decoupled; const int* step_dev; };

__device__ __forceinline__ void adam_one(const AdamK& a, float& p, float g, float& m, float& v) {
    g *= a.gscale;
    if (a.clamp > 0.f) g = fminf(fmaxf(g, -a.clamp), a.clamp);
    if (a.decoupled) p *= (1.f - a.lr * a.wd); else g = fmaf(a.wd, p, g);
    m = a.b1 * m + a.omb1 * g;
    v = a.b2 * v + a.omb2 * g * g;
    const float denom = sqrtf(v) * a.inv_sqrt_bc2 + a.eps;
    p -= (a.lr * a.inv_bc1) * (m / denom);
}

}  // namespace msst
