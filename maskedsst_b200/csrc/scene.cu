// Whole-scene inference: blend the class probabilities of overlapping windows into the scene (msst_scene_blend, include/msst.h).
// The reference classifies a scene window by window with no overlap (inference_example.ipynb cell 13, src/utils.py:477-605), so each
// 8 x 8 window only sees its own pixels and the map shows a seam every window.  Here windows overlap and every scene pixel receives
//   acc[c] += weight(py, px) * softmax_c(logits of each covering window at (py, px)),   wsum += weight(py, px)
// One thread owns one scene pixel and adds its covering windows in ascending global window index, one at a time (acc = acc + c): no
// atomics, so the sums are bitwise independent of how the windows were cut into chunks.  Which windows cover the pixel follows from
// the origin rule of the pixel reader (window_origin, pixel_source.cuh); the windows are never enumerated.
#include "common.cuh"
#include "pixel_source.cuh"

namespace msst {

constexpr int kBlendThreads = 128;
constexpr int kBlendMaxClasses = 256;

struct SceneGeom {
    int B, nc, H, W, win, sy, sx, win_y, win_x;
    int64_t g0, g1;        // the chunk: global windows [g0, g1)
    int64_t pix0, npix;    // the scene pixels it touches, flattened over (scene, row, column)
};

// Candidate window indices along one axis whose span may cover coordinate y: the nominal origins i * step give
// i in [ceil((y - win + 1) / step), y / step]; only the last window can be snapped (msst_scene_blend checks the window count), and it
// is added as a candidate when y lies in its snapped span.  The caller still tests every candidate against its true origin.
__device__ __forceinline__ void covering(int y, int step, int win, int extent, int nwin, int& lo, int& hi) {
    const int t = y - win + 1;
    lo = t > 0 ? (t + step - 1) / step : 0;
    hi = min(y / step, nwin - 1);
    if (hi < nwin - 1 && y >= window_origin(nwin - 1, step, 0, extent, win)) hi = nwin - 1;
}

// dynamic smem: the owning thread's running class sums, [nc][kBlendThreads] (conflict-free: class-major, thread-minor)
__global__ void __launch_bounds__(kBlendThreads) scene_blend_kernel(SceneGeom g, const float* __restrict__ logits,
                                                                    const float* __restrict__ weight, float* __restrict__ acc,
                                                                    float* __restrict__ wsum) {
    extern __shared__ float sacc[];
    const int64_t q = (int64_t)blockIdx.x * kBlendThreads + threadIdx.x;
    if (q >= g.npix) return;
    const int64_t p = g.pix0 + q;
    const int64_t HW = (int64_t)g.H * g.W;
    const int b = (int)(p / HW), y = (int)((p / g.W) % g.H), x = (int)(p % g.W);
    const int nwin = g.win_y * g.win_x, ww = g.win * g.win;
    int ilo, ihi, jlo, jhi;
    covering(y, g.sy, g.win, g.H, g.win_y, ilo, ihi);
    covering(x, g.sx, g.win, g.W, g.win_x, jlo, jhi);
    float* sa = sacc + threadIdx.x;
    float* ap = acc + (int64_t)b * g.nc * HW + (int64_t)y * g.W + x;
    float ws = 0.f;
    bool any = false;
    for (int i = ilo; i <= ihi; ++i) {
        const int oy = window_origin(i, g.sy, 0, g.H, g.win);
        if (y < oy || y >= oy + g.win) continue;
        for (int j = jlo; j <= jhi; ++j) {
            const int ox = window_origin(j, g.sx, 0, g.W, g.win);
            if (x < ox || x >= ox + g.win) continue;
            const int64_t gw = (int64_t)b * nwin + (int64_t)i * g.win_x + j;
            if (gw < g.g0 || gw >= g.g1) continue;
            if (!any) {   // first contribution of this chunk: load the running sums
                any = true;
                ws = wsum[p];
                for (int c = 0; c < g.nc; ++c) sa[c * kBlendThreads] = ap[c * HW];
            }
            const int pix = (y - oy) * g.win + (x - ox);
            const float* lp = logits + (gw - g.g0) * g.nc * ww + pix;
            float mx = -INFINITY;
            for (int c = 0; c < g.nc; ++c) mx = fmaxf(mx, __ldg(lp + c * ww));
            float se = 0.f;
            for (int c = 0; c < g.nc; ++c) se += expf(__ldg(lp + c * ww) - mx);
            const float inv = __frcp_rn(se), wt = weight ? __ldg(weight + pix) : 1.f;
            for (int c = 0; c < g.nc; ++c) {
                const float pc = __fmul_rn(expf(__ldg(lp + c * ww) - mx), inv);
                sa[c * kBlendThreads] = __fadd_rn(sa[c * kBlendThreads], __fmul_rn(wt, pc));
            }
            ws = __fadd_rn(ws, wt);
        }
    }
    if (!any) return;
    wsum[p] = ws;
    for (int c = 0; c < g.nc; ++c) ap[c * HW] = sa[c * kBlendThreads];
}

static int64_t windows_along(int extent, int win, int step) { return (extent - win + step - 1) / step + 1; }

}  // namespace msst
using namespace msst;

extern "C" int msst_scene_blend(const msst_scene_dims* d, const float* logits, const float* weight, float* acc, float* wsum,
                                msst_stream_t stream) {
    MSST_REQUIRE(d && d->B > 0 && d->nc > 0 && d->win > 0, "scene_blend: bad dims");
    MSST_REQUIRE(d->nc <= kBlendMaxClasses, "scene_blend: nc=%d > %d unsupported", d->nc, kBlendMaxClasses);
    MSST_REQUIRE(d->H >= d->win && d->W >= d->win, "scene_blend: scene %dx%d smaller than the window %d", d->H, d->W, d->win);
    MSST_REQUIRE(d->stride_y >= 1 && d->stride_y <= d->win && d->stride_x >= 1 && d->stride_x <= d->win,
                 "scene_blend: stride (%d, %d) must be in [1, window=%d]", d->stride_y, d->stride_x, d->win);
    MSST_REQUIRE(d->win_y >= 1 && d->win_y <= windows_along(d->H, d->win, d->stride_y) && d->win_x >= 1 &&
                 d->win_x <= windows_along(d->W, d->win, d->stride_x),
                 "scene_blend: window grid %dx%d exceeds ceil((extent - window) / stride) + 1", d->win_y, d->win_x);
    const int64_t nwin = (int64_t)d->win_y * d->win_x;
    MSST_REQUIRE(d->win_first >= 0 && d->n >= 1 && d->win_first + (int64_t)d->n <= d->B * nwin,
                 "scene_blend: windows [%d, %d + %d) outside [0, %lld)", d->win_first, d->win_first, d->n, (long long)(d->B * nwin));
    MSST_REQUIRE(logits && acc && wsum, "scene_blend: logits / acc / wsum must be set");
    SceneGeom g;
    g.B = d->B; g.nc = d->nc; g.H = d->H; g.W = d->W; g.win = d->win; g.sy = d->stride_y; g.sx = d->stride_x;
    g.win_y = d->win_y; g.win_x = d->win_x; g.g0 = d->win_first; g.g1 = d->win_first + (int64_t)d->n;
    // rows touched: from the first window's top row to the last window's bottom row (flattened over scenes)
    const int64_t ga = g.g0, gb = g.g1 - 1;
    const int64_t row0 = (ga / nwin) * g.H + window_origin((int)(ga % nwin) / g.win_x, g.sy, 0, g.H, g.win);
    const int64_t row1 = (gb / nwin) * g.H + window_origin((int)(gb % nwin) / g.win_x, g.sy, 0, g.H, g.win) + g.win;
    g.pix0 = row0 * g.W; g.npix = (row1 - row0) * g.W;
    const size_t smem = sizeof(float) * (size_t)g.nc * kBlendThreads;
    cudaStream_t st = (cudaStream_t)stream;
    if (smem > 48 * 1024) MSST_CUDA(cudaFuncSetAttribute(scene_blend_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    scene_blend_kernel<<<(unsigned)ceil_div(g.npix, kBlendThreads), kBlendThreads, smem, st>>>(g, logits, weight, acc, wsum);
    MSST_LAUNCH_CHECK();
    return MSST_OK;
}
