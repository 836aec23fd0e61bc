// Whole-scene inference: blend the class probabilities of overlapping windows into the scene (msst_scene_blend, include/msst.h).
// The reference classifies a scene window by window with no overlap (inference_example.ipynb cell 13, src/utils.py:477-605), so each
// 8 x 8 window only sees its own pixels and the map shows a seam every window.  Here windows overlap and every scene pixel receives
//   acc[c] += weight(py, px) * softmax_c(logits of each covering window at (py, px)),   wsum += weight(py, px)
// One thread owns one scene pixel and adds its covering windows in ascending global window index, one at a time (acc = acc + c): no
// atomics, so the sums are bitwise independent of how the windows were cut into chunks.  Which windows cover the pixel follows from
// the origin rule of the pixel reader (window_origin, pixel_source.cuh); the windows are never enumerated.  msst_scene_embed blends
// per-pixel encoder features the same way (below).
#include "common.cuh"
#include "pixel_source.cuh"

namespace msst {

constexpr int kBlendThreads = 128;
constexpr int kBlendMaxClasses = 256;

struct SceneGeom {
    int B, nc, H, W, win, sy, sx, win_y, win_x;   // nc: channels of acc (classes for the blend, features for the embedding)
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

// Calls fn(gw, py, px) for every window of the chunk that covers scene pixel (b, y, x), in ascending global window index gw; (py, px) is
// the pixel's position inside the window.
template <class Fn>
__device__ __forceinline__ void for_each_covering_window(const SceneGeom& g, int b, int y, int x, Fn&& fn) {
    int ilo, ihi, jlo, jhi;
    covering(y, g.sy, g.win, g.H, g.win_y, ilo, ihi);
    covering(x, g.sx, g.win, g.W, g.win_x, jlo, jhi);
    const int nwin = g.win_y * g.win_x;
    for (int i = ilo; i <= ihi; ++i) {
        const int oy = window_origin(i, g.sy, 0, g.H, g.win);
        if (y < oy || y >= oy + g.win) continue;
        for (int j = jlo; j <= jhi; ++j) {
            const int ox = window_origin(j, g.sx, 0, g.W, g.win);
            if (x < ox || x >= ox + g.win) continue;
            const int64_t gw = (int64_t)b * nwin + (int64_t)i * g.win_x + j;
            if (gw < g.g0 || gw >= g.g1) continue;
            fn(gw, y - oy, x - ox);
        }
    }
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
    const int ww = g.win * g.win;
    float* sa = sacc + threadIdx.x;
    float* ap = acc + (int64_t)b * g.nc * HW + (int64_t)y * g.W + x;
    float ws = 0.f;
    bool any = false;
    for_each_covering_window(g, b, y, x, [&](int64_t gw, int py, int px) {
        if (!any) {   // first contribution of this chunk: load the running sums
            any = true;
            ws = wsum[p];
            for (int c = 0; c < g.nc; ++c) sa[c * kBlendThreads] = ap[c * HW];
        }
        const int pix = py * g.win + px;
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
    });
    if (!any) return;
    wsum[p] = ws;
    for (int c = 0; c < g.nc; ++c) ap[c * HW] = sa[c * kBlendThreads];
}

// Embedding maps (msst_scene_embed): the same ownership and window order, but each covering window contributes its encoder feature at
// the pixel, f = (1/C) sum_c tokens[c*S + s, :] (the spectral mean the default head starts from), instead of a softmax.  A block owns
// kEmbedPix consecutive scene pixels and keeps their running sums in shared memory, [D][kEmbedPix + 1]: acc / wsum are loaded and
// stored with lanes over pixels (consecutive in acc), and the windows are accumulated with one warp per pixel and lanes over features,
// so every token row is read as whole 128-byte lines.  One thread per pixel with the features in a loop would read tokens D floats
// apart across a warp; lanes over features alone would store acc HW floats apart.
constexpr int kEmbedThreads = 256;
constexpr int kEmbedPix = 32;
constexpr int kEmbedMaxDim = 256;

__global__ void __launch_bounds__(kEmbedThreads) scene_embed_kernel(SceneGeom g, int C, int p1, const float* __restrict__ tokens,
                                                                    const float* __restrict__ weight, float* __restrict__ acc,
                                                                    float* __restrict__ wsum) {
    constexpr int LD = kEmbedPix + 1;   // conflict-free in both phases: bank (d + k) mod 32 and (d * 33 + lane) mod 32
    extern __shared__ float sacc[];
    const int D = g.nc;
    float* sws = sacc + D * LD;
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    constexpr int kWarps = kEmbedThreads / 32;
    const int64_t HW = (int64_t)g.H * g.W;
    const int64_t q0 = (int64_t)blockIdx.x * kEmbedPix;
    // every pixel of the visited rows is loaded and stored back; one that no window of the chunk covers keeps its value
    const bool mine = q0 + lane < g.npix;
    const int64_t pl = g.pix0 + q0 + lane;
    float* ap = acc + (pl / HW) * D * HW + pl % HW;
    if (mine) {
        for (int d = warp; d < D; d += kWarps) sacc[d * LD + lane] = ap[d * HW];
        if (warp == 0) sws[lane] = wsum[pl];
    }
    __syncthreads();
    const int G = g.win / p1, S = G * G;
    const float fC = (float)C;
    for (int k = warp; k < kEmbedPix && q0 + k < g.npix; k += kWarps) {
        const int64_t p = g.pix0 + q0 + k;
        const int b = (int)(p / HW), y = (int)((p / g.W) % g.H), x = (int)(p % g.W);
        float ws = sws[k];
        for_each_covering_window(g, b, y, x, [&](int64_t gw, int py, int px) {
            const float wt = weight ? __ldg(weight + py * g.win + px) : 1.f;
            const float* tp = tokens + ((gw - g.g0) * C * S + (py / p1) * G + px / p1) * D;
            for (int d = lane; d < D; d += 32) {
                float s = 0.f;
#pragma unroll 4
                for (int c = 0; c < C; ++c) s = __fadd_rn(s, __ldg(tp + (int64_t)c * S * D + d));
                float* a = sacc + d * LD + k;
                *a = __fadd_rn(*a, __fmul_rn(wt, __fdiv_rn(s, fC)));
            }
            ws = __fadd_rn(ws, wt);
        });
        if (lane == 0) sws[k] = ws;
    }
    __syncthreads();
    if (mine) {
        for (int d = warp; d < D; d += kWarps) ap[d * HW] = sacc[d * LD + lane];
        if (warp == 0) wsum[pl] = sws[lane];
    }
}

static int64_t windows_along(int extent, int win, int step) { return (extent - win + step - 1) / step + 1; }

// Checks the window geometry both entry points share (msst_scene_dims and msst_scene_embed_dims name it alike) and fills g: the
// chunk, and the scene rows it touches -- from the first window's top row to the last window's bottom row, flattened over scenes.
template <class Dims>
static int scene_geom(const char* who, const Dims* d, int nch, SceneGeom& g) {
    MSST_REQUIRE(d->H >= d->win && d->W >= d->win, "%s: scene %dx%d smaller than the window %d", who, d->H, d->W, d->win);
    MSST_REQUIRE(d->stride_y >= 1 && d->stride_y <= d->win && d->stride_x >= 1 && d->stride_x <= d->win,
                 "%s: stride (%d, %d) must be in [1, window=%d]", who, d->stride_y, d->stride_x, d->win);
    MSST_REQUIRE(d->win_y >= 1 && d->win_y <= windows_along(d->H, d->win, d->stride_y) && d->win_x >= 1 &&
                 d->win_x <= windows_along(d->W, d->win, d->stride_x),
                 "%s: window grid %dx%d exceeds ceil((extent - window) / stride) + 1", who, d->win_y, d->win_x);
    const int64_t nwin = (int64_t)d->win_y * d->win_x;
    MSST_REQUIRE(d->win_first >= 0 && d->n >= 1 && d->win_first + (int64_t)d->n <= d->B * nwin,
                 "%s: windows [%d, %d + %d) outside [0, %lld)", who, d->win_first, d->win_first, d->n, (long long)(d->B * nwin));
    g.B = d->B; g.nc = nch; g.H = d->H; g.W = d->W; g.win = d->win; g.sy = d->stride_y; g.sx = d->stride_x;
    g.win_y = d->win_y; g.win_x = d->win_x; g.g0 = d->win_first; g.g1 = d->win_first + (int64_t)d->n;
    const int64_t ga = g.g0, gb = g.g1 - 1;
    const int64_t row0 = (ga / nwin) * g.H + window_origin((int)(ga % nwin) / g.win_x, g.sy, 0, g.H, g.win);
    const int64_t row1 = (gb / nwin) * g.H + window_origin((int)(gb % nwin) / g.win_x, g.sy, 0, g.H, g.win) + g.win;
    g.pix0 = row0 * g.W; g.npix = (row1 - row0) * g.W;
    return MSST_OK;
}

}  // namespace msst
using namespace msst;

extern "C" int msst_scene_blend(const msst_scene_dims* d, const float* logits, const float* weight, float* acc, float* wsum,
                                msst_stream_t stream) {
    MSST_REQUIRE(d && d->B > 0 && d->nc > 0 && d->win > 0, "scene_blend: bad dims");
    MSST_REQUIRE(d->nc <= kBlendMaxClasses, "scene_blend: nc=%d > %d unsupported", d->nc, kBlendMaxClasses);
    SceneGeom g;
    const int rc = scene_geom("scene_blend", d, d->nc, g);
    if (rc != MSST_OK) return rc;
    MSST_REQUIRE(logits && acc && wsum, "scene_blend: logits / acc / wsum must be set");
    const size_t smem = sizeof(float) * (size_t)g.nc * kBlendThreads;
    cudaStream_t st = (cudaStream_t)stream;
    if (smem > 48 * 1024) MSST_CUDA(cudaFuncSetAttribute(scene_blend_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    scene_blend_kernel<<<(unsigned)ceil_div(g.npix, kBlendThreads), kBlendThreads, smem, st>>>(g, logits, weight, acc, wsum);
    MSST_LAUNCH_CHECK();
    return MSST_OK;
}

extern "C" int msst_scene_embed(const msst_scene_embed_dims* d, const float* tokens, const float* weight, float* acc, float* wsum,
                                msst_stream_t stream) {
    MSST_REQUIRE(d && d->B > 0 && d->D > 0 && d->win > 0 && d->C > 0 && d->p1 > 0, "scene_embed: bad dims");
    MSST_REQUIRE(d->D <= kEmbedMaxDim, "scene_embed: D=%d > %d unsupported", d->D, kEmbedMaxDim);
    MSST_REQUIRE(d->win % d->p1 == 0, "scene_embed: window %d is not a multiple of the spatial patch side p1=%d", d->win, d->p1);
    SceneGeom g;
    const int rc = scene_geom("scene_embed", d, d->D, g);
    if (rc != MSST_OK) return rc;
    MSST_REQUIRE(tokens && acc && wsum, "scene_embed: tokens / acc / wsum must be set");
    const size_t smem = sizeof(float) * ((size_t)g.nc * (kEmbedPix + 1) + kEmbedPix);   // <= 33.9 KB at D = 256
    scene_embed_kernel<<<(unsigned)ceil_div(g.npix, kEmbedPix), kEmbedThreads, smem, (cudaStream_t)stream>>>(g, d->C, d->p1, tokens,
                                                                                                          weight, acc, wsum);
    MSST_LAUNCH_CHECK();
    return MSST_OK;
}
