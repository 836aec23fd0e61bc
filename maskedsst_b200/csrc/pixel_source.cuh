// Where pixel (sample b, band, row y, column x) of the model's [B, bands, H, W] cube comes from: either the fp32 standardised
// cube itself, or RAW sensor tiles with the reference's input pipeline applied on the fly (SURVEY.md 8(f) rank 2):
//   (raw - mean[band]) / std[band] in float64, rounded once to fp32  (StandardizeEnMAP / StandardizeHouston2018 on a numpy
//       array + ToTensor: src/data_enmap.py:454-457,517-522; src/data_houston2018.py:442-445)
//   optional clip of the STANDARDISED value                            (src/data_enmap.py:303-304)
//   bands >= raw_bands read as 0                                       (Houston 48 -> 50 zero pad, src/data_houston2018.py:268-269)
//   a crop window (y0, x0) shared by the whole batch                   (pretrain.py:99-107)
//   or ALL win_y x win_x windows of every tile as consecutive samples   (sliding-window inference, inference_example.ipynb cell 13)
//       stepped by (stride_y, stride_x), last row / column snapped to the tile border, from global window win_first on
// so the fp32 cube never exists in HBM and the host ships int16 tiles.
#pragma once
#include <stdint.h>
#include "../../include/msst.h"

namespace msst {

// Origin, along one axis, of window row (or column) i of a tile: o0 + i * step, except that a window which would cross the tile
// border is moved back flush with it.  The single statement of the rule: the pixel reader below and the scene blend
// (scene.cu) both call it.
__host__ __device__ __forceinline__ int window_origin(int i, int step, int o0, int tile, int win) {
    const int o = i * step, last = tile - o0 - win;
    return o0 + (o < last ? o : last);
}

struct PixelSource {
    const float* img;
    const void* raw;
    const double* mean;
    const double* stdv;
    int dtype, raw_bands, tile_h, tile_w, y0, x0, clip;
    float lo, hi;
    int bands, H, W;     // the model-side cube shape
    int win_y, win_x;    // > 1: sample b is window (g % (win_y*win_x)) of tile g / (win_y*win_x), g = win_first + b (no copy)
    int sy, sx;          // window step (the window size unless the windows overlap)
    int win_first;       // global index of sample 0's window

    __device__ __forceinline__ float load(int b, int band, int y, int x) const {
        if (img) return __ldg(img + ((int64_t)(b * bands + band) * H + y) * W + x);
        if (band >= raw_bands) return 0.f;
        int yy = y0 + y, xx = x0 + x;
        const int nwin = win_y * win_x;
        if (nwin > 1 || win_first) {
            const int g = win_first + b, w = g % nwin;
            b = g / nwin;
            yy = window_origin(w / win_x, sy, y0, tile_h, H) + y;
            xx = window_origin(w % win_x, sx, x0, tile_w, W) + x;
        }
        const int64_t o = (((int64_t)b * raw_bands + band) * tile_h + yy) * tile_w + xx;
        double v;
        if (dtype == MSST_RAW_I16) v = (double)__ldg(reinterpret_cast<const int16_t*>(raw) + o);
        else if (dtype == MSST_RAW_U16) v = (double)__ldg(reinterpret_cast<const uint16_t*>(raw) + o);
        else v = (double)__ldg(reinterpret_cast<const float*>(raw) + o);
        float f = (float)((v - __ldg(mean + band)) / __ldg(stdv + band));
        if (clip) f = fminf(fmaxf(f, lo), hi);
        return f;
    }
};

// host: fills a PixelSource from (img, optional raw descriptor); returns 0 or an error string
static inline const char* make_pixel_source(PixelSource& s, const float* img, const msst_raw_input* r, int bands, int H, int W) {
    s = PixelSource{};
    s.bands = bands; s.H = H; s.W = W;
    if (!r) { s.img = img; return img ? nullptr : "img is NULL and no raw input was given"; }
    if (!r->tiles || !r->mean || !r->std) return "raw input: tiles / mean / std must be set";
    if (r->dtype < MSST_RAW_I16 || r->dtype > MSST_RAW_F32) return "raw input: unknown dtype";
    if (r->raw_bands <= 0 || r->raw_bands > bands) return "raw input: raw_bands must be in [1, model bands]";
    const int wy = r->win_y > 0 ? r->win_y : 1, wx = r->win_x > 0 ? r->win_x : 1;
    if (r->stride_y < 0 || r->stride_x < 0 || r->stride_y > H || r->stride_x > W)
        return "raw input: window stride must be in [1, window] (0 = the window size)";
    if (r->win_first < 0) return "raw input: win_first must be >= 0";
    if (r->y0 < 0 || r->x0 < 0 || r->y0 + H > r->tile_h || r->x0 + W > r->tile_w) return "raw input: crop window(s) outside the tile";
    s.win_y = wy; s.win_x = wx;
    s.sy = r->stride_y > 0 ? r->stride_y : H; s.sx = r->stride_x > 0 ? r->stride_x : W; s.win_first = r->win_first;
    s.raw = r->tiles; s.mean = r->mean; s.stdv = r->std; s.dtype = r->dtype; s.raw_bands = r->raw_bands;
    s.tile_h = r->tile_h; s.tile_w = r->tile_w; s.y0 = r->y0; s.x0 = r->x0; s.clip = r->clip; s.lo = r->clip_lo; s.hi = r->clip_hi;
    return nullptr;
}

}  // namespace msst
