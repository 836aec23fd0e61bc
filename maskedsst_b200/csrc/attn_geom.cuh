// Sequence / tile geometry shared by the fp32 and bf16 attention kernels (see attention_f32.cu for the scheme).
#pragma once
#include "common.cuh"

namespace msst {

constexpr int TS = 64;      // slots per tile
constexpr int AT = 256;     // threads

struct AttnGeom {
    int64_t n_seq; int N, inner, H, dh, G, tiles;   // tiles = key/query tiles per sequence (1 when N <= 64)
    int64_t groups;                                 // slot groups along the sequence axis
    float scale;
    int gpb;                                        // > 0: position-major packing, groups per block of `inner` sequences (see below)
};

// Packing of short sequences (N <= 64) into 64-slot groups, G = 64 / N sequences per group:
//   inner == 1 (sequence rows contiguous): group = G consecutive sequences, slot = j * N + pos          (sequence-major)
//   inner  > 1 (the spectral stack: row = blk*N*inner + pos*inner + s): a group takes G consecutive sequences of ONE block of
//       `inner` sequences (gpb = ceil(inner / G) groups per block), slot = pos * G + j                   (position-major)
//     -> the slots of a group are N runs of G consecutive rows: one TMA box {64 cols, G, N} over the (col, s, pos, blk) view
//        of the activation matrix lands them in slot order, and a group never straddles two blocks.
__device__ __forceinline__ int64_t group_seq0(const AttnGeom& g, int64_t group) {   // first sequence of a group (N <= 64)
    if (g.gpb == 0) return group * g.G;
    return (group / g.gpb) * g.inner + (group % g.gpb) * g.G;
}
__device__ __forceinline__ bool slot_to(const AttnGeom& g, int64_t group, int tile, int r, int64_t& seq, int& pos) {
    if (g.N <= TS) {
        if (g.gpb == 0) { seq = group * g.G + r / g.N; pos = r % g.N; return r < g.G * g.N && seq < g.n_seq; }
        const int j = r % g.G, j0 = (int)(group % g.gpb) * g.G;
        pos = r / g.G; seq = (group / g.gpb) * g.inner + j0 + j;
        return r < g.G * g.N && j0 + j < g.inner;
    }
    seq = group; pos = tile * TS + r; return pos < g.N;
}
__device__ __forceinline__ int64_t row_of(const AttnGeom& g, int64_t seq, int pos) {
    return (seq / g.inner) * g.N * g.inner + (seq % g.inner) + (int64_t)pos * g.inner;
}

inline int make_attn_geom(const msst_attn_dims* d, AttnGeom& g, bool any_dh) {
    MSST_REQUIRE(d && d->n_seq >= 0 && d->N > 0 && d->inner > 0 && d->H > 0, "attention: bad dims");
    MSST_REQUIRE(any_dh ? (d->dh == 32 || d->dh == 64 || d->dh == 128) : d->dh == 64, "attention: dim_head=%d unsupported (%s)", d->dh, any_dh ? "32, 64, 128" : "bf16 mode: 64");
    MSST_REQUIRE(d->n_seq % d->inner == 0, "attention: n_seq must be a multiple of inner");
    MSST_REQUIRE(d->H <= 65535, "attention: too many heads");
    MSST_REQUIRE(drop_p_ok(d->drop_p), "attention: drop_p=%g outside [0, 1]", (double)d->drop_p);
    g.n_seq = d->n_seq; g.N = d->N; g.inner = d->inner; g.H = d->H; g.dh = d->dh;
    g.scale = 1.0f / sqrtf((float)d->dh);
    g.gpb = 0;
    if (d->N <= TS) {
        g.G = TS / d->N; g.tiles = 1;
        if (d->inner > 1) { g.gpb = (d->inner + g.G - 1) / g.G; g.groups = (d->n_seq / d->inner) * g.gpb; }
        else g.groups = ceil_div(d->n_seq, g.G);
    } else { g.G = 1; g.tiles = (int)ceil_div(d->N, TS); g.groups = d->n_seq; }
    MSST_REQUIRE(g.groups * g.tiles < (int64_t)2147483647, "attention: grid too large");
    return MSST_OK;
}


}  // namespace msst
