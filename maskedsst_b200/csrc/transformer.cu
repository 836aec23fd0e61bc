// Native orchestration of one Transformer stack (L pre-norm layers) -- all launches of the stack are issued
// from here so the Python host makes one call per stack per direction.
// Reference: Transformer.forward, src/vit_spatial_spectral.py:100-104 (x = attn(LN(x)) + x ; x = ff(LN(x)) + x),
// Attention :47-78, FeedForward :32-44; backward = autograd of the same.
//
// Workspace (device memory owned by the caller, see msst_transformer_workspace_bytes):
//   per layer (only layer 0's slot when save_for_backward == 0):
//     stats1 [R,2] stats2 [R,2] | qkv [R,3I] | o [R,I] | lse [R,H] | xmid [R,D] | u [R,M] | g [R,M] | xout [R,D]
//   shared scratch: h [R,D]; backward adds dqkv [R,3I], do [R,I], du [R,M], dh [R,D], dy [R,D], dxa [R,D], dxb [R,D]
// The residual stream, LN statistics and lse are always fp32.
#include "common.cuh"
#include "kernels.h"
#include "attn_geom.cuh"
#include <stdlib.h>

namespace msst {

static inline size_t al256(size_t b) { return (b + 255) & ~(size_t)255; }

struct TfLayout {
    int64_t R; int I;
    size_t o_stats1, o_stats2, o_qkv, o_o, o_lse, o_xmid, o_u, o_g, o_xout, o_h1, o_h2, layer_bytes;
    size_t o_wq, o_wqT, o_wo, o_woT, o_w1, o_w1T, o_w2, o_w2T, wlayer_bytes, w_base;   // bf16 mode: per-layer bf16 weight copies
    size_t s_h, s_dqkv, s_do, s_du, s_dh, s_dy, s_dxa, s_dxb, total;
    int layer_slots;
};

// bf16 mode: the QKV projection runs inside the attention kernels (attn_block_tc.cu) whenever the geometry allows it: qkv is
// never materialised (forward) and is recomputed from the saved LayerNorm output in the backward, which also folds the
// projection's data gradient in.  MSST_ATTN_FUSED=0 selects the separate GEMM + attention kernels.
static bool attn_fused(const msst_tf_dims* d) {
    static int v = -1;
    if (v < 0) { const char* e = getenv("MSST_ATTN_FUSED"); v = e ? atoi(e) : 1; }
    if (!v || d->prec != MSST_PREC_BF16 || d->dh != 64) return false;
    msst_attn_dims ad{d->n_seq, d->N, d->inner, d->H, d->dh, 0.f, 0, 0, d->prec, nullptr};
    AttnGeom g;
    if (d->n_seq == 0 || make_attn_geom(&ad, g, false)) return false;
    return attn_block_supported(g, d->D);
}

// bf16 mode, fused attention: the out-projection + residual + FeedForward pre-norm run in the tail of the attention forward kernel
// (no gemm_tn<6> launch, o is not re-read).  MSST_ATTN_OUT_FUSED=0 selects the separate GEMM.
static bool attn_out_fused() {
    static int v = -1;
    if (v < 0) { const char* e = getenv("MSST_ATTN_OUT_FUSED"); v = e ? atoi(e) : 1; }
    return v != 0;
}

// bf16 mode: the FeedForward block as one kernel (mlp_block_tc.cu).  MSST_MLP_FUSED=0 selects the two GEMM launches.
static bool mlp_fused(const msst_tf_dims* d) {
    static int v = -1;
    if (v < 0) { const char* e = getenv("MSST_MLP_FUSED"); v = e ? atoi(e) : 1; }
    return v && d->prec == MSST_PREC_BF16 && mlp_block_supported(d->D, d->M);
}

static TfLayout make_layout(const msst_tf_dims* d) {
    TfLayout L{};
    L.R = d->n_seq * d->N; L.I = d->H * d->dh;
    const size_t R = (size_t)L.R, f = sizeof(float);
    const size_t a = d->prec == MSST_PREC_BF16 ? 2 : 4;   // activation element size (qkv, o, u, g, h, d*): bf16 or fp32
    size_t off = 0;
    auto take = [&](size_t bytes) { size_t o = off; off += al256(bytes); return o; };
    L.o_stats1 = take(R * 2 * f); L.o_stats2 = take(R * 2 * f);
    L.o_qkv = take(attn_fused(d) ? 0 : R * 3 * L.I * a); L.o_o = take(R * L.I * a); L.o_lse = take(R * d->H * f);
    L.o_xmid = take(R * d->D * f); L.o_u = take(R * d->M * a); L.o_g = take(R * d->M * a); L.o_xout = take(R * d->D * f);
    L.o_h1 = L.o_h2 = 0;
    if (d->prec == MSST_PREC_BF16 && d->save_for_backward) {   // LN outputs (bf16): 2 x 2D B/token saves 2 LN passes in backward
        L.o_h1 = take(R * d->D * a); L.o_h2 = take(R * d->D * a);
    }
    L.layer_bytes = off;
    L.layer_slots = d->save_for_backward ? d->L : 1;
    off = L.layer_bytes * L.layer_slots;
    if (d->prec == MSST_PREC_BF16) {
        const size_t base = off;
        off = 0;
        const size_t nq = (size_t)3 * L.I * d->D * 2, no = (size_t)d->D * L.I * 2, n1 = (size_t)d->M * d->D * 2;
        L.o_wq = take(nq); L.o_wqT = take(nq); L.o_wo = take(no); L.o_woT = take(no);
        L.o_w1 = take(n1); L.o_w1T = take(n1); L.o_w2 = take(n1); L.o_w2T = take(n1);
        L.wlayer_bytes = off;
        L.w_base = base;
        off = base + L.wlayer_bytes * d->L;
    }
    L.s_h = take(R * d->D * a);
    if (d->save_for_backward) {
        L.s_dqkv = take(R * 3 * L.I * a); L.s_do = take(R * L.I * a); L.s_du = take(R * d->M * a);
        L.s_dh = take(R * d->D * f); L.s_dy = take(R * d->D * a); L.s_dxa = take(R * d->D * f); L.s_dxb = take(R * d->D * f);
    }
    L.total = off;
    return L;
}

static int check_dims(const msst_tf_dims* d) {
    MSST_REQUIRE(d && d->n_seq >= 0 && d->N > 0 && d->inner > 0 && d->L > 0, "transformer: bad dims");
    MSST_REQUIRE(d->D > 0 && d->D <= 256 && d->M > 0 && d->H > 0, "transformer: bad model dims");
    MSST_REQUIRE(d->D % 4 == 0 && d->M % 4 == 0, "transformer: D and M must be multiples of 4");
    MSST_REQUIRE(d->prec == MSST_PREC_FP32 || d->prec == MSST_PREC_BF16, "transformer: unknown precision mode %d", d->prec);
    MSST_REQUIRE(drop_p_ok(d->drop_p), "transformer: drop_p=%g outside [0, 1]", (double)d->drop_p);
    if (d->prec == MSST_PREC_BF16) {
        MSST_REQUIRE(d->dh == 64, "transformer (bf16): dim_head must be 64");
        MSST_REQUIRE(d->D % 8 == 0 && d->M % 8 == 0 && d->L <= 8, "transformer (bf16): D, M must be multiples of 8 and L <= 8");
    }
    return MSST_OK;
}

typedef __nv_bfloat16 bf16;

struct Bf16Weights { bf16 *wq, *wqT, *wo, *woT, *w1, *w1T, *w2, *w2T; };
static Bf16Weights layer_weights(const TfLayout& L, char* ws, int l) {
    char* b = ws + L.w_base + L.wlayer_bytes * l;
    return {(bf16*)(b + L.o_wq), (bf16*)(b + L.o_wqT), (bf16*)(b + L.o_wo), (bf16*)(b + L.o_woT),
            (bf16*)(b + L.o_w1), (bf16*)(b + L.o_w1T), (bf16*)(b + L.o_w2), (bf16*)(b + L.o_w2T)};
}

// MSST_GEMM_LNB=1: LayerNorm backward fused into the epilogue of the data-gradient GEMM that produces its dy (gemm MODE 8).
// Parity-tested, but OFF by default: measured 21.5 vs 21.1 ms/step -- the 16 epilogue warps (96 registers, one row buffer) hide
// the x / skip-gradient load latency worse than the stand-alone kernel's 64 warps per SM, and the K = 1536 GEMM is otherwise
// at 0.94 of the HBM peak.
static bool lnb_enabled() {
    static int v = -1;
    if (v < 0) { const char* e = getenv("MSST_GEMM_LNB"); v = e ? atoi(e) : 0; }
    return v != 0;
}

static GemmBf16Args gemm_args(const bf16* A, const bf16* B, int64_t M, int N, int K, void* out, int out_fp32) {
    GemmBf16Args a{};
    a.A = A; a.B = B; a.M = M; a.N = N; a.K = K; a.out = out; a.out_fp32 = out_fp32; a.drop = make_drop(0.f, 0, 0);
    return a;
}

// ---- bf16 mode: tcgen05 GEMMs + tensor-core attention; residual stream / LN statistics / lse stay fp32 ----
static int tf_fwd_bf16(const msst_tf_dims* d, const msst_layer_params* layers, const float* x_in, float* x_out, char* ws, cudaStream_t st) {
    const TfLayout L = make_layout(d);
    const int64_t R = L.R;
    const int D = d->D, I = L.I, M = d->M;
    // bf16 (and transposed) copies of this stack's weight matrices: one launch
    WeightCastTable tab{}; tab.n = 0;
    for (int l = 0; l < d->L; ++l) {
        const Bf16Weights w = layer_weights(L, ws, l);
        tab.e[tab.n++] = {layers[l].w_qkv, w.wq, w.wqT, 3 * I, D};
        tab.e[tab.n++] = {layers[l].w_out, w.wo, w.woT, D, I};
        tab.e[tab.n++] = {layers[l].w1, w.w1, w.w1T, M, D};
        tab.e[tab.n++] = {layers[l].w2, w.w2, w.w2T, D, M};
    }
    if (int rc = weights_to_bf16(tab, st)) return rc;
    bf16* h = (bf16*)(ws + L.s_h);
    const float* x = x_in;
    const bool fused = attn_fused(d);
    for (int l = 0; l < d->L; ++l) {
        char* lw = ws + L.layer_bytes * (d->save_for_backward ? l : 0);
        const msst_layer_params& p = layers[l];
        const Bf16Weights w = layer_weights(L, ws, l);
        float* stats1 = (float*)(lw + L.o_stats1); float* stats2 = (float*)(lw + L.o_stats2);
        bf16* qkv = (bf16*)(lw + L.o_qkv); bf16* o = (bf16*)(lw + L.o_o); float* lse = (float*)(lw + L.o_lse);
        float* xmid = (float*)(lw + L.o_xmid); bf16* u = (bf16*)(lw + L.o_u); bf16* g = (bf16*)(lw + L.o_g);
        float* y = (l == d->L - 1) ? x_out : (float*)(lw + L.o_xout);
        const uint32_t site = d->site_base + 8u * l;
        bf16* h1 = d->save_for_backward ? (bf16*)(lw + L.o_h1) : h;
        bf16* h2 = d->save_for_backward ? (bf16*)(lw + L.o_h2) : h;
        // pre-norms are produced by the epilogue of the GEMM that finishes the residual-stream row (fused LayerNorm);
        // only the first layer's LN1 is a stand-alone kernel
        const bool fuse_ln = (D % 4 == 0 && D <= 128);
        if (l == 0 || !fuse_ln) { if (int rc = layernorm_fwd(x, p.ln1_w, p.ln1_b, h1, 1, stats1, R, D, 1e-5f, st)) return rc; }
        msst_attn_dims ad{d->n_seq, d->N, d->inner, d->H, d->dh, d->drop_p, d->seed, site + kSiteAttnProb, d->prec, d->seed_dev};
        const bool tail = fused && fuse_ln && attn_out_fused();
        if (fused) {
            AttnGeom ag;
            if (int rc = make_attn_geom(&ad, ag, false)) return rc;
            // tail: xmid = x + drop(o Wo^T + b_out) and h2 = LN2(xmid) leave the same kernel (o is only written, for the Wo weight gradient)
            const AttnBlockOut t{w.wo, p.b_out, x, xmid, p.ln2_w, p.ln2_b, h2, stats2, make_drop(d->drop_p, d->seed, site + kSiteAttnOut, d->seed_dev)};
            if (int rc = attn_block_fwd(ag, D, h1, w.wq, (tail && !d->save_for_backward) ? nullptr : o, lse,
                                        make_drop(d->drop_p, d->seed, site + kSiteAttnProb, d->seed_dev), st, tail ? &t : nullptr)) return rc;
        } else {
            if (int rc = gemm_tn_bf16(gemm_args(h1, w.wq, R, 3 * I, D, qkv, 0), st)) return rc;
            if (int rc = attention_fwd_bf16(&ad, qkv, o, lse, st)) return rc;
        }
        GemmBf16Args a{};
        if (!tail) {
            a = gemm_args(o, w.wo, R, D, I, xmid, 1);
            a.bias = p.b_out; a.residual = x; a.drop = make_drop(d->drop_p, d->seed, site + kSiteAttnOut, d->seed_dev);
            if (fuse_ln) { a.ln_w = p.ln2_w; a.ln_b = p.ln2_b; a.ln_out = h2; a.ln_stats = stats2; }
            if (int rc = gemm_tn_bf16(a, st)) return rc;
            if (!fuse_ln) { if (int rc = layernorm_fwd(xmid, p.ln2_w, p.ln2_b, h2, 1, stats2, R, D, 1e-5f, st)) return rc; }
        }
        if (mlp_fused(d)) {   // Linear -> GELU -> dropout -> Linear -> dropout -> + xmid (-> LN1 of the next layer): one kernel
            const bool next_ln = l + 1 < d->L;
            char* nlw = ws + L.layer_bytes * (d->save_for_backward ? l + 1 : 0);
            if (int rc = mlp_block_fwd(h2, xmid, w.w1, w.w2, p.b1, p.b2, u, g, y, next_ln ? layers[l + 1].ln1_w : nullptr,
                                       next_ln ? layers[l + 1].ln1_b : nullptr,
                                       next_ln ? (d->save_for_backward ? (bf16*)(nlw + L.o_h1) : h) : nullptr,
                                       next_ln ? (float*)(nlw + L.o_stats1) : nullptr, R, D, M,
                                       make_drop(d->drop_p, d->seed, site + kSiteMlpHidden, d->seed_dev),
                                       make_drop(d->drop_p, d->seed, site + kSiteMlpOut, d->seed_dev), st)) return rc;
            x = y;
            continue;
        }
        a = gemm_args(h2, w.w1, R, M, D, g, 0);
        a.bias = p.b1; a.pre_act = u; a.act = 1; a.drop = make_drop(d->drop_p, d->seed, site + kSiteMlpHidden, d->seed_dev);
        if (int rc = gemm_tn_bf16(a, st)) return rc;
        a = gemm_args(g, w.w2, R, D, M, y, 1);
        a.bias = p.b2; a.residual = xmid; a.drop = make_drop(d->drop_p, d->seed, site + kSiteMlpOut, d->seed_dev);
        if (fuse_ln && l + 1 < d->L) {   // LN1 of the next layer
            char* nlw = ws + L.layer_bytes * (d->save_for_backward ? l + 1 : 0);
            a.ln_w = layers[l + 1].ln1_w; a.ln_b = layers[l + 1].ln1_b;
            a.ln_out = d->save_for_backward ? (bf16*)(nlw + L.o_h1) : h; a.ln_stats = (float*)(nlw + L.o_stats1);
        }
        if (int rc = gemm_tn_bf16(a, st)) return rc;
        x = y;
    }
    return MSST_OK;
}

static int tf_bwd_bf16(const msst_tf_dims* d, const msst_layer_params* layers, const msst_layer_grads* grads, const float* x_in,
                       const float* d_x_out, float* d_x_in, char* ws, cudaStream_t st) {
    const TfLayout L = make_layout(d);
    const int64_t R = L.R;
    const int D = d->D, I = L.I, M = d->M;
    bf16* dqkv = (bf16*)(ws + L.s_dqkv); bf16* dO = (bf16*)(ws + L.s_do);
    bf16* du = (bf16*)(ws + L.s_du); float* dh = (float*)(ws + L.s_dh); bf16* dyb = (bf16*)(ws + L.s_dy);
    float* dxa = (float*)(ws + L.s_dxa); float* dxb = (float*)(ws + L.s_dxb);
    const float* dcur = d_x_out;
    const Drop none = make_drop(0.f, 0, 0);
    bool dyb_ready = false;
    const bool fused = attn_fused(d);
    for (int l = d->L - 1; l >= 0; --l) {
        char* lw = ws + L.layer_bytes * l;
        const msst_layer_params& p = layers[l];
        const msst_layer_grads& gr = grads[l];
        const Bf16Weights w = layer_weights(L, ws, l);
        float* stats1 = (float*)(lw + L.o_stats1); float* stats2 = (float*)(lw + L.o_stats2);
        bf16* qkv = (bf16*)(lw + L.o_qkv); bf16* o = (bf16*)(lw + L.o_o); float* lse = (float*)(lw + L.o_lse);
        float* xmid = (float*)(lw + L.o_xmid); bf16* u = (bf16*)(lw + L.o_u); bf16* g = (bf16*)(lw + L.o_g);
        const float* x = (l == 0) ? x_in : (const float*)(ws + L.layer_bytes * (l - 1) + L.o_xout);
        const uint32_t site = d->site_base + 8u * l;
        // ---- MLP branch ----
        // dyb = bf16(dropout_mlp_out(dcur)) and db2: produced by the previous layer-iteration's LN1 backward (fused), or by a
        // stand-alone cast for the gradient that enters the stack
        if (!dyb_ready) {
            if (int rc = cast_rows_f32(dcur, dyb, gr.b2, R, D, make_drop(d->drop_p, d->seed, site + kSiteMlpOut, d->seed_dev), st)) return rc;
        }
        const bool fuse_lnb = (D % 4 == 0 && D <= 128) && lnb_enabled();
        if (mlp_fused(d) && !fuse_lnb) {
            // the whole FeedForward backward in one kernel: du never reaches HBM, dW1 / dW2 accumulate in TMEM across the launch
            if (int rc = mlp_block_bwd(dyb, u, g, (const bf16*)(lw + L.o_h2), w.w2T, w.w1T, gr.w1, gr.w2, gr.b1, dh, R, D, M,
                                       make_drop(d->drop_p, d->seed, site + kSiteMlpHidden, d->seed_dev), st)) return rc;
            if (int rc = layernorm_bwd(xmid, p.ln2_w, stats2, dh, dcur, dxa, gr.ln2_w, gr.ln2_b, R, D, st, dyb,
                                       make_drop(d->drop_p, d->seed, site + kSiteAttnOut, d->seed_dev), gr.b_out)) return rc;
        } else {
        if (int rc = gemm_wgrad_bf16(dyb, g, gr.w2, R, D, M, st)) return rc;
        GemmBf16Args a = gemm_args(dyb, w.w2T, R, M, D, du, 0);        // du = (dy . W2) * gelu'(u) * hidden-dropout
        a.aux = u; a.act = 2; a.drop = make_drop(d->drop_p, d->seed, site + kSiteMlpHidden, d->seed_dev);
        const bool fuse_db1 = M <= 64 && M % 4 == 0;      // db1 = column sums of du, from the same epilogue
        if (fuse_db1) a.colsum = gr.b1;
        if (int rc = gemm_tn_bf16(a, st)) return rc;
        if (!fuse_db1) { if (int rc = cast_rows_bf16(du, nullptr, gr.b1, R, M, none, st)) return rc; }
        if (int rc = gemm_wgrad_bf16(du, (const bf16*)(lw + L.o_h2), gr.w1, R, M, D, st)) return rc;
        // LN2 backward -> dxa (fp32) + fused: dyb = bf16(dropout_attn_out(dxa)), db_out += colsum.  With fuse_lnb the LayerNorm
        // backward runs in the epilogue of the data-gradient GEMM that produces its dy (no [R,D] fp32 round trip, one launch less)
        if (fuse_lnb) {
            GemmBf16Args b = gemm_args(du, w.w1T, R, D, M, dxa, 1);
            b.residual = dcur; b.ln_w = p.ln2_w; b.lnb_x = xmid; b.lnb_stats = stats2; b.lnb_dw = gr.ln2_w; b.lnb_db = gr.ln2_b;
            b.lnb_cast = dyb; b.lnb_colsum = gr.b_out; b.drop = make_drop(d->drop_p, d->seed, site + kSiteAttnOut, d->seed_dev);
            if (int rc = gemm_tn_bf16(b, st)) return rc;
        } else {
            if (int rc = gemm_tn_bf16(gemm_args(du, w.w1T, R, D, M, dh, 1), st)) return rc;
            if (int rc = layernorm_bwd(xmid, p.ln2_w, stats2, dh, dcur, dxa, gr.ln2_w, gr.ln2_b, R, D, st, dyb,
                                       make_drop(d->drop_p, d->seed, site + kSiteAttnOut, d->seed_dev), gr.b_out)) return rc;
        }
        }
        // ---- attention branch ----
        if (int rc = gemm_wgrad_bf16(dyb, o, gr.w_out, R, D, I, st)) return rc;
        if (int rc = gemm_tn_bf16(gemm_args(dyb, w.woT, R, I, D, dO, 0), st)) return rc;
        msst_attn_dims ad{d->n_seq, d->N, d->inner, d->H, d->dh, d->drop_p, d->seed, site + kSiteAttnProb, d->prec, d->seed_dev};
        if (fused) {   // q/k/v recomputed from h1 inside the kernel, which also produces dh = dqkv . Wqkv (no data-gradient GEMM)
            AttnGeom ag;
            if (int rc = make_attn_geom(&ad, ag, false)) return rc;
            if (int rc = attn_block_bwd(ag, D, (const bf16*)(lw + L.o_h1), w.wq, w.wqT, dO, lse, dqkv, dh,
                                        make_drop(d->drop_p, d->seed, site + kSiteAttnProb, d->seed_dev), st)) return rc;
        } else {
            if (int rc = attention_bwd_bf16(&ad, qkv, o, lse, dO, dqkv, st)) return rc;
        }
        if (int rc = gemm_wgrad_bf16(dqkv, (const bf16*)(lw + L.o_h1), gr.w_qkv, R, 3 * I, D, st)) return rc;
        float* dx = (l == 0) ? d_x_in : dxb;
        if (fuse_lnb && !fused) {   // LN1 backward in the epilogue of the Wqkv data-gradient GEMM (+ the cast for layer l-1's MLP branch)
            GemmBf16Args b = gemm_args(dqkv, w.wqT, R, D, 3 * I, dx, 1);
            b.residual = dxa; b.ln_w = p.ln1_w; b.lnb_x = x; b.lnb_stats = stats1; b.lnb_dw = gr.ln1_w; b.lnb_db = gr.ln1_b;
            if (l > 0) {
                b.lnb_cast = dyb; b.lnb_colsum = grads[l - 1].b2; b.drop = make_drop(d->drop_p, d->seed, site - 8u + kSiteMlpOut, d->seed_dev);
                dyb_ready = true;
            }
            if (int rc = gemm_tn_bf16(b, st)) return rc;
            dcur = dx;
            continue;
        }
        if (!fused) { if (int rc = gemm_tn_bf16(gemm_args(dqkv, w.wqT, R, D, 3 * I, dh, 1), st)) return rc; }
        // LN1 backward -> dx (fp32) + fused for the next iteration (layer l-1): dyb = bf16(dropout_mlp_out(dx)), db2(l-1)
        if (l > 0) {
            if (int rc = layernorm_bwd(x, p.ln1_w, stats1, dh, dxa, dx, gr.ln1_w, gr.ln1_b, R, D, st, dyb,
                                       make_drop(d->drop_p, d->seed, site - 8u + kSiteMlpOut, d->seed_dev), grads[l - 1].b2)) return rc;
            dyb_ready = true;
        } else {
            if (int rc = layernorm_bwd(x, p.ln1_w, stats1, dh, dxa, dx, gr.ln1_w, gr.ln1_b, R, D, st)) return rc;
        }
        dcur = dx;
    }
    return MSST_OK;
}

}  // namespace msst
using namespace msst;

extern "C" int64_t msst_transformer_workspace_bytes(const msst_tf_dims* d) {
    if (check_dims(d)) return -1;
    return (int64_t)make_layout(d).total;
}

extern "C" int msst_transformer_fwd(const msst_tf_dims* d, const msst_layer_params* layers, const float* x_in, float* x_out,
                                    void* workspace, msst_stream_t stream) {
    if (int rc = check_dims(d)) return rc;
    MSST_REQUIRE(layers && x_in && x_out && workspace, "transformer_fwd: null pointer");
    if (d->prec == MSST_PREC_BF16) return tf_fwd_bf16(d, layers, x_in, x_out, (char*)workspace, (cudaStream_t)stream);
    const TfLayout L = make_layout(d);
    cudaStream_t st = (cudaStream_t)stream;
    char* ws = (char*)workspace;
    const int64_t R = L.R;
    const int D = d->D, I = L.I, M = d->M;
    float* h = (float*)(ws + L.s_h);
    const float* x = x_in;
    for (int l = 0; l < d->L; ++l) {
        char* lw = ws + L.layer_bytes * (d->save_for_backward ? l : 0);
        const msst_layer_params& p = layers[l];
        float* stats1 = (float*)(lw + L.o_stats1); float* stats2 = (float*)(lw + L.o_stats2);
        float* qkv = (float*)(lw + L.o_qkv); float* o = (float*)(lw + L.o_o); float* lse = (float*)(lw + L.o_lse);
        float* xmid = (float*)(lw + L.o_xmid); float* u = (float*)(lw + L.o_u); float* g = (float*)(lw + L.o_g);
        float* y = (l == d->L - 1) ? x_out : (float*)(lw + L.o_xout);
        const uint32_t site = d->site_base + 8u * l;
        const Drop none = make_drop(0.f, 0, 0);
        if (int rc = layernorm_fwd(x, p.ln1_w, p.ln1_b, h, 0, stats1, R, D, 1e-5f, st)) return rc;
        if (int rc = linear_fwd_f32(h, p.w_qkv, nullptr, nullptr, qkv, nullptr, R, 3 * I, D, 0, none, st)) return rc;
        msst_attn_dims ad{d->n_seq, d->N, d->inner, d->H, d->dh, d->drop_p, d->seed, site + kSiteAttnProb, d->prec, d->seed_dev};
        if (int rc = attention_fwd_f32(&ad, qkv, o, lse, st)) return rc;
        if (int rc = linear_fwd_f32(o, p.w_out, p.b_out, x, xmid, nullptr, R, D, I, 0, make_drop(d->drop_p, d->seed, site + kSiteAttnOut, d->seed_dev), st)) return rc;
        if (int rc = layernorm_fwd(xmid, p.ln2_w, p.ln2_b, h, 0, stats2, R, D, 1e-5f, st)) return rc;
        if (int rc = linear_fwd_f32(h, p.w1, p.b1, nullptr, g, u, R, M, D, 1, make_drop(d->drop_p, d->seed, site + kSiteMlpHidden, d->seed_dev), st)) return rc;
        if (int rc = linear_fwd_f32(g, p.w2, p.b2, xmid, y, nullptr, R, D, M, 0, make_drop(d->drop_p, d->seed, site + kSiteMlpOut, d->seed_dev), st)) return rc;
        x = y;
    }
    return MSST_OK;
}

extern "C" int msst_transformer_bwd(const msst_tf_dims* d, const msst_layer_params* layers, const msst_layer_grads* grads,
                                    const float* x_in, const float* d_x_out, float* d_x_in, void* workspace,
                                    msst_stream_t stream) {
    if (int rc = check_dims(d)) return rc;
    MSST_REQUIRE(d->save_for_backward, "transformer_bwd: forward was not run with save_for_backward");
    MSST_REQUIRE(layers && grads && x_in && d_x_out && d_x_in && workspace, "transformer_bwd: null pointer");
    if (d->prec == MSST_PREC_BF16) return tf_bwd_bf16(d, layers, grads, x_in, d_x_out, d_x_in, (char*)workspace, (cudaStream_t)stream);
    const TfLayout L = make_layout(d);
    cudaStream_t st = (cudaStream_t)stream;
    char* ws = (char*)workspace;
    const int64_t R = L.R;
    const int D = d->D, I = L.I, M = d->M;
    float* h = (float*)(ws + L.s_h); float* dqkv = (float*)(ws + L.s_dqkv); float* dO = (float*)(ws + L.s_do);
    float* du = (float*)(ws + L.s_du); float* dh = (float*)(ws + L.s_dh); float* dyb = (float*)(ws + L.s_dy);
    float* dxa = (float*)(ws + L.s_dxa); float* dxb = (float*)(ws + L.s_dxb);
    const float* dcur = d_x_out;
    const Drop none = make_drop(0.f, 0, 0);
    for (int l = d->L - 1; l >= 0; --l) {
        char* lw = ws + L.layer_bytes * l;
        const msst_layer_params& p = layers[l];
        const msst_layer_grads& gr = grads[l];
        float* stats1 = (float*)(lw + L.o_stats1); float* stats2 = (float*)(lw + L.o_stats2);
        float* qkv = (float*)(lw + L.o_qkv); float* o = (float*)(lw + L.o_o); float* lse = (float*)(lw + L.o_lse);
        float* xmid = (float*)(lw + L.o_xmid); float* u = (float*)(lw + L.o_u); float* g = (float*)(lw + L.o_g);
        const float* x = (l == 0) ? x_in : (const float*)(ws + L.layer_bytes * (l - 1) + L.o_xout);
        const uint32_t site = d->site_base + 8u * l;
        // ---- MLP branch: y = xmid + drop(W2 g + b2) ----
        const float* dy = dcur;
        if (d->drop_p > 0.f) {
            if (int rc = dropout_apply_f32(dcur, dyb, R * D, make_drop(d->drop_p, d->seed, site + kSiteMlpOut, d->seed_dev), st)) return rc;
            dy = dyb;
        }
        if (int rc = linear_bwd_weight_f32(dy, g, gr.w2, gr.b2, R, D, M, st)) return rc;
        if (int rc = linear_bwd_data_f32(dy, p.w2, u, nullptr, du, R, D, M, make_drop(d->drop_p, d->seed, site + kSiteMlpHidden, d->seed_dev), st)) return rc;
        if (int rc = layernorm_fwd(xmid, p.ln2_w, p.ln2_b, h, 0, nullptr, R, D, 1e-5f, st)) return rc;
        if (int rc = linear_bwd_weight_f32(du, h, gr.w1, gr.b1, R, M, D, st)) return rc;
        if (int rc = linear_bwd_data_f32(du, p.w1, nullptr, nullptr, dh, R, M, D, none, st)) return rc;
        if (int rc = layernorm_bwd(xmid, p.ln2_w, stats2, dh, dcur, dxa, gr.ln2_w, gr.ln2_b, R, D, st)) return rc;
        // ---- attention branch: xmid = x + drop(Wo o + bo) ----
        dy = dxa;
        if (d->drop_p > 0.f) {
            if (int rc = dropout_apply_f32(dxa, dyb, R * D, make_drop(d->drop_p, d->seed, site + kSiteAttnOut, d->seed_dev), st)) return rc;
            dy = dyb;
        }
        if (int rc = linear_bwd_weight_f32(dy, o, gr.w_out, gr.b_out, R, D, I, st)) return rc;
        if (int rc = linear_bwd_data_f32(dy, p.w_out, nullptr, nullptr, dO, R, D, I, none, st)) return rc;
        msst_attn_dims ad{d->n_seq, d->N, d->inner, d->H, d->dh, d->drop_p, d->seed, site + kSiteAttnProb, d->prec, d->seed_dev};
        if (int rc = attention_bwd_f32(&ad, qkv, o, lse, dO, dqkv, st)) return rc;
        if (int rc = layernorm_fwd(x, p.ln1_w, p.ln1_b, h, 0, nullptr, R, D, 1e-5f, st)) return rc;
        if (int rc = linear_bwd_weight_f32(dqkv, h, gr.w_qkv, nullptr, R, 3 * I, D, st)) return rc;
        if (int rc = linear_bwd_data_f32(dqkv, p.w_qkv, nullptr, nullptr, dh, R, 3 * I, D, none, st)) return rc;
        float* dx = (l == 0) ? d_x_in : dxb;
        if (int rc = layernorm_bwd(x, p.ln1_w, stats1, dh, dxa, dx, gr.ln1_w, gr.ln1_b, R, D, st)) return rc;
        dcur = dx;
    }
    return MSST_OK;
}

// ---- stand-alone entry points (unit tests, microbench) ----
extern "C" int msst_linear_fwd(const msst_linear_dims* d, const void* x, const void* W, const float* bias, const float* residual,
                               void* y, void* pre_act, msst_stream_t stream) {
    MSST_REQUIRE(d, "linear_fwd: null dims");
    MSST_REQUIRE(drop_p_ok(d->drop_p), "linear_fwd: drop_p=%g outside [0, 1]", (double)d->drop_p);
    const Drop drop = make_drop(d->drop_p, d->seed, d->site, d->seed_dev);
    if (d->prec == MSST_PREC_BF16) {
        GemmBf16Args a{(const __nv_bfloat16*)x, (const __nv_bfloat16*)W, d->M, d->N, d->K, bias, residual, y, d->y_fp32,
                       (__nv_bfloat16*)pre_act, nullptr, d->act, drop};
        return gemm_tn_bf16(a, (cudaStream_t)stream);
    }
    return linear_fwd_f32((const float*)x, (const float*)W, bias, residual, (float*)y, (float*)pre_act, d->M, d->N, d->K, d->act,
                          drop, (cudaStream_t)stream);
}
extern "C" int msst_linear_bwd_data(const msst_linear_dims* d, const void* dy, const void* W, const void* pre_act,
                                    const float* dx_add, void* dx, msst_stream_t stream) {
    MSST_REQUIRE(d, "linear_bwd_data: null dims");
    MSST_REQUIRE(drop_p_ok(d->drop_p), "linear_bwd_data: drop_p=%g outside [0, 1]", (double)d->drop_p);
    const Drop drop = make_drop(d->drop_p, d->seed, d->site, d->seed_dev);
    if (d->prec == MSST_PREC_BF16) {   // dx[M,K] = dy[M,N] . (W^T)[K,N]^T
        GemmBf16Args a{(const __nv_bfloat16*)dy, (const __nv_bfloat16*)W, d->M, d->K, d->N, nullptr, dx_add, dx, d->y_fp32,
                       nullptr, (const __nv_bfloat16*)pre_act, pre_act ? 2 : 0, drop};
        return gemm_tn_bf16(a, (cudaStream_t)stream);
    }
    return linear_bwd_data_f32((const float*)dy, (const float*)W, (const float*)pre_act, dx_add, (float*)dx, d->M, d->N, d->K, drop,
                               (cudaStream_t)stream);
}
extern "C" int msst_linear_bwd_weight(const msst_linear_dims* d, const void* dy, const void* x, float* dW, float* db,
                                      msst_stream_t stream) {
    MSST_REQUIRE(d, "linear_bwd_weight: null dims");
    if (d->prec == MSST_PREC_BF16) {
        MSST_REQUIRE(db == nullptr, "linear_bwd_weight: bias gradient is not fused in bf16 mode");
        return gemm_wgrad_bf16((const __nv_bfloat16*)dy, (const __nv_bfloat16*)x, dW, d->M, d->N, d->K, (cudaStream_t)stream);
    }
    return linear_bwd_weight_f32((const float*)dy, (const float*)x, dW, db, d->M, d->N, d->K, (cudaStream_t)stream);
}
extern "C" int msst_attention_fwd(const msst_attn_dims* d, const void* qkv, void* out, float* lse, msst_stream_t stream) {
    MSST_REQUIRE(d, "attention_fwd: null dims");
    if (d->prec == MSST_PREC_BF16) return attention_fwd_bf16(d, (const bf16*)qkv, (bf16*)out, lse, (cudaStream_t)stream);
    return attention_fwd_f32(d, (const float*)qkv, (float*)out, lse, (cudaStream_t)stream);
}
extern "C" int msst_attention_bwd(const msst_attn_dims* d, const void* qkv, const void* out, const float* lse, const void* d_out,
                                  void* d_qkv, msst_stream_t stream) {
    MSST_REQUIRE(d, "attention_bwd: null dims");
    if (d->prec == MSST_PREC_BF16)
        return attention_bwd_bf16(d, (const bf16*)qkv, (const bf16*)out, lse, (const bf16*)d_out, (bf16*)d_qkv, (cudaStream_t)stream);
    return attention_bwd_f32(d, (const float*)qkv, (const float*)out, lse, (const float*)d_out, (float*)d_qkv, (cudaStream_t)stream);
}
extern "C" int msst_attn_block_fwd(const msst_attn_dims* d, int D, const void* h, const void* w_qkv, void* out, float* lse, msst_stream_t stream) {
    MSST_REQUIRE(d && d->prec == MSST_PREC_BF16, "attn_block_fwd: bf16 mode only");
    AttnGeom g;
    if (int rc = make_attn_geom(d, g, false)) return rc;
    if (g.n_seq == 0) return MSST_OK;
    return attn_block_fwd(g, D, (const bf16*)h, (const bf16*)w_qkv, (bf16*)out, lse, make_drop(d->drop_p, d->seed, d->site, d->seed_dev), (cudaStream_t)stream);
}
extern "C" int msst_attn_block_out_fwd(const msst_attn_dims* d, int D, const void* h, const void* w_qkv, void* out, float* lse, const void* w_out,
                                       const float* b_out, const float* x, float* xmid, const float* ln_w, const float* ln_b, void* h2, float* ln_stats,
                                       uint32_t site_out, msst_stream_t stream) {
    MSST_REQUIRE(d && d->prec == MSST_PREC_BF16, "attn_block_out_fwd: bf16 mode only");
    AttnGeom g;
    if (int rc = make_attn_geom(d, g, false)) return rc;
    if (g.n_seq == 0) return MSST_OK;
    const AttnBlockOut t{(const bf16*)w_out, b_out, x, xmid, ln_w, ln_b, (bf16*)h2, ln_stats, make_drop(d->drop_p, d->seed, site_out, d->seed_dev)};
    return attn_block_fwd(g, D, (const bf16*)h, (const bf16*)w_qkv, (bf16*)out, lse, make_drop(d->drop_p, d->seed, d->site, d->seed_dev), (cudaStream_t)stream, &t);
}
extern "C" int msst_attn_block_bwd(const msst_attn_dims* d, int D, const void* h, const void* w_qkv, const void* w_qkv_t, const void* d_out,
                                   const float* lse, void* d_qkv, float* d_h, msst_stream_t stream) {
    MSST_REQUIRE(d && d->prec == MSST_PREC_BF16, "attn_block_bwd: bf16 mode only");
    AttnGeom g;
    if (int rc = make_attn_geom(d, g, false)) return rc;
    if (g.n_seq == 0) return MSST_OK;
    return attn_block_bwd(g, D, (const bf16*)h, (const bf16*)w_qkv, (const bf16*)w_qkv_t, (const bf16*)d_out, lse, (bf16*)d_qkv, d_h,
                          make_drop(d->drop_p, d->seed, d->site, d->seed_dev), (cudaStream_t)stream);
}
extern "C" int msst_mlp_block_fwd(const void* h2, const float* xmid, const void* w1, const void* w2, const float* b1, const float* b2, void* u,
                                  void* g, float* y, const float* ln_w, const float* ln_b, void* h1, float* ln_stats, int64_t R, int D, int M,
                                  float drop_p, uint64_t seed, uint32_t site_hidden, uint32_t site_out, const uint64_t* seed_dev, msst_stream_t stream) {
    MSST_REQUIRE(h2 && xmid && w1 && w2 && b1 && b2 && u && g && y, "mlp_block_fwd: null pointer");
    MSST_REQUIRE(!h1 || (ln_w && ln_b && ln_stats), "mlp_block_fwd: h1 needs ln_w, ln_b and ln_stats");
    MSST_REQUIRE(drop_p_ok(drop_p), "mlp_block_fwd: drop_p=%g outside [0, 1]", (double)drop_p);
    return mlp_block_fwd((const bf16*)h2, xmid, (const bf16*)w1, (const bf16*)w2, b1, b2, (bf16*)u, (bf16*)g, y, ln_w, ln_b, (bf16*)h1, ln_stats, R, D, M,
                         make_drop(drop_p, seed, site_hidden, seed_dev), make_drop(drop_p, seed, site_out, seed_dev), (cudaStream_t)stream);
}
extern "C" int msst_mlp_block_bwd(const void* dyb, const void* u, const void* g, const void* h2, const void* w2_t, const void* w1_t, float* d_w1,
                                  float* d_w2, float* d_b1, float* d_h, int64_t R, int D, int M, float drop_p, uint64_t seed, uint32_t site_hidden,
                                  const uint64_t* seed_dev, msst_stream_t stream) {
    MSST_REQUIRE(dyb && u && g && h2 && w2_t && w1_t && d_w1 && d_w2 && d_b1 && d_h, "mlp_block_bwd: null pointer");
    MSST_REQUIRE(drop_p_ok(drop_p), "mlp_block_bwd: drop_p=%g outside [0, 1]", (double)drop_p);
    return mlp_block_bwd((const bf16*)dyb, (const bf16*)u, (const bf16*)g, (const bf16*)h2, (const bf16*)w2_t, (const bf16*)w1_t, d_w1, d_w2, d_b1, d_h,
                         R, D, M, make_drop(drop_p, seed, site_hidden, seed_dev), (cudaStream_t)stream);
}
extern "C" int msst_dropout_apply(const float* x, float* y, int64_t n, float p, uint64_t seed, uint32_t site,
                                  const uint64_t* seed_dev, msst_stream_t stream) {
    MSST_REQUIRE(drop_p_ok(p), "dropout_apply: p=%g outside [0, 1]", (double)p);
    return dropout_apply_f32(x, y, n, make_drop(p, seed, site, seed_dev), (cudaStream_t)stream);
}
