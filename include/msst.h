/* msst.h -- C ABI of the B200-native MaskedSST hot path (libmsst.so).
 *
 * The upstream project (HSG-AIML/MaskedSST) is pure Python/PyTorch: it has no FFI of its own, so the
 * drop-in boundary is the nn.Module surface of src/vit_spatial_spectral.py / src/vit_simmim_original.py
 * (mirrored by maskedsst_b200/ and the `src/` alias package).  Below that surface every arithmetic
 * step is one of the entry points declared here; each cites the reference code (file:line relative to
 * the upstream repo) whose arithmetic it replaces.
 *
 * Conventions
 *   - all pointers are DEVICE pointers unless the name ends in _host; fp32 unless stated
 *   - every function is asynchronous on `stream` (a cudaStream_t passed as void*), never synchronises
 *     the device, allocates nothing, and is CUDA-graph capturable
 *   - return value: 0 = ok, otherwise an MSST_ERR_* code; msst_last_error() gives the message
 *   - token order t = c*S + s (spectral block major), patch vector order (p0 p1 p2), qkv rows q|k|v each
 *     head-major (h d)  -- reference vit_spatial_spectral.py:198,218,68-69 (SURVEY.md C18)
 *   - dropout masks are never stored: (seed, site, element index) -> counter hash (lowbias32, 16-bit lanes); p = 0 disables;
 *     `seed_dev` (optional device uint64) is added to the seed so a captured CUDA graph draws fresh masks per replay.
 *     An element is kept iff its 16-bit lane >= floor(p * 2^32) >> 16, so p is resolved to 2^-16: a p below 2^-16 drops
 *     nothing but still scales by 1/(1-p).  p = 1 drops everything (factor 0, as nn.Dropout(1.0)).  A p outside [0, 1],
 *     NaN included, is MSST_ERR_ARG before any launch.
 */
#ifndef MSST_H_
#define MSST_H_
#if defined(__GNUC__)
#define MSST_API __attribute__((visibility("default")))
#else
#define MSST_API
#endif
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define MSST_OK 0
#define MSST_ERR_ARG 1      /* unsupported shape / bad argument */
#define MSST_ERR_CUDA 2     /* a CUDA runtime call or launch failed */

#define MSST_PREC_FP32 0    /* FFMA everywhere; parity target rel-err <= 1e-5 */
#define MSST_PREC_BF16 1    /* tcgen05 bf16 operands, fp32 accumulate / residual stream / statistics */

typedef void* msst_stream_t;

MSST_API const char* msst_last_error(void);
MSST_API int msst_version(void);
/* number of kernels this library has launched in this process (bench.py reports it as gpu_launches) */
MSST_API long long msst_launch_count(void);

/* ---------------------------------------------------------------------------------------------
 * (1) fused patch embedding.  Replaces BlockwisePatchEmbedding.to_patch/.embed
 *     (vit_spatial_spectral.py:197-229), PatchEmbed (:232-253, n_weight_blocks = 1), the pos-embed add
 *     (:522-528 / vit_simmim_original.py:236-242), emb-dropout (:530) and the SimMIM mask-token
 *     substitution (vit_simmim_original.py:245-249,285).
 *       img      [B, C*p0, G*p1, G*p1]  NCHW cube
 *       pos      [T, D] positional rows (learned table rows [0,T) or the materialised sincos cat)
 *       mask     [B, T] uint8 or NULL; mask_token [D] or NULL
 *       tokens   [B, T, D] out
 *       patches_ln [B,T,P] optional out: pre-norm'ed patches (PatchEmbed SimMIM target, C6), or NULL
 * ------------------------------------------------------------------------------------------- */
/* Optional RAW input: the cube is read from sensor tiles with the reference's input pipeline applied on the fly inside
 * the patch-embedding and decoder kernels (no fp32 cube in HBM; the host ships int16).  Replaces, per pixel:
 *   (raw - means[band]) / stds[band] in float64 -> fp32   StandardizeEnMAP.__call__ / StandardizeHouston2018.__call__ + ToTensor
 *                                                         (src/data_enmap.py:454-457,517-522; src/data_houston2018.py:442-445)
 *   torch.clip(img, clip_lo, clip_hi) of the standardised value (src/data_enmap.py:303-304), when clip != 0
 *   zero bands raw_bands .. C*p0-1                        (Houston 48 -> 50: F.pad, src/data_houston2018.py:268-269)
 *   img[:, :, y0:y0+H, x0:x0+W], one window for the batch (pretrain.py:99-107)
 * When `raw` is set in the dims struct the `img` argument of the entry point is ignored (may be NULL). */
enum { MSST_RAW_I16 = 0, MSST_RAW_U16 = 1, MSST_RAW_F32 = 2 };
typedef struct {
    const void* tiles;           /* device [B, raw_bands, tile_h, tile_w], element type `dtype` */
    int dtype;                   /* MSST_RAW_* */
    int raw_bands;               /* <= C*p0; model bands beyond it are zero */
    int tile_h, tile_w;
    int y0, x0;                  /* crop window origin inside the tile */
    const double* mean;          /* device [raw_bands] float64 */
    const double* std;           /* device [raw_bands] float64 */
    int clip; float clip_lo, clip_hi;
    int win_y, win_x;            /* 0 / 1: one crop window per tile (above).  > 1: whole-tile sliding-window inference (notebook cell 13,
                                    src/utils.py:477-605): the windows of all tiles are consecutive samples, never copied out of the tile */
    int stride_y, stride_x;      /* window step in pixels, 1 <= stride <= window; 0 = the window size (non-overlapping) */
    int win_first;               /* global index of the first window this launch reads (0: the first window of tile 0) */
    /* Sample b is global window g = win_first + b: window w = g % (win_y*win_x) of tile g / (win_y*win_x), origin
     *   oy = y0 + min((w / win_x) * stride_y, tile_h - y0 - H),   ox = x0 + min((w % win_x) * stride_x, tile_w - x0 - W)
     * so a last window row / column that would cross the tile border is snapped flush to it. */
} msst_raw_input;

typedef struct {
    int B, C, G, p0, p1, D;      /* G = spatial patches per side, P = p0*p1*p1, S = G*G, T = C*S */
    int n_weight_blocks;         /* C for blockwise embedding, 1 for PatchEmbed */
    float drop_p; uint64_t seed; /* emb-dropout (encoder.forward path only) */
    const uint64_t* seed_dev;    /* optional device u64 added to seed (fresh masks per CUDA-graph replay); may be NULL */
    const msst_raw_input* raw;   /* optional (host pointer): read pixels from raw tiles instead of `img`; may be NULL */
} msst_embed_dims;

MSST_API int msst_patch_embed_fwd(const msst_embed_dims* d, const float* img, const float* pre_w, const float* pre_b,
                         const float* W /*[nb,D,P]*/, const float* bias /*[nb,D]*/, const float* post_w,
                         const float* post_b, const float* pos, const uint8_t* mask, const float* mask_token,
                         float* tokens, float* patches_ln, msst_stream_t stream);
/* grads ACCUMULATE (+=) into d_* (caller zeroes); d_pos [T,D]; d_mask_token may be NULL */
MSST_API int msst_patch_embed_bwd(const msst_embed_dims* d, const float* img, const float* pre_w, const float* pre_b,
                         const float* W, const float* bias, const float* post_w, const float* post_b,
                         const uint8_t* mask, const float* d_tokens, const float* d_patches_ln /*or NULL*/,
                         float* d_pre_w, float* d_pre_b, float* d_W, float* d_bias, float* d_post_w,
                         float* d_post_b, float* d_pos, float* d_mask_token, msst_stream_t stream);
/* Data gradient of the same map: d_img [B, C*p0, G*p1, G*p1] fp32 = d(tokens, patches_ln) / d(img) applied to d_tokens [B,T,D] and
 * d_patches_ln [B,T,P] (or NULL), for the fp32 cube `img`.  Per token: g_o = d_tokens * emb-dropout factor (0 when the token is
 * masked: mask-token select), g_z = LN_D'(g_o * post_w), g_h = W_blk^T g_z + d_patches_ln (which still flows for masked tokens),
 * g_x = LN_P'(g_h * pre_w), written to the patch's pixels.  Patches tile the image: every element of d_img is written exactly once
 * (plain stores, bitwise deterministic; the caller need not zero it).  No parameter gradient is formed (msst_patch_embed_bwd).
 * D in {32, 64, 96, 128}, P <= 64, n_weight_blocks in {1, C}, drop_p in [0, 1], d->raw == NULL (raw tiles have no gradient),
 * img / d_tokens / d_img non-NULL; MSST_ERR_ARG before any launch otherwise, d_img untouched. */
MSST_API int msst_patch_embed_bwd_data(const msst_embed_dims* d, const float* img, const float* pre_w, const float* pre_b,
                                       const float* W, const float* bias, const float* post_w, const float* post_b,
                                       const uint8_t* mask, const float* d_tokens, const float* d_patches_ln /*or NULL*/,
                                       float* d_img, msst_stream_t stream);

/* ---------------------------------------------------------------------------------------------
 * (4) LayerNorm (nn.LayerNorm, biased variance, eps inside sqrt; PreNorm vit_spatial_spectral.py:22-29)
 *     stats [rows,2] = (mean, rstd).  y may be fp32 or bf16 (y_bf16 != 0).
 * ------------------------------------------------------------------------------------------- */
MSST_API int msst_layernorm_fwd(const float* x, const float* w, const float* b, void* y, int y_bf16, float* stats,
                       int64_t rows, int D, float eps, msst_stream_t stream);
/* dx = (accumulate ? dx_add : 0) + LN'(dy); dw/db accumulate */
MSST_API int msst_layernorm_bwd(const float* x, const float* w, const float* stats, const float* dy, const float* dx_add,
                       float* dx, float* dw, float* db, int64_t rows, int D, msst_stream_t stream);

/* ---------------------------------------------------------------------------------------------
 * (2) linear layers.  y = epilogue(x @ W^T).  Replaces nn.Linear call sites to_qkv / to_out / net.0 /
 *     net.3 (vit_spatial_spectral.py:35-41,59-65) with fused bias, GELU(erf), dropout, residual.
 *       x [M,K] (ldx), W [N,K], y [M,N] (ldy), residual [M,N] (ldy) or NULL, pre_act [M,N] optional out
 *     order: t = xW^T + bias; pre_act = t; t = act(t); t = dropout(t); y = t + residual
 *     prec = MSST_PREC_BF16 (tcgen05 path): x, W, pre_act are bf16; bias / residual fp32; y bf16 or fp32 (y_fp32);
 *     K % 8 == 0.  In that mode msst_linear_bwd_data takes dy bf16, W = the TRANSPOSED bf16 copy W^T [K,N], pre_act bf16,
 *     dx bf16/fp32 (y_fp32); msst_linear_bwd_weight takes dy, x bf16 and accumulates fp32 dW (db must be NULL).
 * ------------------------------------------------------------------------------------------- */
typedef struct {
    int64_t M; int N, K;
    int act;                       /* 0 none, 1 GELU(erf) */
    float drop_p; uint64_t seed; uint32_t site;
    int prec;
    const uint64_t* seed_dev;
    int y_fp32;                    /* BF16 mode only: 1 = the output (y / dx) is fp32, 0 = bf16 */
} msst_linear_dims;
MSST_API int msst_linear_fwd(const msst_linear_dims* d, const void* x, const void* W, const float* bias,
                    const float* residual, void* y, void* pre_act, msst_stream_t stream);
/* dx = epilogue(dy @ W).  With pre_act != NULL the output is multiplied by gelu'(pre_act) and by the hidden
 * dropout factor of (seed, site) -- i.e. the backward of  g = dropout(gelu(u))  fused into the data-gradient GEMM of
 * the following layer; then + dx_add (optional).  Output-dropout sites are applied to dy beforehand with
 * msst_dropout_apply (same (seed, site) => same mask as the forward). */
MSST_API int msst_linear_bwd_data(const msst_linear_dims* d, const void* dy, const void* W, const void* pre_act,
                         const float* dx_add, void* dx, msst_stream_t stream);
/* dW += dy^T x, db += colsum(dy)  (db may be NULL) */
MSST_API int msst_linear_bwd_weight(const msst_linear_dims* d, const void* dy, const void* x, float* dW, float* db,
                           msst_stream_t stream);

/* y = x * dropout_factor(seed, site, element index), n % 4 == 0 (inverted dropout, nn.Dropout call sites
 * vit_spatial_spectral.py:38,40,57,62,391) */
MSST_API int msst_dropout_apply(const float* x, float* y, int64_t n, float p, uint64_t seed, uint32_t site,
                                const uint64_t* seed_dev, msst_stream_t stream);

/* ---------------------------------------------------------------------------------------------
 * (3) fused attention.  softmax(q k^T * dh^-0.5) v per (sequence, head), flash-style (scores never
 *     reach HBM).  Replaces Attention.forward :69-77.  Rows of sequence s, position i live at
 *       row = (s / inner) * N * inner + (s % inner) + i * inner
 *     so the spectral transformer (sequences of C tokens strided by S) needs no transpose copy
 *     (reference Rearrange copies, vit_spatial_spectral.py:418-430).
 *       qkv [R, 3*H*dh], out [R, H*dh], lse [R, H]  (R = n_seq * N)
 * ------------------------------------------------------------------------------------------- */
typedef struct {
    int64_t n_seq; int N, inner, H, dh;
    float drop_p; uint64_t seed; uint32_t site;
    int prec;
    const uint64_t* seed_dev;
} msst_attn_dims;
MSST_API int msst_attention_fwd(const msst_attn_dims* d, const void* qkv, void* out, float* lse, msst_stream_t stream);
MSST_API int msst_attention_bwd(const msst_attn_dims* d, const void* qkv, const void* out, const float* lse,
                       const void* d_out, void* d_qkv, msst_stream_t stream);

/* Fused projection + attention (bf16 / tcgen05 only; N <= 64, dh = 64, D in {32, 64, 96, 128}): Attention.forward
 * vit_spatial_spectral.py:67-77 INCLUDING to_qkv (:59,68) in one kernel -- q, k, v never reach HBM.
 *   h [R, D] bf16 = the pre-norm output, w_qkv [3*H*dh, D] bf16 (reference layout of to_qkv.weight), out [R, H*dh] bf16, lse [R, H]
 * Backward recomputes q, k, v from h and returns d_qkv [R, 3*H*dh] bf16 (input of the weight gradient dW = d_qkv^T h) and
 * d_h [R, D] fp32 = d_qkv . w_qkv (w_qkv_t = the transposed copy [D, 3*H*dh] bf16). */
MSST_API int msst_attn_block_fwd(const msst_attn_dims* d, int D, const void* h, const void* w_qkv, void* out, float* lse,
                                 msst_stream_t stream);
/* The same forward kernel with the tail of the attention block folded in (Attention.to_out vit_spatial_spectral.py:62-65,77, the
 * residual add of Transformer.forward :102 and the FeedForward PreNorm :25-29):
 *   xmid [R, D] fp32 = x + dropout(out . w_out^T + b_out)   (w_out [D, H*dh] bf16, b_out [D], x [R, D] fp32; dropout site `site_out`,
 *                                                             probability / seed of `d`)
 *   h2 [R, D] bf16 = LayerNorm(xmid; ln_w, ln_b),  ln_stats [R, 2] = (mean, rstd)
 * `out` may be NULL when the attention output itself is not needed (inference). */
MSST_API int msst_attn_block_out_fwd(const msst_attn_dims* d, int D, const void* h, const void* w_qkv, void* out, float* lse,
                                     const void* w_out, const float* b_out, const float* x, float* xmid, const float* ln_w,
                                     const float* ln_b, void* h2, float* ln_stats, uint32_t site_out, msst_stream_t stream);
MSST_API int msst_attn_block_bwd(const msst_attn_dims* d, int D, const void* h, const void* w_qkv, const void* w_qkv_t,
                                 const void* d_out, const float* lse, void* d_qkv, float* d_h, msst_stream_t stream);

/* Fused FeedForward block (bf16 / tcgen05 only; mlp_dim = 64, D in {32, 64, 96}): FeedForward.forward vit_spatial_spectral.py:35-44 +
 * the residual add (:103) + the next layer's pre-norm (:25-29) in one kernel; the hidden activation goes from the first to the second
 * GEMM through shared memory.   h2 [R,D] bf16 (the pre-norm output), xmid [R,D] fp32 (residual), w1 [64,D] / w2 [D,64] bf16,
 * outputs u (pre-GELU) and g = dropout(gelu(u)) [R,64] bf16 (saved for the backward), y [R,D] fp32, and -- when h1 != NULL --
 * h1 = LayerNorm(y; ln_w, ln_b) bf16 with ln_stats [R,2] = (mean, rstd).  Dropout sites: site_hidden on g, site_out on the branch output. */
MSST_API int msst_mlp_block_fwd(const void* h2, const float* xmid, const void* w1, const void* w2, const float* b1, const float* b2,
                                void* u, void* g, float* y, const float* ln_w, const float* ln_b, void* h1, float* ln_stats,
                                int64_t R, int D, int M, float drop_p, uint64_t seed, uint32_t site_hidden, uint32_t site_out,
                                const uint64_t* seed_dev, msst_stream_t stream);
/* Backward of the block (autograd of FeedForward.forward :35-44) in one kernel: dyb [R,D] bf16 = the branch-output gradient after the
 * output dropout, u / g as saved by the forward, h2 the block's input, w2_t = W2^T [64,D] and w1_t = W1^T [D,64] bf16.
 * du = (dyb W2) * gelu'(u) * hidden-dropout stays on the SM;  d_w1 [64,D] += du^T h2,  d_w2 [D,64] += dyb^T g,  d_b1 [64] += colsum(du)
 * (fp32, accumulated in TMEM over the launch),  d_h [R,D] fp32 = du W1 (the gradient w.r.t. h2). */
MSST_API int msst_mlp_block_bwd(const void* dyb, const void* u, const void* g, const void* h2, const void* w2_t, const void* w1_t,
                                float* d_w1, float* d_w2, float* d_b1, float* d_h, int64_t R, int D, int M, float drop_p, uint64_t seed,
                                uint32_t site_hidden, const uint64_t* seed_dev, msst_stream_t stream);

/* ---------------------------------------------------------------------------------------------
 * Transformer stack: L x { x = attn(LN(x)) + x ; x = ff(LN(x)) + x }  (Transformer.forward :100-104),
 * all launches of one stack issued from native code.  Parameter pointers per layer, in reference
 * state_dict order.  workspace holds what backward needs (see msst_transformer_workspace_bytes).
 * ------------------------------------------------------------------------------------------- */
typedef struct {
    const float *ln1_w, *ln1_b, *w_qkv, *w_out, *b_out, *ln2_w, *ln2_b, *w1, *b1, *w2, *b2;
} msst_layer_params;
typedef struct {
    float *ln1_w, *ln1_b, *w_qkv, *w_out, *b_out, *ln2_w, *ln2_b, *w1, *b1, *w2, *b2;
} msst_layer_grads;
typedef struct {
    int64_t n_seq; int N, inner;       /* sequence geometry (see attention) */
    int D, H, dh, M, L;
    float drop_p; uint64_t seed; uint32_t site_base;
    int prec;
    int save_for_backward;             /* 0: inference, workspace only needs scratch */
    const uint64_t* seed_dev;
} msst_tf_dims;
MSST_API int64_t msst_transformer_workspace_bytes(const msst_tf_dims* d);
MSST_API int msst_transformer_fwd(const msst_tf_dims* d, const msst_layer_params* layers, const float* x_in, float* x_out,
                         void* workspace, msst_stream_t stream);
/* d_x_in = grad wrt x_in; parameter grads accumulate. Needs the workspace written by the matching fwd. */
MSST_API int msst_transformer_bwd(const msst_tf_dims* d, const msst_layer_params* layers, const msst_layer_grads* grads,
                         const float* x_in, const float* d_x_out, float* d_x_in, void* workspace,
                         msst_stream_t stream);

/* ---------------------------------------------------------------------------------------------
 * Classification head: mean over spectral blocks, LN, Linear, 'b h w (p1 p2 nc) -> b nc (h p1)(w p2)'
 * (vit_spatial_spectral.py:550-562, 481-493).  x [B, C*S, D] -> logits [B, nc, G*p1, G*p1].
 * ------------------------------------------------------------------------------------------- */
typedef struct { int B, C, G, p1, D, nc; } msst_head_dims;
MSST_API int msst_head_fwd(const msst_head_dims* d, const float* x, const float* ln_w, const float* ln_b, const float* W,
                  const float* bias, float* logits, msst_stream_t stream);
MSST_API int msst_head_bwd(const msst_head_dims* d, const float* x, const float* ln_w, const float* ln_b, const float* W,
                  const float* d_logits, float* d_x, float* d_ln_w, float* d_ln_b, float* d_W, float* d_bias,
                  msst_stream_t stream);
/* nn.CrossEntropyLoss(ignore_index) over [B,nc,H,W] logits (finetune.py:136): loss_sum_count[0] = sum of
 * NLL over valid pixels, [1] = number of valid pixels (so data-parallel ranks can all-reduce both, §8(e));
 * d_logits = softmax - onehot for valid pixels, 0 otherwise (UNSCALED: caller divides by the count).
 * A pixel is valid when its label is in [0, nc) and != ignore_index.  A label outside [0, nc) is SKIPPED like ignore_index
 * (no loss, not counted, zero gradient), where torch's cross_entropy raises an error. */
MSST_API int msst_cross_entropy_fwd_bwd(const float* logits, const int64_t* labels, int B, int nc, int HW, int ignore_index,
                               float* loss_sum_count, float* d_logits, msst_stream_t stream);

/* ---------------------------------------------------------------------------------------------
 * Whole-scene inference: blend overlapping window predictions into the scene (the usual fix for the seams of
 * window-by-window classification).  Windows are laid out as in msst_raw_input with y0 = x0 = 0 and the scene as the tile:
 * global window g is window g % (win_y*win_x) of scene g / (win_y*win_x), origins stepped by (stride_y, stride_x), the
 * last row / column snapped to the border.  One call blends the chunk of windows [win_first, win_first + n):
 *   logits [n, nc, win, win]   the chunk's head output (as msst_head_fwd writes it), read in place
 *   weight [win, win] or NULL  per-window-pixel weight (NULL: 1)
 *   acc  [B, nc, H, W] +=  weight * softmax_nc(logits)   summed over the chunk's windows covering the pixel
 *   wsum [B, H, W]     +=  weight
 * Deterministic: every scene pixel is owned by one thread that adds its windows in ascending g (acc = acc + c, no atomics),
 * so the result is bitwise the same for any chunking as long as chunks are issued in ascending order.  Only the scene rows
 * the chunk touches are visited.  1 <= stride <= win <= H, W;  win_y <= ceil((H - win) / stride_y) + 1 (ditto x); nc <= 256.
 * ------------------------------------------------------------------------------------------- */
typedef struct {
    int B, nc, H, W;             /* scenes, classes, scene rows / columns */
    int win, stride_y, stride_x; /* square window side, window step */
    int win_y, win_x;            /* windows per scene column / row */
    int win_first, n;            /* this chunk: global windows [win_first, win_first + n) */
} msst_scene_dims;
MSST_API int msst_scene_blend(const msst_scene_dims* d, const float* logits, const float* weight, float* acc, float* wsum,
                              msst_stream_t stream);
/* Whole-scene embedding maps: the same windows, chunks, weight and ownership contract as msst_scene_blend, but each covering window
 * contributes its encoder feature at the pixel instead of class probabilities.  One call blends the chunk [win_first, win_first + n):
 *   tokens [n, C*S, D]         the chunk's forward_features output (fp32, t = c*S + s, S = G*G, G = win / p1), read in place
 *   weight [win, win] or NULL  per-window-pixel weight (NULL: 1)
 *   f(y, x) = (1/C) sum_c tokens[g - win_first, c*S + s, :],  s = ((y - oy) / p1) * G + (x - ox) / p1   ((oy, ox): origin of window g)
 *              -- the spectral mean the default head normalises (vit_spatial_spectral.py:550-553), repeated over the p1 x p1 pixels
 *              of each spatial patch
 *   acc  [B, D, H, W] +=  weight * f                   summed over the chunk's windows covering the pixel, ascending g
 *   wsum [B, H, W]    +=  weight
 * Bitwise independent of the chunking (chunks in ascending order); only the scene rows the chunk touches are visited.
 * 1 <= stride <= win <= H, W;  win_y <= ceil((H - win) / stride_y) + 1 (ditto x);  D <= 256;  C, p1 >= 1;  win % p1 == 0.
 * ------------------------------------------------------------------------------------------- */
typedef struct {
    int B, D, H, W;              /* scenes, feature width, scene rows / columns */
    int win, stride_y, stride_x; /* square window side, window step */
    int win_y, win_x;            /* windows per scene column / row */
    int win_first, n;            /* this chunk: global windows [win_first, win_first + n) */
    int C, p1;                   /* spectral blocks, spatial patch side */
} msst_scene_embed_dims;
MSST_API int msst_scene_embed(const msst_scene_embed_dims* d, const float* tokens, const float* weight, float* acc, float* wsum,
                              msst_stream_t stream);
/* Whole-scene masked reconstruction (SimMIM decoding): the same windows, chunks, weight and ownership contract as msst_scene_blend,
 * but each covering window contributes the decoder's prediction of the scene entries a scene mask hides.  One call blends the chunk
 * [win_first, win_first + n):
 *   tokens [n, C*S, D]         the chunk's encoder output with the masked tokens replaced by the mask token (fp32, t = c*S + s,
 *                              S = G*G, G = win / p1), read in place
 *   mask   [B, C, H, W] uint8  scene mask: nonzero = the p0 bands of spectral block c at pixel (y, x) are hidden
 *   W [n_wb, P, D], bias [n_wb, P]   the decoder: to_pixels (n_wb = 1) or BlockwiseToPixels (n_wb = C, block c uses row block c);
 *                              P = p0 * p1 * p1, output p = j * p1^2 + i1 * p1 + i2 is band c*p0 + j at (i1, i2) inside the patch
 *   weight [win, win] or NULL  per-window-pixel weight (NULL: 1)
 *   for every masked entry (b, band = c*p0 + j, y, x), over the chunk's windows covering (y, x) (origin (oy, ox), py = y - oy, px = x - ox):
 *     acc [B, C*p0, H, W] +=  weight(py, px) * (W[blk] . tokens[g - win_first, c*S + s, :] + bias[blk])[p],
 *                             s = (py / p1) * G + px / p1,  p = j * p1^2 + (py % p1) * p1 + px % p1,  blk = n_wb == 1 ? 0 : c
 *   wsum [B, H, W]      +=  weight(py, px)   once per covering window (entries of visible blocks are left as they are)
 * Bitwise independent of the chunking (chunks in ascending order); only the scene rows the chunk touches are visited.
 * 1 <= stride <= win <= H, W;  win_y <= ceil((H - win) / stride_y) + 1 (ditto x);  D a multiple of 32 in [32, 256];  P <= 16;
 * n_wb in {1, C};  win % p1 == 0;  C * p0 <= 1760 (shared memory).  MSST_ERR_ARG before any launch otherwise, outputs untouched.
 * ------------------------------------------------------------------------------------------- */
typedef struct {
    int B, D, H, W;              /* scenes, feature width, scene rows / columns */
    int win, stride_y, stride_x; /* square window side, window step */
    int win_y, win_x;            /* windows per scene column / row */
    int win_first, n;            /* this chunk: global windows [win_first, win_first + n) */
    int C, p0, p1, n_wb;         /* spectral blocks, spectral / spatial patch side, decoder weight blocks (1 or C) */
} msst_scene_reconstruct_dims;
MSST_API int msst_scene_reconstruct(const msst_scene_reconstruct_dims* d, const float* tokens, const uint8_t* mask, const float* W,
                                    const float* bias, const float* weight, float* acc, float* wsum, msst_stream_t stream);
/* Whole-scene integrated-gradients attribution: the same windows, chunks, weight and ownership contract as msst_scene_blend, but each
 * covering window contributes its input gradients at the pixel, summed over the integration steps.  One call adds the chunk
 * [win_first, win_first + n):
 *   grads [n, steps, bands, win, win]  d objective / d input of every interpolated window (window-major, step-minor), read in place
 *   weight [win, win] or NULL          per-window-pixel weight (NULL: 1)
 *   acc  [B, bands, H, W] +=  weight(py, px) * sum_{k ascending} grads[g - win_first, k, band, py, px]   over covering windows g, ascending
 *   wsum [B, H, W]        +=  weight(py, px)
 * Bitwise independent of the chunking (chunks in ascending order); only the scene rows the chunk touches are visited.
 * 1 <= stride <= win <= H, W;  win_y <= ceil((H - win) / stride_y) + 1 (ditto x);  bands, steps >= 1.  MSST_ERR_ARG before any launch
 * otherwise, outputs untouched.
 * ------------------------------------------------------------------------------------------- */
typedef struct { int B, bands, H, W, win, stride_y, stride_x, win_y, win_x, win_first, n, steps; } msst_scene_attribute_dims;
MSST_API int msst_scene_attribute(const msst_scene_attribute_dims* d, const float* grads, const float* weight, float* acc, float* wsum,
                                  msst_stream_t stream);

/* ---------------------------------------------------------------------------------------------
 * k-nearest-neighbour probing of embeddings (e.g. msst_scene_embed maps): cosine similarity, k best references per query, class vote.
 *   msst_knn_prepare   x [n, dim] fp32 rows -> out [n, 3*dim] bf16: y = x / max(||x||, 1e-12) (F.normalize) split into three bf16
 *                      parts y = hi + mid + lo, stored [hi | mid | lo].  Run once on the references and once per query chunk.
 *   msst_knn_topk      scores [n_query, k] fp32 (descending) and index [n_query, k] int64 of the k references with the largest cosine
 *                      similarity to each query, from prepared ref [n_ref, 3*dim] and query [n_query, 3*dim].  A score is
 *                      sum_{i+j<=2} part_i(q) . part_j(r) with fp32 accumulation: |score - exact cosine| <= 2.4e-7 + the fp32
 *                      accumulation error (DESIGN.md §3).  Order (score descending, reference index ascending): an equal score goes to the
 *                      lower index.  Bitwise independent of how the queries are chunked.  No atomics.
 *   msst_knn_vote      probs [n_query, nc] fp32 and pred [n_query] int64 from (scores, index) and ref_labels [n_ref] int64:
 *                      w_j = exp((s_j - s_0) / temperature), probs[c] = sum_{j: label(index_j) == c} w_j / sum_j w_j (the DINO k-NN
 *                      vote; subtracting the top score s_0 keeps exp in range), pred = argmax, lowest class on ties.
 *                      temperature = +inf is the uniform vote.  A label outside [0, nc) casts no vote but its weight stays in the sum.
 * Limits (MSST_ERR_ARG before any launch, outputs untouched): dim a multiple of 32 in [32, 256]; 1 <= k <= 64; k <= n_ref < 2^31;
 * 1 <= nc <= 256; temperature > 0; no NULL pointer.
 * ------------------------------------------------------------------------------------------- */
typedef struct {
    int64_t n_ref, n_query;      /* reference rows, query rows of this call */
    int dim, k;                  /* feature width, neighbours per query */
} msst_knn_dims;
MSST_API int msst_knn_prepare(const float* x, int64_t n, int dim, void* out, msst_stream_t stream);
MSST_API int msst_knn_topk(const msst_knn_dims* d, const void* ref, const void* query, float* scores, int64_t* index,
                           msst_stream_t stream);
MSST_API int msst_knn_vote(int64_t n_query, int k, int64_t n_ref, const float* scores, const int64_t* index, const int64_t* ref_labels,
                           int nc, float temperature, float* probs, int64_t* pred, msst_stream_t stream);

/* ---------------------------------------------------------------------------------------------
 * Linear probing of embeddings: softmax regression on frozen fp32 feature rows, H heads (learning rate / weight decay pairs)
 * trained in the same launches.
 *   z = LN(x):   mean and biased variance over dim, eps 1e-5, no affine (F.layer_norm(x, (dim,)), the default head's LayerNorm
 *                with weight 1 and bias 0); one device function normalises a row in training and in prediction.
 *   params [heads][nc*dim + nc]: head h is W_h [nc, dim] row-major followed by b_h [nc]; logits = W_h z + b_h.  The Adam moments
 *                m, v use the same layout.
 *   msst_linprobe_workspace  bytes of the workspace of msst_linprobe_grad / msst_linprobe_update for d->batch rows:
 *                ceil(batch / 128) * heads * (nc*dim + nc + 1) * 4; -1 (and the error message) on bad dims.
 *   msst_linprobe_grad       rows i = 0 .. batch-1 of the minibatch are x[index[i]] with label labels[index[i]].  Per 128-row slice
 *                of the minibatch and head it writes to the workspace sum_i (softmax(W_h z_i + b_h) - onehot(y_i)) (x) [z_i | 1]
 *                (the slice's dW_h and db_h sums) and sum_i CE_i.  A row whose index is outside [0, n) or whose label is outside
 *                [0, nc) contributes nothing (it still counts in the batch size).
 *   msst_linprobe_update     sums the slices' partials in ascending slice order, divides by batch and applies torch.optim.AdamW to
 *                every head in one launch: betas (0.9, 0.999), eps 1e-8, decoupled weight decay wd[h] on W_h and b_h, learning
 *                rate lr[h], 1-based step `step`, no clamp.  loss_sum [heads] = the step's CE sums (ascending slice order).
 *   msst_linprobe_predict    probs [n_query, nc] = softmax(W z + b), pred [n_query] int64 = argmax of probs, lowest class on ties,
 *                for the single head `params` [nc*dim + nc].
 * Deterministic: every sum runs in a fixed order (no atomics), a (slice, head) pair is one CTA and a parameter one thread, so the
 * results are bitwise independent of the SM count, of how many heads are trained together, and of how queries are chunked.
 * Limits (MSST_ERR_ARG before any launch, outputs untouched): dim a multiple of 32 in [32, 256]; 1 <= nc <= 256; 1 <= heads <= 16;
 * 1 <= n < 2^31; 1 <= batch; step >= 1; every lr[h], wd[h] finite and >= 0; 1 <= n_query < 2^31; no NULL pointer.
 * ------------------------------------------------------------------------------------------- */
#define MSST_LINPROBE_MAX_HEADS 16
typedef struct {
    int64_t n;                   /* rows of x (and labels) */
    int dim, nc, heads;          /* feature width, classes, heads */
    int batch;                   /* rows of this minibatch (entries of index) */
    int step;                    /* 1-based AdamW step (msst_linprobe_update) */
    float lr[MSST_LINPROBE_MAX_HEADS], wd[MSST_LINPROBE_MAX_HEADS];   /* per head; entries >= heads are ignored */
} msst_linprobe_dims;
MSST_API int64_t msst_linprobe_workspace(const msst_linprobe_dims* d);
MSST_API int msst_linprobe_grad(const msst_linprobe_dims* d, const float* x, const int64_t* labels, const int64_t* index,
                                const float* params, float* workspace, msst_stream_t stream);
MSST_API int msst_linprobe_update(const msst_linprobe_dims* d, const float* workspace, float* params, float* m, float* v,
                                  float* loss_sum, msst_stream_t stream);
MSST_API int msst_linprobe_predict(int64_t n_query, int dim, int nc, const float* x, const float* params, float* probs, int64_t* pred,
                                   msst_stream_t stream);

/* ---------------------------------------------------------------------------------------------
 * k-means clustering of embeddings (Lloyd's algorithm with k-means++ seeding), R restarts run together in the same launches.
 *   rows:        x [n, dim] fp32.  normalize = 1 uses every row as F.normalize(x, dim=1, eps=1e-12), y = x / max(||x||, 1e-12) in fp32
 *                (one device function, so every kernel sees the same bits); the normalised row is never stored.  normalize = 0 uses x.
 *   centroids    [R, K, dim] fp32; restart r owns centroids[r].
 *   distance     d(y, c) = sum_d (y_d - c_d)^2 in fp32, the direct difference form (not |y|^2 - 2 y.c + |c|^2, which cancels
 *                catastrophically for rows far from the origin).
 *   slices       rows [4096 s, 4096 s + 4096): a fixed length, independent of the grid and the SM count.  S = ceil(n / 4096).
 *   msst_kmeans_workspace  bytes of the workspace of msst_kmeans_seed / _assign / _update: 8*R*S + 4*R*S*K*dim + 4*R*S*K + 4*R*S;
 *                -1 (and the error message) on bad dims.
 *   msst_kmeans_assign     labels [R, n] int64 = argmin_k d(y_i, c_rk), the LOWEST k on ties; dist [R, n] fp32 = that minimum (dist may
 *                be NULL).  With a workspace it also writes, per (slice, restart): the per-cluster sums of the assigned rows (fp64 in
 *                ascending row order, stored rounded to fp32), the per-cluster counts, the slice's inertia (fp64 sum of the minima in
 *                ascending row order) and the number of rows whose label differs from the one in `labels` on entry (-1 before the
 *                first pass).  workspace = NULL is prediction: labels and distances only, `labels` is not read.
 *   msst_kmeans_update     thread = (restart, cluster, feature): c = (fp32)(sum_s sums_s / sum_s counts_s), the slices added in
 *                ascending order in fp64.  An EMPTY cluster keeps its previous centroid bit for bit (no relocation).  Per restart:
 *                inertia [R] fp64 = sum of the slices' inertias (ascending slice order) of the assignment that produced the sums,
 *                changed [R] int32 = rows whose label changed, empty [R] int32 = clusters with no row.  centroids are updated in place.
 *   msst_kmeans_seed       round j of k-means++ for every restart, u [R, K] fp64 uniforms in [0, 1) from the host:
 *                j = 0:  row i = min(floor(u[r][0] * n), n - 1)
 *                j > 0:  mindist [R, n] fp32 holds the distance of each row to the nearest of centroids 0 .. j-1 of its restart and
 *                        the workspace the fp64 per-slice sums of it (ascending row order); P_s = sum of the sums of slices < s and
 *                        T = P_S (ascending slice order), t = u[r][j] * T.  The round takes the first row i, in ascending order, with
 *                        P_s + L_i > t (strictly), L_i = the fp64 running sum of mindist over rows 4096 s .. i of its slice s.  When
 *                        T == 0 (fewer distinct rows than K) it falls back to the j = 0 rule with u[r][j].
 *                The chosen row (normalised when normalize = 1) becomes centroid j, index [R, K] int64 records it.  Unless j = K-1,
 *                a second launch then folds d(y_i, c_j) into mindist (j = 0: sets it) and refreshes the slice sums.  Rounds must
 *                run in order 0 .. K-1 on the same mindist / workspace.
 * Deterministic: no float atomics; a (slice, restart) pair is one CTA, every sum runs in a fixed order.  A restart's results depend
 * only on x, its own u row (or its given centroids) and the dims, so fits are bitwise reproducible, a restart run among others equals
 * the same restart run alone, and labels / dist of prediction are bitwise independent of how the rows are chunked.
 * Limits (MSST_ERR_ARG before any launch, outputs untouched): dim a multiple of 32 in [32, 256]; 1 <= K <= 256 and
 * K * dim <= MSST_KMEANS_MAX_KD (the per-cluster fp64 sums and the centroids live in shared memory: K = 128 at dim = 96, K = 64
 * at dim = 256); 1 <= R <= 16; n < 2^31 with K <= n for seeding and for assignment with a workspace, n >= 1 for prediction;
 * 0 <= round < K; no NULL pointer where one is required.
 * ------------------------------------------------------------------------------------------- */
#define MSST_KMEANS_MAX_RESTARTS 16
#define MSST_KMEANS_MAX_KD 16384
typedef struct {
    int64_t n;                   /* rows of x */
    int dim, k, restarts;        /* feature width, clusters, restarts R */
    int normalize;               /* 1: rows are F.normalize'd when staged */
} msst_kmeans_dims;
MSST_API int64_t msst_kmeans_workspace(const msst_kmeans_dims* d);
MSST_API int msst_kmeans_seed(const msst_kmeans_dims* d, int round, const float* x, const double* u, float* centroids, int64_t* index,
                              float* mindist, void* workspace, msst_stream_t stream);
MSST_API int msst_kmeans_assign(const msst_kmeans_dims* d, const float* x, const float* centroids, int64_t* labels, float* dist,
                                void* workspace, msst_stream_t stream);
MSST_API int msst_kmeans_update(const msst_kmeans_dims* d, const void* workspace, float* centroids, double* inertia, int32_t* changed,
                                int32_t* empty, msst_stream_t stream);

/* ---------------------------------------------------------------------------------------------
 * Mean, covariance and projection of rows (the device half of PCA and of the global RX anomaly detector).  All arithmetic is FP64.
 *   rows:        x [n, dim] fp32, centred as c = (double)x - mean (fp64 subtraction; the mean is never rounded to fp32).
 *   slices       rows [16384 s, 16384 s + 16384): a fixed length, independent of the grid and the SM count.  S = ceil(n / 16384).
 *   msst_moments_workspace  bytes of the workspace of msst_moments_mean / _cov: 8 * S * dim * (dim + 1) (46 MB at n = 1.43 M,
 *                dim = 256); -1 (and the error message) on bad dims.  Layout: the mean partials [S][dim] fp64, then the covariance
 *                partials [S][dim][dim] fp64 (only entries i <= j are written).
 *   msst_moments_mean      mean [dim] fp64 = (sum_s P_s) / n, the slices added in ascending order, P_s = the slice's column sums
 *                (fp64, rows added in ascending order).
 *   msst_moments_cov       cov [dim, dim] fp64 = (sum_s Q_s) / (n - 1), the slices added in ascending order, Q_s[i][j] = the fp64 FMA
 *                chain sum_r c_ri * c_rj over the slice's rows in ascending order (two passes: `mean` is an input, normally from
 *                msst_moments_mean).  Entry (i, j), i <= j, is written to (i, j) and (j, i): the matrix is exactly symmetric.
 *   msst_moments_project   W [k, dim] fp64 row-major, 1 <= k <= dim.  y [n, k] fp32: y_ij = fp32(sum_d c_id * W_jd), one fp64 FMA
 *                chain in ascending d.  score [n] fp32: fp32(sum_j y_ij^2) over the unrounded fp64 y_ij, one fp64 FMA chain in
 *                ascending j.  Either of y, score may be NULL, not both.  A row's y and score depend only on that row: bitwise
 *                independent of how the rows are chunked.  PCA: W = the components; RX: W = the whitening matrix, score = the
 *                squared Mahalanobis distance.
 * Deterministic: no atomics, every sum runs in the order given.
 * Limits (MSST_ERR_ARG before any launch, outputs untouched): 1 <= dim <= 256; 2 <= n < 2^31 for the workspace, mean and covariance,
 * 1 <= n < 2^31 for the projection; 1 <= k <= dim; no NULL pointer other than one of y / score.
 * ------------------------------------------------------------------------------------------- */
MSST_API int64_t msst_moments_workspace(int64_t n, int dim);
MSST_API int msst_moments_mean(int64_t n, int dim, const float* x, void* workspace, double* mean, msst_stream_t stream);
MSST_API int msst_moments_cov(int64_t n, int dim, const float* x, const double* mean, void* workspace, double* cov, msst_stream_t stream);
MSST_API int msst_moments_project(int64_t n, int dim, int k, const float* x, const double* mean, const double* W, float* y, float* score,
                                  msst_stream_t stream);

/* ---------------------------------------------------------------------------------------------
 * SimMIM decoder + masked L1 loss (vit_simmim_original.py:314-338, BlockwiseToPixels :9-40):
 *   pred[b,n,:] = W[blk] enc[b, idx[b,n], :] + bias[blk],  blk = idx / S (0 when n_weight_blocks == 1)
 *   target      = raw pixels of patch idx gathered from img (or target_tokens [B,T,P] if not NULL)
 *   loss        = mean |pred - target| / num_masked          (double normalisation, SURVEY C4)
 * idx [B,nm] int64 may disagree with the bool mask and may repeat (C3): backward accumulates.
 * ------------------------------------------------------------------------------------------- */
typedef struct { int B, C, G, p0, p1, D, nm, n_weight_blocks;
                 const msst_raw_input* raw;   /* optional: gather the target pixels from raw tiles (see msst_raw_input); may be NULL */
} msst_decode_dims;
MSST_API int msst_simmim_decode_l1_fwd(const msst_decode_dims* d, const float* enc, const int64_t* idx, const float* img,
                              const float* target_tokens, const float* W, const float* bias, float* pred /*or NULL*/,
                              float* partial /*[B*nm] scratch*/, float* loss, msst_stream_t stream);
/* d_enc [B,T,D] must be zeroed by the caller (scatter-add); d_W/d_bias accumulate; d_loss device scalar */
MSST_API int msst_simmim_decode_l1_bwd(const msst_decode_dims* d, const float* enc, const int64_t* idx, const float* img,
                              const float* target_tokens, const float* W, const float* bias, const float* d_loss,
                              float* d_enc, float* d_W, float* d_bias, float* d_target_tokens /*or NULL*/,
                              msst_stream_t stream);

/* ---------------------------------------------------------------------------------------------
 * SimMIM block / tube mask generation on the device (SURVEY 8(f) rank 1): replaces MaskGenerator.get_batch /
 * get_batch_tube_masked / bool_mask_to_indices (vit_simmim_original.py:343-416) with one launch.  A draw = a uniformly random
 * subset of mask_count of the rand_size^2 cells, upsampled by `scale` to the token grid; tube: one draw per sample shared by its C
 * spectral blocks, else one per (sample, block).  idx follows the reference's slicing (quirk C3): the ascending set positions of all
 * samples concatenated and cut into runs of nm.   mask [B, C*(rand_size*scale)^2] uint8, idx [B, nm] int64.
 * ------------------------------------------------------------------------------------------- */
typedef struct {
    int B, C, rand_size, scale, mask_count, nm, tube;
    uint64_t seed; const uint64_t* seed_dev;
} msst_maskgen_dims;
MSST_API int msst_draw_masks(const msst_maskgen_dims* d, uint8_t* mask, int64_t* idx, msst_stream_t stream);

/* ---------------------------------------------------------------------------------------------
 * (5) fused Adam/AdamW over a flat fp32 arena segment (torch.optim.AdamW/Adam as configured by
 *     src/utils.py:36-44, finetune.py:133-135) with the reference's elementwise grad clamp
 *     (pretrain.py:71-73) and the data-parallel 1/world scaling folded in.
 *     step_host = 1-based step number.  bf16_out (optional) receives a bf16 copy of the new params.
 * ------------------------------------------------------------------------------------------- */
typedef struct {
    float lr, beta1, beta2, eps, weight_decay;
    int decoupled;          /* 1 AdamW, 0 Adam with L2 added to the gradient */
    float clamp;            /* > 0: g = clamp(g, -clamp, clamp) after scaling; <= 0 off */
    float grad_scale;       /* e.g. 1/world_size */
    int step;
    const int* step_dev;    /* optional: device int32 holding the 1-based step (CUDA-graph capturable optimiser); overrides step */
} msst_adam_args;
MSST_API int msst_adam_step(const msst_adam_args* a, float* p, const float* g, float* m, float* v, void* bf16_out, int64_t n,
                   msst_stream_t stream);

#ifdef __cplusplus
}
#endif
#endif /* MSST_H_ */
