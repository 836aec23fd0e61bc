"""torch.autograd bindings of the C-ABI kernels (include/msst.h).  PyTorch is used for device memory,
streams and the autograd graph only; every arithmetic step is a libmsst.so launch on the current stream."""
import ctypes as C
import itertools

import torch

from . import _lib
from ._lib import check, PREC_FP32, PREC_BF16
from .input import RawTiles

_SITE_EMB = 1
SITE_LAYER_BASE = 16

# ---- dropout seeds -----------------------------------------------------------------------------------
_seed_counter = itertools.count(1)


def next_seed() -> int:
    """Fresh 64-bit dropout key per training forward, derived from torch's seed (torch.manual_seed reproducible)."""
    return (torch.initial_seed() * 0x9E3779B97F4A7C15 + next(_seed_counter) * 0xD1B54A32D192ED03) & 0xFFFFFFFFFFFFFFFF


_device_seed = None   # optional uint64-as-int64 device tensor added to every dropout seed (CUDA-graph replays)


def set_device_seed(t):
    """t: 0-dim int64 CUDA tensor (or None).  When set, kernels add its CURRENT device value to their dropout seed, so a
    captured graph that increments it once per replay draws fresh masks every step."""
    global _device_seed
    _device_seed = t


def _seed_dev():
    return None if _device_seed is None else _device_seed.data_ptr()


def _check_drop_p(p):
    """nn.Dropout's range: p in [0, 1] (p = 1 zeroes the branch); NaN or anything outside is an error, not a silent mask."""
    if not 0.0 <= float(p) <= 1.0:
        raise ValueError(f"maskedsst_b200: dropout probability must be in [0, 1], got {p}")


def _stream():
    return torch.cuda.current_stream().cuda_stream


def _p(t):
    return None if t is None else t.data_ptr()


def _chk(t, name, dtype=torch.float32):
    if t is None:
        return
    if not t.is_cuda:
        raise RuntimeError(f"maskedsst_b200: {name} must be a CUDA tensor (there is no CPU path)")
    if t.dtype != dtype:
        raise RuntimeError(f"maskedsst_b200: {name} must be {dtype}, got {t.dtype}")
    if not t.is_contiguous():
        raise RuntimeError(f"maskedsst_b200: {name} must be contiguous")


def _c(t):
    return t if t.is_contiguous() else t.contiguous()


# ---- gradient buffers -----------------------------------------------------------------------------------
# The backward kernels ACCUMULATE (+=) parameter gradients.  Handing them freshly zeroed tensors makes autograd's
# AccumulateGrad add every one of them into p.grad afterwards: one elementwise launch per parameter (~100 per step), which
# is what a small-batch step spends its time on.  When the parameters live in a FusedAdam arena whose gradient arena has
# just been zeroed (optimizer.zero_grad(): one memset, p.grad = None), the kernels write straight into the arena views and
# autograd adopts the returned view as p.grad without launching anything.
_arenas = []


def register_grad_arena(arena):
    _arenas.append(arena)


def _grad_buffers(params):
    """One fp32 buffer per tensor in `params` for a kernel to accumulate into; arena views for leaf parameters when allowed
    (see above), slices of ONE zero-filled allocation for the rest."""
    out = [None] * len(params)
    fresh = []
    for i, p in enumerate(params):
        if p.is_leaf and p.requires_grad and p.grad is None:
            for a in _arenas:
                v = a.claim(p)
                if v is not None:
                    out[i] = v
                    break
        if out[i] is None:
            fresh.append(i)
    if fresh:
        sizes = [params[i].numel() for i in fresh]
        flat = torch.zeros(sum(sizes), device=params[fresh[0]].device, dtype=torch.float32)
        for i, g in zip(fresh, torch.split(flat, sizes)):
            out[i] = g.view(params[i].shape)
    return out


# ---- (1) patch embedding ------------------------------------------------------------------------------
class PatchEmbedFn(torch.autograd.Function):
    """tokens[B,T,D] = [mask-select](LN_D(W_c LN_P(patch) + b_c)) + pos  (+ emb-dropout)."""

    @staticmethod
    def forward(ctx, img, pre_w, pre_b, W, bias, post_w, post_b, pos, mask_token, mask, geom, drop_p, seed, want_ln):
        C_, G, p0, p1, D = geom
        B = img.shape[0]
        T = C_ * G * G
        raw = img if isinstance(img, RawTiles) else None     # pixels come from raw tiles through the fused input pipeline
        if raw is not None:
            if tuple(raw.shape[1:]) != (C_ * p0, G * p1, G * p1):
                raise RuntimeError(f"maskedsst_b200: RawTiles cube shape {tuple(raw.shape)} does not match the model ({C_ * p0} bands, {G * p1} px)")
            ctx.raw_struct = raw.c_struct()
            img = None
        else:
            img = _c(img)
            _chk(img, "img")
        for n, t in (("pre_w", pre_w), ("W", W), ("pos", pos)):
            _chk(t, n)
        mask_u8 = None
        if mask is not None:
            mask_u8 = _c(mask.to(torch.uint8))
        dims = _lib.EmbedDims(B, C_, G, p0, p1, D, W.shape[0], float(drop_p), seed, _seed_dev(),
                              C.pointer(ctx.raw_struct) if raw is not None else None)
        tokens = torch.empty(B, T, D, device=pos.device, dtype=torch.float32)
        pln = torch.empty(B, T, p0 * p1 * p1, device=pos.device, dtype=torch.float32) if want_ln else None
        pos_c = _c(pos)
        check(_lib.lib().msst_patch_embed_fwd(C.byref(dims), _p(img), _p(pre_w), _p(pre_b), _p(W), _p(bias), _p(post_w),
                                              _p(post_b), _p(pos_c), _p(mask_u8), _p(mask_token), _p(tokens), _p(pln), _stream()))
        ctx.save_for_backward(img, pre_w, pre_b, W, bias, post_w, post_b, mask_u8)
        ctx.raw = raw            # keeps the tiles / statistics alive until backward
        ctx.dims = dims
        ctx.has_mt = mask_token is not None
        ctx.pos_shape = pos.shape
        return tokens, pln

    @staticmethod
    def backward(ctx, d_tokens, d_pln):
        img, pre_w, pre_b, W, bias, post_w, post_b, mask_u8 = ctx.saved_tensors
        dims = ctx.dims
        T, D = ctx.pos_shape
        g = _grad_buffers([pre_w, pre_b, W, bias, post_w, post_b])
        g += list(torch.split(torch.zeros(T * D + D, device=pre_w.device, dtype=torch.float32), [T * D, D]))   # pos rows, mask token
        d_tokens = _c(d_tokens)
        d_pln = _c(d_pln) if d_pln is not None else None
        check(_lib.lib().msst_patch_embed_bwd(C.byref(dims), _p(img), _p(pre_w), _p(pre_b), _p(W), _p(bias), _p(post_w),
                                              _p(post_b), _p(mask_u8), _p(d_tokens), _p(d_pln), _p(g[0]), _p(g[1]), _p(g[2]),
                                              _p(g[3]), _p(g[4]), _p(g[5]), _p(g[6]), _p(g[7]) if ctx.has_mt else None,
                                              _stream()))
        return (None, g[0], g[1], g[2], g[3], g[4], g[5], g[6].view(T, D),
                g[7] if ctx.has_mt else None, None, None, None, None, None)


def patch_embed(img, pre_w, pre_b, W, bias, post_w, post_b, pos, mask_token=None, mask=None, *, geom, drop_p=0.0,
                seed=0, want_ln=False):
    _check_drop_p(drop_p)
    out, pln = PatchEmbedFn.apply(img, pre_w, pre_b, W, bias, post_w, post_b, pos, mask_token, mask, geom, drop_p, seed, want_ln)
    return (out, pln) if want_ln else out


# ---- transformer stack --------------------------------------------------------------------------------
_LAYER_FIELDS = ("ln1_w", "ln1_b", "w_qkv", "w_out", "b_out", "ln2_w", "ln2_b", "w1", "b1", "w2", "b2")


def _layer_array(tensors, L):
    arr = (_lib.LayerPtrs * L)()
    for l in range(L):
        for k, name in enumerate(_LAYER_FIELDS):
            setattr(arr[l], name, tensors[l * 11 + k].data_ptr())
    return arr


class TransformerStackFn(torch.autograd.Function):
    """L pre-norm layers over rows [R, D]; sequence geometry (n_seq, N, inner) as in msst_attention_*."""

    @staticmethod
    def forward(ctx, x, cfg, *params):
        n_seq, N, inner, H, dh, M, L, drop_p, seed, site_base, prec, need_grad = cfg
        _chk(x, "x")
        for t in params:
            _chk(t, "transformer parameter")
        R, D = x.shape
        assert R == n_seq * N, (R, n_seq, N)
        dims = _lib.TfDims(n_seq, N, inner, D, H, dh, M, L, float(drop_p), seed, site_base, prec, int(need_grad), _seed_dev())
        nbytes = _lib.lib().msst_transformer_workspace_bytes(C.byref(dims))
        if nbytes < 0:
            check(1)
        ws = torch.empty(nbytes, device=x.device, dtype=torch.uint8)
        y = torch.empty_like(x)
        arr = _layer_array(params, L)
        check(_lib.lib().msst_transformer_fwd(C.byref(dims), arr, _p(x), _p(y), _p(ws), _stream()))
        if need_grad:
            ctx.save_for_backward(x, ws, *params)
            ctx.dims = dims
        return y

    @staticmethod
    def backward(ctx, dy):
        x, ws, *params = ctx.saved_tensors
        dims = ctx.dims
        L = dims.L
        dy = _c(dy)
        grads = _grad_buffers(params)
        dx = torch.empty_like(x)
        check(_lib.lib().msst_transformer_bwd(C.byref(dims), _layer_array(params, L), _layer_array(grads, L), _p(x), _p(dy),
                                              _p(dx), _p(ws), _stream()))
        return (dx, None, *grads)


def transformer_stack(x, layer_params, *, n_seq, N, inner, heads, dim_head, mlp_dim, drop_p=0.0, seed=0, site_base=SITE_LAYER_BASE,
                      prec=PREC_FP32):
    """layer_params: list (per layer) of the 11 tensors in _LAYER_FIELDS order."""
    _check_drop_p(drop_p)
    flat = [t for lp in layer_params for t in lp]
    # Function.forward runs with grad mode off, so decide here whether activations must be kept for backward
    need_grad = torch.is_grad_enabled() and (x.requires_grad or any(t.requires_grad for t in flat))
    cfg = (n_seq, N, inner, heads, dim_head, mlp_dim, len(layer_params), drop_p, seed, site_base, prec, need_grad)
    return TransformerStackFn.apply(x, cfg, *flat)


# ---- classification head + CE ---------------------------------------------------------------------------
class HeadFn(torch.autograd.Function):
    @staticmethod
    def forward(ctx, x, ln_w, ln_b, W, bias, geom):
        B, C_, G, p1, D, nc = geom
        x = _c(x)
        _chk(x, "x")
        dims = _lib.HeadDims(B, C_, G, p1, D, nc)
        logits = torch.empty(B, nc, G * p1, G * p1, device=x.device, dtype=torch.float32)
        check(_lib.lib().msst_head_fwd(C.byref(dims), _p(x), _p(ln_w), _p(ln_b), _p(W), _p(bias), _p(logits), _stream()))
        ctx.save_for_backward(x, ln_w, ln_b, W, bias)
        ctx.dims = dims
        return logits

    @staticmethod
    def backward(ctx, d_logits):
        x, ln_w, ln_b, W, bias = ctx.saved_tensors
        dims = ctx.dims
        d_logits = _c(d_logits)
        g = _grad_buffers([ln_w, ln_b, W, bias])
        dx = torch.empty_like(x)
        check(_lib.lib().msst_head_bwd(C.byref(dims), _p(x), _p(ln_w), _p(ln_b), _p(W), _p(d_logits), _p(dx), _p(g[0]), _p(g[1]),
                                       _p(g[2]), _p(g[3]), _stream()))
        return dx, g[0], g[1], g[2], g[3], None


def head(x, ln_w, ln_b, W, bias, *, geom):
    return HeadFn.apply(x, ln_w, ln_b, W, bias, geom)


class CrossEntropyFn(torch.autograd.Function):
    """mean NLL over pixels with label != ignore_index (nn.CrossEntropyLoss(ignore_index=-1), finetune.py:136)."""

    @staticmethod
    def forward(ctx, logits, labels, ignore_index):
        logits = _c(logits)
        _chk(logits, "logits")
        labels = _c(labels)
        _chk(labels, "labels", torch.int64)
        B, nc = logits.shape[:2]
        HW = logits[0, 0].numel()
        sc = torch.empty(2, device=logits.device, dtype=torch.float32)
        dl = torch.empty_like(logits)
        check(_lib.lib().msst_cross_entropy_fwd_bwd(_p(logits), _p(labels), B, nc, HW, ignore_index, _p(sc), _p(dl), _stream()))
        ctx.save_for_backward(dl, sc)
        return sc[0] / sc[1]

    @staticmethod
    def backward(ctx, g):
        dl, sc = ctx.saved_tensors
        return dl * (g / sc[1]), None, None


def cross_entropy(logits, labels, ignore_index=-1):
    return CrossEntropyFn.apply(logits, labels, ignore_index)


class CrossEntropySumFn(torch.autograd.Function):
    """(sum of NLL over valid pixels, number of valid pixels) -- the two pieces a data-parallel run all-reduces."""

    @staticmethod
    def forward(ctx, logits, labels, ignore_index):
        logits = _c(logits)
        _chk(logits, "logits")
        labels = _c(labels)
        _chk(labels, "labels", torch.int64)
        B, nc = logits.shape[:2]
        HW = logits[0, 0].numel()
        sc = torch.empty(2, device=logits.device, dtype=torch.float32)
        dl = torch.empty_like(logits)
        check(_lib.lib().msst_cross_entropy_fwd_bwd(_p(logits), _p(labels), B, nc, HW, ignore_index, _p(sc), _p(dl), _stream()))
        ctx.save_for_backward(dl)
        ctx.mark_non_differentiable(sc[1])
        return sc[0], sc[1]

    @staticmethod
    def backward(ctx, g, _):
        (dl,) = ctx.saved_tensors
        return dl * g, None, None


def cross_entropy_sum_count(logits, labels, ignore_index=-1):
    return CrossEntropySumFn.apply(logits, labels, ignore_index)


# ---- SimMIM decoder + masked L1 ---------------------------------------------------------------------------
class DecodeL1Fn(torch.autograd.Function):
    @staticmethod
    def forward(ctx, enc, idx, img, target_tokens, W, bias, geom):
        B, C_, G, p0, p1, D, nm = geom
        enc = _c(enc)
        _chk(enc, "enc")
        idx = _c(idx)
        _chk(idx, "idx", torch.int64)
        raw = img if isinstance(img, RawTiles) else None
        if target_tokens is not None:
            target_tokens = _c(target_tokens)
            raw = img = None
        elif raw is not None:
            ctx.raw_struct = raw.c_struct()
            img = None
        else:
            img = _c(img)
        ctx.raw = raw
        dims = _lib.DecodeDims(B, C_, G, p0, p1, D, nm, W.shape[0], C.pointer(ctx.raw_struct) if raw is not None else None)
        partial = torch.empty(B * nm, device=enc.device, dtype=torch.float32)
        loss = torch.empty((), device=enc.device, dtype=torch.float32)
        check(_lib.lib().msst_simmim_decode_l1_fwd(C.byref(dims), _p(enc), _p(idx), _p(img), _p(target_tokens), _p(W), _p(bias),
                                                   None, _p(partial), _p(loss), _stream()))
        ctx.save_for_backward(enc, idx, img if target_tokens is None else None, target_tokens, W, bias)
        ctx.dims = dims
        return loss

    @staticmethod
    def backward(ctx, d_loss):
        enc, idx, img, target_tokens, W, bias = ctx.saved_tensors
        dims = ctx.dims
        d_loss = _c(d_loss.to(torch.float32))
        d_enc = torch.zeros_like(enc)
        g = _grad_buffers([W, bias])
        d_tgt = None
        if target_tokens is not None and ctx.needs_input_grad[3]:
            d_tgt = torch.zeros_like(target_tokens)
        check(_lib.lib().msst_simmim_decode_l1_bwd(C.byref(dims), _p(enc), _p(idx), _p(img), _p(target_tokens), _p(W), _p(bias),
                                                   _p(d_loss), _p(d_enc), _p(g[0]), _p(g[1]), _p(d_tgt), _stream()))
        return d_enc, None, None, d_tgt, g[0], g[1], None


def simmim_decode_l1(enc, idx, img, target_tokens, W, bias, *, geom):
    return DecodeL1Fn.apply(enc, idx, img, target_tokens, W, bias, geom)


# ---- fine-grained ops (generic heads, unit tests, microbench) -------------------------------------------------
class LayerNormFn(torch.autograd.Function):
    @staticmethod
    def forward(ctx, x, w, b, eps):
        x = _c(x)
        _chk(x, "x")
        D = x.shape[-1]
        rows = x.numel() // D
        y = torch.empty_like(x)
        stats = torch.empty(rows, 2, device=x.device, dtype=torch.float32)
        check(_lib.lib().msst_layernorm_fwd(_p(x), _p(w), _p(b), _p(y), 0, _p(stats), rows, D, eps, _stream()))
        ctx.save_for_backward(x, w, stats)
        return y

    @staticmethod
    def backward(ctx, dy):
        x, w, stats = ctx.saved_tensors
        dy = _c(dy)
        D = x.shape[-1]
        rows = x.numel() // D
        dx = torch.empty_like(x)
        g = torch.zeros(2, D, device=x.device, dtype=torch.float32)
        check(_lib.lib().msst_layernorm_bwd(_p(x), _p(w), _p(stats), _p(dy), None, _p(dx), _p(g[0]), _p(g[1]), rows, D, _stream()))
        return dx, g[0], g[1], None


def layer_norm(x, w, b, eps=1e-5):
    return LayerNormFn.apply(x, w, b, eps)


class LinearFn(torch.autograd.Function):
    """y = x W^T + b (+ residual); fp32 parity-mode GEMMs (activation epilogues are used inside the fused stack only)."""

    @staticmethod
    def forward(ctx, x, W, bias, residual):
        act = 0
        x = _c(x)
        _chk(x, "x")
        _chk(W, "W")
        K = x.shape[-1]
        M = x.numel() // K
        N = W.shape[0]
        y = torch.empty(*x.shape[:-1], N, device=x.device, dtype=torch.float32)
        pre = torch.empty_like(y) if act else None
        if residual is not None:
            residual = _c(residual)
        dims = _lib.LinearDims(M, N, K, act, 0.0, 0, 0, PREC_FP32, None, 1)
        check(_lib.lib().msst_linear_fwd(C.byref(dims), _p(x), _p(W), _p(bias), _p(residual), _p(y), _p(pre), _stream()))
        ctx.save_for_backward(x, W, pre)
        ctx.dims = dims
        ctx.has_bias = bias is not None
        ctx.has_res = residual is not None
        return y

    @staticmethod
    def backward(ctx, dy):
        x, W, pre = ctx.saved_tensors
        dims = ctx.dims
        dy = _c(dy)
        lib = _lib.lib()
        dx = torch.empty_like(x)
        check(lib.msst_linear_bwd_data(C.byref(dims), _p(dy), _p(W), None, None, _p(dx), _stream()))
        dW = torch.zeros_like(W)
        db = torch.zeros(W.shape[0], device=x.device, dtype=torch.float32) if ctx.has_bias else None
        check(lib.msst_linear_bwd_weight(C.byref(dims), _p(dy), _p(x), _p(dW), _p(db), _stream()))
        return dx, dW, db, (dy if ctx.has_res else None)


def linear(x, W, bias=None, residual=None):
    return LinearFn.apply(x, W, bias, residual)


class AttentionFn(torch.autograd.Function):
    @staticmethod
    def forward(ctx, qkv, cfg):
        n_seq, N, inner, H, dh, drop_p, seed, site = cfg
        qkv = _c(qkv)
        prec = PREC_BF16 if qkv.dtype == torch.bfloat16 else PREC_FP32   # bf16 tensors -> tensor-core kernels
        _chk(qkv, "qkv", qkv.dtype if prec == PREC_BF16 else torch.float32)
        R = n_seq * N
        dims = _lib.AttnDims(n_seq, N, inner, H, dh, float(drop_p), seed, site, prec, None)
        out = torch.empty(R, H * dh, device=qkv.device, dtype=qkv.dtype)
        lse = torch.empty(R, H, device=qkv.device, dtype=torch.float32)
        check(_lib.lib().msst_attention_fwd(C.byref(dims), _p(qkv), _p(out), _p(lse), _stream()))
        ctx.save_for_backward(qkv, out, lse)
        ctx.dims = dims
        return out

    @staticmethod
    def backward(ctx, d_out):
        qkv, out, lse = ctx.saved_tensors
        d_out = _c(d_out.to(qkv.dtype))
        d_qkv = torch.empty_like(qkv)
        check(_lib.lib().msst_attention_bwd(C.byref(ctx.dims), _p(qkv), _p(out), _p(lse), _p(d_out), _p(d_qkv), _stream()))
        return d_qkv, None


def attention(qkv, *, n_seq, N, inner=1, heads=8, dim_head=64, drop_p=0.0, seed=0, site=0):
    """qkv [n_seq*N, 3*heads*dim_head] -> [n_seq*N, heads*dim_head]."""
    _check_drop_p(drop_p)
    return AttentionFn.apply(qkv, (n_seq, N, inner, heads, dim_head, drop_p, seed, site))
