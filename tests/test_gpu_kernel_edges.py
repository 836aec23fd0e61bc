"""GPU: the embedding, head, cross-entropy, SimMIM decoder and LayerNorm kernels through the C ABI at the edges of the shapes they
accept, each against a plain float64 torch statement of the same operation (computed on the device).  Gradient buffers start
non-zero, so the tests also hold the kernels to their `+=` contract.  fp32 outputs: rel-l2 <= 1e-5; fp32 gradients (float atomics
in a different order): <= 1e-4; bf16 outputs: <= 4e-3 (one bf16 rounding, 2^-8 relative per element)."""
import ctypes as C
import itertools

import pytest
import torch
import torch.nn.functional as F

from maskedsst_b200 import _lib, ops
from maskedsst_b200.input import RawTiles
from oracle import maskedsst_oracle as O
from tests import dropout_ref

pytestmark = pytest.mark.gpu
DEV = "cuda"
F64 = torch.float64


def _st():
    return torch.cuda.current_stream().cuda_stream


def _p(t):
    return None if t is None else t.data_ptr()


def _err(got, want, floor=1e-7):
    """rel-l2 of got against want; a reference that is exactly zero (e.g. LayerNorm over one element) needs got ~ 0."""
    got, want = got.detach().to(F64), want.detach().to(F64)
    return float((got - want).norm() / max(float(want.norm()), floor))


def _ln(x, w, b):
    return O._ln(x, w, b)


def _rand(*shape, scale=1.0):
    return torch.randn(*shape, device=DEV) * scale


def _grad_bufs(shapes, scale=1.0):
    """Non-zero starting values for accumulated gradients, and a copy to subtract afterwards."""
    bufs = [_rand(*s, scale=scale) for s in shapes]
    return bufs, [b.clone() for b in bufs]


# ---------------------------------------------------------------------------------------------------------------------
# patch embedding
# ---------------------------------------------------------------------------------------------------------------------
def _to_patches(img, C_, G, p0, p1):
    B = img.shape[0]
    return img.reshape(B, C_, p0, G, p1, G, p1).permute(0, 1, 3, 5, 2, 4, 6).reshape(B, C_, G * G, p0 * p1 * p1)


def _embed_ref(img, prm, mask, C_, G, p0, p1, fac=None):
    """tokens [B,T,D] and patches_ln [B,T,P] in float64 (BlockwisePatchEmbedding / PatchEmbed + mask token + pos + dropout)."""
    pre_w, pre_b, W, bias, post_w, post_b, pos, mt = prm
    B, D = img.shape[0], W.shape[1]
    h = _ln(_to_patches(img, C_, G, p0, p1), pre_w, pre_b)               # [B,C,S,P]
    Wc, bc = (W, bias) if W.shape[0] == C_ else (W.expand(C_, -1, -1), bias.expand(C_, -1))
    y = torch.einsum("bcsp,cdp->bcsd", h, Wc) + bc[None, :, None, :]
    o = _ln(y, post_w, post_b).reshape(B, -1, D)
    if mask is not None:
        o = torch.where(mask[..., None], mt, o)
    o = o + pos
    if fac is not None:
        o = o * fac
    return o, h.reshape(B, -1, h.shape[-1])


def _embed_params(C_, nwb, D, P, T):
    return [1 + 0.1 * _rand(P), 0.1 * _rand(P), _rand(nwb, D, P, scale=P ** -0.5), 0.1 * _rand(nwb, D),
            1 + 0.1 * _rand(D), 0.1 * _rand(D), _rand(T, D), _rand(D)]


def _run_embed(B, C_, G, p0, p1, D, nwb, mask_mode, with_ln, drop_p=0.0, seed=0, check_bwd=True):
    P, S = p0 * p1 * p1, G * G
    T = C_ * S
    torch.manual_seed(B * 1000 + C_ * 100 + G * 10 + P + D)
    img = _rand(B, C_ * p0, G * p1, G * p1)
    prm = _embed_params(C_, nwb, D, P, T)
    mask = None if mask_mode == "none" else (torch.rand(B, T, device=DEV) < 0.4 if mask_mode == "some" else
                                             torch.ones(B, T, dtype=torch.bool, device=DEV))
    mask_u8 = None if mask is None else mask.to(torch.uint8).contiguous()
    dims = _lib.EmbedDims(B, C_, G, p0, p1, D, nwb, drop_p, seed, None, None)
    lib = _lib.lib()
    tokens = torch.full((B, T, D), float("nan"), device=DEV)
    pln = torch.full((B, T, P), float("nan"), device=DEV) if with_ln else None
    _lib.check(lib.msst_patch_embed_fwd(C.byref(dims), _p(img), *[_p(t) for t in prm[:7]], _p(mask_u8),
                                        _p(prm[7]) if mask is not None else None, _p(tokens), _p(pln), _st()))
    fac = None
    if drop_p > 0:   # the embedding's dropout site is 1, element row * D + f of the tokens: the host model of the mask
        fac = torch.from_numpy(dropout_ref.elem_mask(drop_p, seed, 1, B * T * D)).view(B, T, D).double().to(DEV)
    ref = [t.double().requires_grad_(True) for t in prm]
    want, want_ln = _embed_ref(img.double(), ref, mask, C_, G, p0, p1, fac)
    assert _err(tokens, want) < 1e-5
    if with_ln:
        assert _err(pln, want_ln) < 1e-5
    if not check_bwd:
        return
    d_tok = _rand(B, T, D)
    d_ln = _rand(B, T, P) if with_ln else None
    (want * d_tok.double()).sum().add((want_ln * d_ln.double()).sum() if with_ln else 0.0).backward()
    g, g0 = _grad_bufs([t.shape for t in prm])
    _lib.check(lib.msst_patch_embed_bwd(C.byref(dims), _p(img), *[_p(t) for t in prm[:6]], _p(mask_u8), _p(d_tok), _p(d_ln),
                                        *[_p(t) for t in g[:7]], _p(g[7]) if mask is not None else None, _st()))
    names = ["pre_w", "pre_b", "W", "bias", "post_w", "post_b", "pos", "mask_token"]
    for k in range(8 if mask is not None else 7):
        assert _err(g[k] - g0[k], ref[k].grad) < 1e-4, names[k]
    if mask is None:
        assert torch.equal(g[7], g0[7])


EMBED_P = [(1, 1), (10, 1), (11, 1), (16, 1), (4, 2)]    # (p0, p1): P = 1, 10, 11 (PMAX-16 backward), 16, and 16 with p1 = 2


@pytest.mark.parametrize("G", [1, 8, 9])
@pytest.mark.parametrize("p0,p1", EMBED_P)
@pytest.mark.parametrize("D", [32, 64, 96, 128])
def test_patch_embed(D, p0, p1, G):
    """S = 1 / 64 / 81 (a full 64-token chunk, a chunk tail), both weight layouts, no / some / all tokens masked, patches_ln."""
    i = EMBED_P.index((p0, p1)) + [1, 8, 9].index(G) + D // 32
    _run_embed(B=3, C_=3, G=G, p0=p0, p1=p1, D=D, nwb=3 if i % 2 else 1, mask_mode=("none", "some", "all")[i % 3],
               with_ln=i % 2 == 0)


def test_patch_embed_backward_loops_over_samples():
    """C * chunks = 40 CTAs along x leaves room for 14 along y: each backward CTA walks 2-3 samples of the batch of 30."""
    _run_embed(B=30, C_=20, G=9, p0=10, p1=1, D=64, nwb=20, mask_mode="some", with_ln=True)


@pytest.mark.parametrize("D", [64, 128])
def test_patch_embed_dropout(D):
    _run_embed(B=4, C_=5, G=8, p0=10, p1=1, D=D, nwb=5, mask_mode="some", with_ln=False, drop_p=0.3, seed=1234)


def test_patch_embed_wide_patches_forward_only():
    """P = 64 runs forward; the backward keeps 16 accumulators per lane, so P = 17 and P = 64 are argument errors."""
    _run_embed(B=2, C_=2, G=3, p0=16, p1=2, D=128, nwb=2, mask_mode="some", with_ln=True, check_bwd=False)
    for p0, p1 in [(17, 1), (16, 2)]:
        P = p0 * p1 * p1
        dims = _lib.EmbedDims(1, 1, 2, p0, p1, 32, 1, 0.0, 0, None, None)
        img = _rand(1, p0, 2 * p1, 2 * p1)
        prm = _embed_params(1, 1, 32, P, 4)
        g = [torch.zeros_like(t) for t in prm]
        d_tok = _rand(1, 4, 32)
        rc = _lib.lib().msst_patch_embed_bwd(C.byref(dims), _p(img), *[_p(t) for t in prm[:6]], None, _p(d_tok), None,
                                             *[_p(t) for t in g[:7]], None, _st())
        assert rc == 1 and b"16" in _lib.lib().msst_last_error()
        assert all(float(t.abs().max()) == 0.0 for t in g)


# ---------------------------------------------------------------------------------------------------------------------
# classification head
# ---------------------------------------------------------------------------------------------------------------------
def _head_ref(x, ln_w, ln_b, W, bias, B, C_, G, p1, nc):
    D = x.shape[-1]
    z = _ln(x.reshape(B, C_, G, G, D).mean(dim=1), ln_w, ln_b)
    y = z @ W.T + bias                                                     # [B,G,G,p1*p1*nc], outputs (p1 p2 nc)
    y = y.reshape(B, G, G, p1, p1, nc).permute(0, 1, 3, 2, 4, 5).reshape(B, G * p1, G * p1, nc)
    return y.permute(0, 3, 1, 2)


def _head_fits(nc, p1, D):
    return nc * p1 * p1 * D * 8 + 4096 * 4 < 200 * 1024


def _run_head(B, C_, G, p1, D, nc):
    torch.manual_seed(B + C_ + G + p1 + D + nc)
    NO = nc * p1 * p1
    x = _rand(B, C_ * G * G, D)
    prm = [1 + 0.1 * _rand(D), 0.1 * _rand(D), _rand(NO, D, scale=D ** -0.5), 0.1 * _rand(NO)]
    dims = _lib.HeadDims(B, C_, G, p1, D, nc)
    lib = _lib.lib()
    logits = torch.full((B, nc, G * p1, G * p1), float("nan"), device=DEV)
    rc = lib.msst_head_fwd(C.byref(dims), _p(x), *[_p(t) for t in prm], _p(logits), _st())
    if not _head_fits(nc, p1, D):
        assert rc == 1 and b"too large" in lib.msst_last_error()
        assert torch.isnan(logits).all()
        return
    _lib.check(rc)
    ref = [t.double().requires_grad_(True) for t in prm]
    xr = x.double().requires_grad_(True)
    want = _head_ref(xr, *ref, B, C_, G, p1, nc)
    assert _err(logits, want) < 1e-5
    dl = _rand(*logits.shape)
    (want * dl.double()).sum().backward()
    g, g0 = _grad_bufs([t.shape for t in prm])
    dx = torch.full_like(x, float("nan"))                                   # d_x is written, not accumulated
    _lib.check(lib.msst_head_bwd(C.byref(dims), _p(x), *[_p(t) for t in prm[:3]], _p(dl), _p(dx), *[_p(t) for t in g], _st()))
    assert _err(dx, xr.grad) < 1e-5
    for k, name in enumerate(["ln_w", "ln_b", "W", "bias"]):
        assert _err(g[k] - g0[k], ref[k].grad) < 1e-4, name


@pytest.mark.parametrize("nc", [1, 20])
@pytest.mark.parametrize("p1", [1, 2, 3])
@pytest.mark.parametrize("D", [32, 64, 96, 128, 192, 256])
def test_head(D, p1, nc):
    """Every D the head is built for, 1-3 pixels per patch side, one or 20 classes; shapes whose weight table does not fit the
    shared-memory budget (NO * D * 8 B + 16 KiB < 200 KiB) must be refused before any launch."""
    _run_head(B=2, C_=3, G=5, p1=p1, D=D, nc=nc)


def test_head_shared_memory_bound():
    assert _head_fits(735, 1, 32) and not _head_fits(736, 1, 32)
    _run_head(B=2, C_=2, G=3, p1=1, D=32, nc=735)     # just under the bound: runs, and is right
    _run_head(B=2, C_=2, G=3, p1=1, D=32, nc=736)     # just over: MSST_ERR_ARG


def test_head_grid_stride():
    """B * S = 16384 (sample, position) items: more than the forward's 1184 CTAs x 8 warps and the backward's 148 x 8."""
    _run_head(B=64, C_=2, G=16, p1=1, D=96, nc=20)


def test_head_rejects_unbuilt_width():
    x = _rand(1, 4, 160)
    prm = [_rand(160), _rand(160), _rand(20, 160), _rand(20)]
    logits = torch.full((1, 20, 2, 2), float("nan"), device=DEV)
    dims = _lib.HeadDims(1, 1, 2, 1, 160, 20)
    assert _lib.lib().msst_head_fwd(C.byref(dims), _p(x), *[_p(t) for t in prm], _p(logits), _st()) == 1
    g = [torch.zeros_like(t) for t in prm]
    dx = torch.zeros_like(x)
    assert _lib.lib().msst_head_bwd(C.byref(dims), _p(x), *[_p(t) for t in prm[:3]], _p(logits), _p(dx),
                                    *[_p(t) for t in g], _st()) == 1
    torch.cuda.synchronize()
    assert torch.isnan(logits).all() and all(float(t.abs().max()) == 0.0 for t in g + [dx])


# ---------------------------------------------------------------------------------------------------------------------
# cross-entropy
# ---------------------------------------------------------------------------------------------------------------------
def _run_ce(logits, labels, ignore_index):
    B, nc = logits.shape[:2]
    HW = logits[0, 0].numel()
    sc = torch.full((2,), float("nan"), device=DEV)                       # set, not accumulated
    dl = torch.full_like(logits, float("nan"))
    _lib.check(_lib.lib().msst_cross_entropy_fwd_bwd(_p(logits), _p(labels), B, nc, HW, ignore_index, _p(sc), _p(dl), _st()))
    return sc, dl


def _ce_ref(logits, labels, ignore_index):
    lg = logits.double().requires_grad_(True)
    loss = F.cross_entropy(lg, labels, ignore_index=ignore_index, reduction="sum")
    loss.backward()
    return loss.detach(), float((labels != ignore_index).sum()), lg.grad


@pytest.mark.parametrize("scale", [3.0, 1e4])
@pytest.mark.parametrize("ignore_index", [-1, 255])
@pytest.mark.parametrize("nc", [1, 2, 300])
def test_cross_entropy(nc, ignore_index, scale):
    torch.manual_seed(nc)
    B, H, W = 3, 25, 40
    logits = _rand(B, nc, H, W, scale=scale)
    labels = torch.randint(0, nc, (B, H, W), device=DEV)
    labels[torch.rand(B, H, W, device=DEV) < 0.2] = ignore_index
    if nc > 255:
        labels[0, 0, :7] = 254                                          # class 254 counts, class 255 is ignored
    sc, dl = _run_ce(logits, labels, ignore_index)
    loss, cnt, grad = _ce_ref(logits, labels, ignore_index)
    assert float(sc[1]) == cnt
    assert abs(float(sc[0]) - float(loss)) <= 1e-5 * abs(float(loss))
    assert _err(dl, grad) < 1e-5                                        # softmax - onehot on valid pixels, 0 elsewhere


def test_cross_entropy_skips_labels_outside_the_classes():
    """A label outside [0, nc) that is not ignore_index is skipped like an ignored pixel (torch raises instead): it adds
    nothing to the loss, not 1 to the count, and its logits get a zero gradient."""
    torch.manual_seed(3)
    B, nc, H, W = 2, 5, 8, 8
    logits = _rand(B, nc, H, W)
    labels = torch.randint(0, nc, (B, H, W), device=DEV)
    labels[0, 0, 0] = -1
    labels[0, 1, :3] = torch.tensor([-7, nc, nc + 40], device=DEV)
    labels[1, 2, 5] = 2 ** 40
    bad = (labels < 0) | (labels >= nc)
    sc, dl = _run_ce(logits, labels, ignore_index=-100)
    loss, cnt, grad = _ce_ref(logits, torch.where(bad, torch.full_like(labels, -100), labels), -100)
    assert float(sc[1]) == cnt == B * H * W - 5
    assert abs(float(sc[0]) - float(loss)) <= 1e-5 * abs(float(loss))
    assert _err(dl, grad) < 1e-5 and float(dl.permute(0, 2, 3, 1)[bad].abs().max()) == 0.0


# ---------------------------------------------------------------------------------------------------------------------
# SimMIM decoder + masked L1
# ---------------------------------------------------------------------------------------------------------------------
def _decode_ref(enc, idx, tgt, W, bias, S):
    """tgt [B,T,P]; W [nwb,P,D]; blk = idx // S (0 for one weight block); loss = mean|pred - target| / nm."""
    B, nm = idx.shape
    br = torch.arange(B, device=DEV)[:, None]
    blk = idx // S if W.shape[0] > 1 else torch.zeros_like(idx)
    pred = torch.einsum("bnd,bnpd->bnp", enc[br, idx], W[blk]) + bias[blk]
    return (pred - tgt[br, idx]).abs().mean() / nm, pred


def _decode_case(D, p0, p1, path, target, raw=False):
    """Returns the decoder dims and tensors; `path` picks C so that the [C][P][D] weight-gradient table does ("smem") or does not
    ("global") fit the 100 KiB shared-memory budget of the backward."""
    P, G = p0 * p1 * p1, 3
    S = G * G
    C_ = 3 if path == "smem" else 25600 // (P * (D + 1)) + 2
    assert (C_ * P * (D + 1) * 4 > 100 * 1024) == (path == "global")
    T, B = C_ * S, 2
    nm = max(8, T // 2)
    torch.manual_seed(D + P + C_)
    enc = _rand(B, T, D)
    idx = torch.randint(0, T, (B, nm), device=DEV)                        # not ascending, with repeats
    idx[:, 1] = idx[:, 0]
    idx[1, 5] = idx[0, 5]
    W = _rand(C_, P, D, scale=D ** -0.5)
    bias = 0.1 * _rand(C_, P)
    img = tgt_tok = rt = None
    if target == "tokens":
        tgt_tok = _rand(B, T, P)
        tgt = tgt_tok
    elif raw:
        tiles = torch.randint(-400, 12000, (B, C_ * p0, G * p1 + 3, G * p1 + 2), dtype=torch.int16, device=DEV)
        rt = RawTiles(tiles, torch.rand(C_ * p0) * 3000 + 1000, torch.rand(C_ * p0) * 1000 + 500, image_size=G * p1, crop=(2, 1))
        tgt = _to_patches(rt.materialize(), C_, G, p0, p1).reshape(B, T, P)
    else:
        img = _rand(B, C_ * p0, G * p1, G * p1)
        tgt = _to_patches(img, C_, G, p0, p1).reshape(B, T, P)
    return (B, C_, G, p0, p1, D, nm, S), enc, idx, img, tgt_tok, rt, tgt, W, bias


@pytest.mark.parametrize("target", ["image", "tokens", "raw"])
@pytest.mark.parametrize("path", ["smem", "global"])
@pytest.mark.parametrize("p0,p1", [(1, 1), (16, 1), (4, 2), (1, 2)])
@pytest.mark.parametrize("D", [32, 128])
def test_simmim_decode(D, p0, p1, path, target):
    (B, C_, G, p0, p1, D, nm, S), enc, idx, img, tgt_tok, rt, tgt, W, bias = _decode_case(D, p0, p1, path,
                                                                                          "tokens" if target == "tokens" else "image",
                                                                                          raw=target == "raw")
    P = p0 * p1 * p1
    raw_struct = rt.c_struct() if rt is not None else None
    dims = _lib.DecodeDims(B, C_, G, p0, p1, D, nm, C_, C.pointer(raw_struct) if raw_struct is not None else None)
    lib = _lib.lib()
    pred = torch.full((B, nm, P), float("nan"), device=DEV)
    partial = torch.empty(B * nm, device=DEV)
    loss = torch.full((), float("nan"), device=DEV)
    _lib.check(lib.msst_simmim_decode_l1_fwd(C.byref(dims), _p(enc), _p(idx), _p(img), _p(tgt_tok), _p(W), _p(bias), _p(pred),
                                             _p(partial), _p(loss), _st()))
    ref = [t.double().requires_grad_(True) for t in (enc, tgt, W, bias)]
    want, want_pred = _decode_ref(ref[0], idx, ref[1], ref[2], ref[3], S)
    assert _err(pred, want_pred) < 1e-5
    assert abs(float(loss) - float(want)) <= 1e-5 * abs(float(want))
    d_loss = torch.full((), 1.7, device=DEV)
    (want * 1.7).backward()
    # the gradients are tiny (1.7 / (B nm P nm) per element): start the buffers at their scale, or fp32 could not hold the sum
    scale = 1.7 / (B * nm * P * nm)
    d_enc, g0_enc = _grad_bufs([enc.shape], scale)
    (d_W, d_b), g0 = _grad_bufs([W.shape, bias.shape], scale)
    d_tgt, g0_tgt = _grad_bufs([tgt_tok.shape], scale) if tgt_tok is not None else ([None], [None])
    _lib.check(lib.msst_simmim_decode_l1_bwd(C.byref(dims), _p(enc), _p(idx), _p(img), _p(tgt_tok), _p(W), _p(bias), _p(d_loss),
                                             _p(d_enc[0]), _p(d_W), _p(d_b), _p(d_tgt[0]), _st()))
    assert _err(d_enc[0] - g0_enc[0], ref[0].grad) < 1e-4
    assert _err(d_W - g0[0], ref[2].grad) < 1e-4
    assert _err(d_b - g0[1], ref[3].grad) < 1e-4
    if tgt_tok is not None:
        assert _err(d_tgt[0] - g0_tgt[0], ref[1].grad) < 1e-4


def test_simmim_decode_single_weight_block():
    """to_pixels as one Linear (n_weight_blocks = 1): every index uses block 0."""
    (B, C_, G, p0, p1, D, nm, S), enc, idx, img, _, _, tgt, W, bias = _decode_case(64, 4, 2, "smem", "image")
    W, bias = W[:1].contiguous(), bias[:1].contiguous()
    dims = _lib.DecodeDims(B, C_, G, p0, p1, D, nm, 1, None)
    lib = _lib.lib()
    partial = torch.empty(B * nm, device=DEV)
    loss = torch.empty((), device=DEV)
    _lib.check(lib.msst_simmim_decode_l1_fwd(C.byref(dims), _p(enc), _p(idx), _p(img), None, _p(W), _p(bias), None, _p(partial),
                                             _p(loss), _st()))
    ref = [t.double().requires_grad_(True) for t in (enc, W, bias)]
    want, _ = _decode_ref(ref[0], idx, tgt.double(), ref[1], ref[2], S)
    want.backward()
    assert abs(float(loss) - float(want)) <= 1e-5 * abs(float(want))
    d_enc = torch.zeros_like(enc)
    d_W, d_b = torch.zeros_like(W), torch.zeros_like(bias)
    _lib.check(lib.msst_simmim_decode_l1_bwd(C.byref(dims), _p(enc), _p(idx), _p(img), None, _p(W), _p(bias),
                                             _p(torch.ones((), device=DEV)), _p(d_enc), _p(d_W), _p(d_b), None, _st()))
    assert _err(d_enc, ref[0].grad) < 1e-4 and _err(d_W, ref[1].grad) < 1e-4 and _err(d_b, ref[2].grad) < 1e-4


# ---------------------------------------------------------------------------------------------------------------------
# LayerNorm
# ---------------------------------------------------------------------------------------------------------------------
def _ln_case(rows, D, y_bf16, with_add, offset=0):
    """One forward + backward; `offset` floats shift every buffer off 16-byte alignment (the generic kernels)."""
    lib = _lib.lib()

    def buf(*shape, fill=None, scale=1.0, shift=0.0):
        n = 1
        for s in shape:
            n *= s
        t = (torch.randn(n + offset, device=DEV) * scale + shift if fill is None else torch.full((n + offset,), fill, device=DEV))
        return t[offset:].view(*shape)

    x = buf(rows, D, scale=2.0, shift=0.5)
    assert offset == 0 or x.data_ptr() % 16 != 0
    w, b = 1 + 0.1 * _rand(D), 0.1 * _rand(D)
    y = torch.full((rows, D), float("nan"), device=DEV, dtype=torch.bfloat16) if y_bf16 else buf(rows, D, fill=float("nan"))
    stats = torch.full((rows, 2), float("nan"), device=DEV)
    _lib.check(lib.msst_layernorm_fwd(_p(x), _p(w), _p(b), _p(y), int(y_bf16), _p(stats), rows, D, 1e-5, _st()))
    xr, wr, br = x.double(), w.double().requires_grad_(True), b.double().requires_grad_(True)
    xr.requires_grad_(True)
    want = _ln(xr, wr, br)
    if rows == 0:
        return
    assert _err(y, want) < (4e-3 if y_bf16 else 1e-5)
    mu = xr.detach().mean(-1)
    rstd = 1.0 / torch.sqrt(((xr.detach() - mu[:, None]) ** 2).mean(-1) + 1e-5)
    assert _err(stats[:, 0], mu, floor=1.0) < 1e-5 and _err(stats[:, 1], rstd) < 1e-5
    dy = buf(rows, D)
    add = buf(rows, D) if with_add else None
    (want * dy.double()).sum().backward()
    dx = buf(rows, D, fill=float("nan"))
    (dw, db), g0 = _grad_bufs([(D,), (D,)])
    _lib.check(lib.msst_layernorm_bwd(_p(x), _p(w), _p(stats), _p(dy), _p(add), _p(dx), _p(dw), _p(db), rows, D, _st()))
    want_dx = xr.grad + (add.double() if with_add else 0.0)
    assert _err(dx, want_dx) < 1e-5
    assert _err(dw - g0[0], wr.grad) < 1e-4 and _err(db - g0[1], br.grad) < 1e-4


@pytest.mark.parametrize("rows", [0, 1, 5, 100003])
@pytest.mark.parametrize("D", [1, 3, 33, 96, 130, 160, 256, 257, 1536])
def test_layernorm(D, rows):
    """Quad kernel (D % 4 == 0, D <= 128), register kernel (other D <= 256) and wide kernel (D > 256); fp32 and bf16 output;
    with and without the added skip gradient."""
    for y_bf16, with_add in itertools.product((0, 1), (False, True)):
        _ln_case(rows, D, y_bf16, with_add)


def test_layernorm_rows_zero_touches_nothing():
    x, w, b = _rand(4, 96), _rand(96), _rand(96)
    dw, db = torch.full((96,), 3.0, device=DEV), torch.full((96,), 4.0, device=DEV)
    lib = _lib.lib()
    _lib.check(lib.msst_layernorm_bwd(_p(x), _p(w), _p(x), _p(x), None, _p(x), _p(dw), _p(db), 0, 96, _st()))
    torch.cuda.synchronize()
    assert bool((dw == 3.0).all()) and bool((db == 4.0).all())


@pytest.mark.parametrize("rows", [5, 1001])
def test_layernorm_unaligned_rows(rows):
    """A view 4 bytes into its allocation cannot use the float4 kernel at D = 96: the generic kernel must give the same answer."""
    for y_bf16, with_add in itertools.product((0, 1), (False, True)):
        _ln_case(rows, 96, y_bf16, with_add, offset=1)


# ---------------------------------------------------------------------------------------------------------------------
# bf16 transformer stack wider than the fused kernels (D > 128: LayerNorm backward without its fused cast)
# ---------------------------------------------------------------------------------------------------------------------
def _stack_ref(x, prm, n_seq, N, H, dh):
    sd = {}
    for l, lp in enumerate(prm):
        b = f"layers.{l}."
        for k, t in zip(["0.norm.weight", "0.norm.bias", "0.fn.to_qkv.weight", "0.fn.to_out.0.weight", "0.fn.to_out.0.bias",
                         "1.norm.weight", "1.norm.bias", "1.fn.net.0.weight", "1.fn.net.0.bias", "1.fn.net.3.weight",
                         "1.fn.net.3.bias"], lp):
            sd[b + k] = t
    spec = O.Spec(depth=len(prm), heads=H, dim_head=dh)
    return O.transformer(x.reshape(n_seq, N, -1), sd, "", spec).reshape(n_seq * N, -1)


@pytest.mark.parametrize("D", [128, 192, 256])
def test_transformer_stack_bf16_wide(D):
    """H = 4 heads of 64, mlp_dim 64, L = 2, bf16 mode, forward and backward against float64."""
    torch.manual_seed(D)
    H, dh, M, L, n_seq, N = 4, 64, 64, 2, 6, 40
    I = H * dh
    prm = [[1 + 0.1 * _rand(D), 0.1 * _rand(D), _rand(3 * I, D, scale=D ** -0.5), _rand(D, I, scale=I ** -0.5), 0.1 * _rand(D),
            1 + 0.1 * _rand(D), 0.1 * _rand(D), _rand(M, D, scale=D ** -0.5), 0.1 * _rand(M), _rand(D, M, scale=M ** -0.5),
            0.1 * _rand(D)] for _ in range(L)]
    x = _rand(n_seq * N, D)
    xg = x.clone().requires_grad_(True)
    pg = [[t.clone().requires_grad_(True) for t in lp] for lp in prm]
    y = ops.transformer_stack(xg, pg, n_seq=n_seq, N=N, inner=1, heads=H, dim_head=dh, mlp_dim=M, prec=_lib.PREC_BF16)
    dy = _rand(*y.shape)
    (y * dy).sum().backward()
    xr = x.double().requires_grad_(True)
    pr = [[t.double().requires_grad_(True) for t in lp] for lp in prm]
    want = _stack_ref(xr, pr, n_seq, N, H, dh)
    (want * dy.double()).sum().backward()
    assert _err(y, want) < 1e-2
    pairs = [(xg.grad, xr.grad)] + [(a.grad, b.grad) for la, lb in zip(pg, pr) for a, b in zip(la, lb)]
    for k, (got, ref) in enumerate(pairs):
        e = _err(got, ref)
        cos = float((got.double().flatten() @ ref.flatten()) / (got.double().norm() * ref.norm()))
        assert e < 5e-2 and cos > 0.998, (k, e, cos)
