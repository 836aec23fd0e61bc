"""GPU: input gradients and integrated-gradients attribution.  msst_patch_embed_bwd_data (csrc/patch_embed.cu) teacher-forced against
float64 autograd of the embedding map; torch.autograd.grad(., img) through every model surface against float64 autograd of
oracle/maskedsst_oracle.py; attribute_windows / attribute_scene / msst_scene_attribute (csrc/scene.cu) against float64 IG blended in
numpy."""
import ctypes as C

import numpy as np
import pytest
import torch

import maskedsst_b200 as M
from maskedsst_b200 import _lib, ops
from maskedsst_b200.inference import (attribute_scene, attribute_sum, attribute_windows, band_importance, ig_alphas, scene_windows)
from maskedsst_b200.optim import FusedAdam
from oracle import maskedsst_oracle as O
from tests.dropout_ref import elem_mask
from tests.helpers import rel_l2
from tests.test_gpu_parity import make_encoder
from tests.test_gpu_scene_reconstruct import _gauss, _origins, _sim, _stats

pytestmark = pytest.mark.gpu
DEV = "cuda"
P2X4 = dict(channels=48, num_classes=20, spatial_patch_size=2, spectral_patch_size=4)   # G = 4, C = 12, P = 16


# ---- kernel level: msst_patch_embed_bwd_data ------------------------------------------------------------------------------------
def _ln(x, w, b):
    mu = x.mean(-1, keepdim=True)
    var = ((x - mu) ** 2).mean(-1, keepdim=True)
    return (x - mu) / torch.sqrt(var + 1e-5) * w + b


def _embed64(img, pre_w, pre_b, W, bias, post_w, post_b, mask, factor, C_, G, p0, p1):
    """float64 embedding map: (tokens without pos [B, T, D] with mask-token select (a constant) and dropout factors, patches_ln)."""
    B, D = img.shape[0], W.shape[1]
    S, P = G * G, p0 * p1 * p1
    x = img.reshape(B, C_, p0, G, p1, G, p1).permute(0, 1, 3, 5, 2, 4, 6).reshape(B, C_, S, P)
    h = _ln(x, pre_w, pre_b)
    Wc, bc = (W, bias) if W.shape[0] == C_ else (W.expand(C_, -1, -1), bias.expand(C_, -1))
    z = _ln(torch.einsum("bcsp,cdp->bcsd", h, Wc) + bc[None, :, None, :], post_w, post_b).reshape(B, C_ * S, D)
    if mask is not None:
        z = torch.where(mask[..., None], torch.zeros_like(z), z)
    return z * factor, h.reshape(B, C_ * S, P)


def _bwd_data(dims, t, mask_u8, d_tok, d_pln, out):
    return _lib.lib().msst_patch_embed_bwd_data(C.byref(dims), t["img"].data_ptr(), t["pre_w"].data_ptr(), t["pre_b"].data_ptr(),
                                                t["W"].data_ptr(), t["bias"].data_ptr(), t["post_w"].data_ptr(), t["post_b"].data_ptr(),
                                                None if mask_u8 is None else mask_u8.data_ptr(), d_tok.data_ptr(),
                                                None if d_pln is None else d_pln.data_ptr(), out.data_ptr(),
                                                torch.cuda.current_stream().cuda_stream)


KCASES = {   # name: (B, C, G, p0, p1, D, n_wb, masked, with d_patches_ln, drop_p, offset, flat patch)
    "houston_blockwise_d96": (3, 5, 8, 10, 1, 96, 5, False, False, 0.0, 0.0, False),
    "patchembed_d32_p2x4": (2, 12, 4, 4, 2, 32, 1, True, True, 0.0, 0.0, False),
    "v1_layout_d128_p4x1": (2, 6, 2, 1, 4, 128, 1, True, False, 0.0, 0.0, False),
    "p16x2_d96": (2, 3, 5, 16, 2, 96, 3, False, True, 0.0, 0.0, False),
    "dropout_0p1": (2, 5, 8, 10, 1, 96, 5, False, False, 0.1, 0.0, False),
    "offset_rows_1e3": (2, 5, 9, 10, 1, 64, 5, True, True, 0.0, 1e3, False),
    "flat_patch": (2, 5, 8, 10, 1, 128, 1, False, True, 0.0, 0.0, True),
}


@pytest.mark.parametrize("case", sorted(KCASES))
def test_patch_embed_bwd_data_vs_float64(case):
    B, C_, G, p0, p1, D, nwb, masked, with_pln, drop_p, offset, flat = KCASES[case]
    rng = np.random.default_rng(sum(map(ord, case)))
    S, P, T = G * G, p0 * p1 * p1, C_ * G * G
    f = lambda *s: torch.from_numpy(rng.standard_normal(s))
    img = f(B, C_ * p0, G * p1, G * p1) + offset
    if flat:   # one patch with variance far below eps
        img.view(B, C_, p0, G, p1, G, p1)[0, 1, :, 2, :, 3, :] = 0.25 + 1e-4 * f(p0, p1, p1)
    t64 = dict(img=img, pre_w=1 + 0.3 * f(P), pre_b=0.1 * f(P), W=f(nwb, D, P) / P ** 0.5, bias=0.1 * f(nwb, D), post_w=1 + 0.3 * f(D),
               post_b=0.1 * f(D))
    t64 = {k: v.float().double() for k, v in t64.items()}    # the reference differentiates at the fp32 inputs the kernel reads
    mask = torch.from_numpy(rng.random((B, T)) < 0.4) if masked else None
    seed = 1234567
    factor = torch.from_numpy(elem_mask(drop_p, seed, ops._SITE_EMB, B * T * D).reshape(B, T, D)).double() if drop_p else torch.ones(1)
    d_tok, d_pln = f(B, T, D).float().double(), (f(B, T, P).float().double() if with_pln else None)
    # float64 reference
    x = t64["img"].clone().requires_grad_(True)
    z, h = _embed64(x, *[t64[k] for k in ("pre_w", "pre_b", "W", "bias", "post_w", "post_b")], mask, factor, C_, G, p0, p1)
    obj = (z * d_tok).sum() + ((h * d_pln).sum() if with_pln else 0.0)
    (want,) = torch.autograd.grad(obj, x)
    # kernel
    t = {k: v.float().to(DEV).contiguous() for k, v in t64.items()}
    dims = _lib.EmbedDims(B, C_, G, p0, p1, D, nwb, drop_p, seed, None, None)
    mask_u8 = mask.to(torch.uint8).to(DEV) if masked else None
    dt, dp = d_tok.float().to(DEV), (d_pln.float().to(DEV) if with_pln else None)
    out = torch.full_like(t["img"], float("nan"))
    assert _bwd_data(dims, t, mask_u8, dt, dp, out) == 0
    again = torch.full_like(t["img"], 7.0)
    assert _bwd_data(dims, t, mask_u8, dt, dp, again) == 0
    torch.cuda.synchronize()
    assert torch.equal(out, again)                              # every element written, bitwise reproducible
    got = out.cpu().double()
    errs = [rel_l2(got[b], want[b]) for b in range(B)]
    print(f"{case}: per-sample rel-l2 {max(errs):.2e}")
    assert max(errs) <= 1e-5
    if masked:   # a masked token's pixels get only the d_patches_ln term (zero without it)
        m_img = mask.reshape(B, C_, G, G)[:, :, :, None, :, None].expand(B, C_, G, p1, G, p1).reshape(B, C_, 1, G * p1, G * p1)
        m_img = m_img.expand(B, C_, p0, G * p1, G * p1).reshape(B, C_ * p0, G * p1, G * p1)
        if not with_pln:
            assert (got[m_img] == 0).all()


def test_patch_embed_bwd_data_limits_leave_output_untouched():
    B, C_, G, p0, p1, D = 1, 5, 8, 10, 1, 96
    t = dict(img=torch.randn(B, 50, 8, 8, device=DEV), pre_w=torch.ones(10, device=DEV), pre_b=torch.zeros(10, device=DEV),
             W=torch.randn(5, 96, 10, device=DEV), bias=torch.zeros(5, 96, device=DEV), post_w=torch.ones(96, device=DEV),
             post_b=torch.zeros(96, device=DEV))
    dt = torch.randn(B, 320, 96, device=DEV)
    out = torch.full_like(t["img"], 3.0)
    raw = _lib.RawInput()
    bad = [dict(D=160), dict(D=80), dict(n_weight_blocks=2), dict(drop_p=1.5), dict(p0=65, C=1), dict(raw=C.pointer(raw))]
    for kw in bad:
        d = dict(B=B, C=C_, G=G, p0=p0, p1=p1, D=D, n_weight_blocks=5, drop_p=0.0, seed=0, seed_dev=None, raw=None)
        d.update(kw)
        dims = _lib.EmbedDims(*[d[k] for k, _ in _lib.EmbedDims._fields_])
        assert _bwd_data(dims, t, None, dt, None, out) == 1, kw
    torch.cuda.synchronize()
    assert (out == 3.0).all()


# ---- module level: gradients reach img ------------------------------------------------------------------------------------------
def _model(kind):
    if kind == "v1":
        spec = O.Spec(**O.HOUSTON, v1=True, depth=2)
        m = M.ViTSpatialSpectral_V1(image_size=8, spatial_patch_size=1, spectral_patch_size=10, num_classes=20, dim=96, depth=2,
                                    heads=8, mlp_dim=64, channels=50)
        m.load_state_dict(O.synthetic_state_dict(spec, seed=11), strict=True)
        return m.to(DEV), spec
    kw = dict(O.HOUSTON)
    extra = {}
    if kind == "p1_2":
        kw = dict(P2X4)
    elif kind == "patchembed":
        kw["blockwise_patch_embed"] = False
    elif kind == "spectral_only":
        kw["spectral_only"] = True
    elif kind == "spectral_pos":
        kw["spectral_pos_embed"] = True
    elif kind in ("pixelwise", "spectral_mlp"):
        extra = {kind if kind == "pixelwise" else "spectral_mlp_head": True}
    spec = O.Spec(**kw, depth=2)
    m = M.ViTSpatialSpectral(image_size=8, spatial_patch_size=spec.spatial_patch_size, spectral_patch_size=spec.spectral_patch_size,
                             num_classes=spec.num_classes, dim=96, depth=2, heads=8, mlp_dim=64, channels=spec.channels,
                             spectral_pos_embed=spec.spectral_pos_embed, blockwise_patch_embed=spec.blockwise_patch_embed,
                             spectral_pos=spec.pos(), spectral_only=spec.spectral_only, **extra)
    own = m.state_dict()
    m.load_state_dict({k: v for k, v in O.synthetic_state_dict(spec, seed=12).items() if k in own and own[k].shape == v.shape},
                      strict=False)   # the pixelwise / spectral-MLP heads keep their initialisation
    return m.to(DEV), spec


def _forward64(m, spec, x, kind):
    """float64 ViTSpatialSpectral forward from the model's own state dict: the oracle for the default head, the heads' modules in
    float64 otherwise."""
    sd = {k: v.detach().double().cpu() for k, v in m.state_dict().items()}
    if kind not in ("pixelwise", "spectral_mlp"):
        return O.encoder_forward(x, sd, spec)
    z = O.transformer_forward(O.encoder_tokens(x, sd, spec), sd, spec)
    B, c, g, D = x.shape[0], spec.C, spec.S_sqrt, spec.dim
    if kind == "pixelwise":
        z = _ln(z.reshape(B, c, g, g, D).mean(1), sd["mlp_head.0.weight"], sd["mlp_head.0.bias"]).reshape(B, -1)
        return (z @ sd["mlp_head.2.weight"].T + sd["mlp_head.2.bias"]).reshape(B, 1, 1, -1).squeeze()
    z = z.reshape(B, c, g, g, D).permute(0, 2, 3, 1, 4).reshape(B, g, g, c * D)
    y = _ln(z, sd["mlp_head.0.weight"], sd["mlp_head.0.bias"]) @ sd["mlp_head.1.weight"].T + sd["mlp_head.1.bias"]
    p = spec.spatial_patch_size
    return y.reshape(B, g, g, p, p, -1).permute(0, 1, 3, 2, 4, 5).reshape(B, g * p, g * p, -1).permute(0, 3, 1, 2)


MODULE_KINDS = ["houston", "p1_2", "patchembed", "spectral_only", "spectral_pos", "pixelwise", "spectral_mlp", "v1"]


@pytest.mark.parametrize("kind", MODULE_KINDS)
def test_input_gradient_vs_float64_oracle(kind):
    m, spec = _model(kind)
    m.eval()
    x = O.synthetic_cube(spec, 3, seed=4)
    x64 = x.double().requires_grad_(True)
    y64 = _forward64(m, spec, x64, kind)
    g_out = torch.from_numpy(np.random.default_rng(3).standard_normal(tuple(y64.shape)))
    (want,) = torch.autograd.grad(y64, x64, g_out)
    xi = x.to(DEV).requires_grad_(True)
    (got,) = torch.autograd.grad(m(xi), xi, g_out.float().to(DEV))
    err = rel_l2(got, want)
    print(f"{kind}: rel-l2 {err:.2e}")
    assert err <= 1e-5
    if kind in ("houston", "p1_2", "v1"):   # the bf16 model against fp32
        m.precision = "bf16"
        (gb,) = torch.autograd.grad(m(xi), xi, g_out.float().to(DEV))
        eb = rel_l2(gb, got)
        print(f"{kind}: bf16 vs fp32 rel-l2 {eb:.2e}")
        assert eb <= 1e-2


def test_embed_patches_path_gets_gradient():
    m, spec = _model("houston")
    x = O.synthetic_cube(spec, 2, seed=6)
    patches = O.to_patch(x, spec)
    p = patches.to(DEV).requires_grad_(True)
    g_out = torch.randn(2, spec.T, spec.dim, device=DEV)
    (got,) = torch.autograd.grad(m.to_patch_embedding.embed(p), p, g_out)
    sd = {k: v.detach().double().cpu() for k, v in m.state_dict().items()}
    p64 = patches.double().requires_grad_(True)
    (want,) = torch.autograd.grad(O.embed(p64, sd, spec), p64, g_out.double().cpu())
    assert rel_l2(got, want) <= 1e-5


SIM_CASES = {   # name: (kwargs, blockwise decoder, duplicate indices)
    "shared_decoder": (O.HOUSTON, False, False),
    "blockwise_decoder_duplicates": (O.HOUSTON, True, True),
    "patchembed_target": (dict(**O.HOUSTON, blockwise_patch_embed=False), False, True),
    "p2x4_blockwise": (P2X4, True, False),
}


@pytest.mark.parametrize("case", sorted(SIM_CASES) + ["v1"])
def test_simmim_input_gradient_vs_float64_oracle(case):
    if case == "v1":
        spec = O.Spec(**O.HOUSTON, v1=True, depth=2)
        enc = M.ViTSpatialSpectral_V1(image_size=8, spatial_patch_size=1, spectral_patch_size=10, num_classes=20, dim=96, depth=2,
                                      heads=8, mlp_dim=64, channels=50)
        m = M.SimMIMSpatialSpectral(encoder=enc, masking_ratio=0.7, mask_patch_size=4, tube_masking=True)
        sd = O.synthetic_state_dict(spec, seed=21, simmim=True, blockwise_decoder=False)
        m.load_state_dict(sd, strict=False)
        m, blockwise, dup = m.to(DEV).train(), False, False
    else:
        kw, blockwise, dup = SIM_CASES[case]
        m, spec, sd = _sim(kw, 22, blockwise)
    B = 3
    x = O.synthetic_cube(spec, B, seed=8)
    np.random.seed(8)
    mask, idx = m.draw_masks(B, DEV)
    if dup:   # quirk C3: an index list may name a token twice
        idx = idx.clone()
        idx[:, 1] = idx[:, 0]
    for p in m.parameters():
        p.requires_grad_(False)
    xi = x.to(DEV).requires_grad_(True)
    (got,) = torch.autograd.grad(m(xi, masks=(mask, idx)), xi)
    x64 = x.double().requires_grad_(True)
    sd64 = {k: v.double() for k, v in sd.items()}
    (want,) = torch.autograd.grad(O.simmim_forward(x64, sd64, spec, mask.cpu(), idx.cpu(), blockwise_decoder=blockwise), x64)
    err = rel_l2(got, want)
    print(f"simmim {case}: rel-l2 {err:.2e}")
    assert err <= 1e-5
    if spec.blockwise_patch_embed and not spec.v1:   # masked patches: only the L1-target term, zero where no index names them
        G, p0, p1 = spec.S_sqrt, spec.spectral_patch_size, spec.spatial_patch_size
        named = torch.zeros(B, spec.T, dtype=torch.bool)
        named[torch.arange(B)[:, None], idx.cpu()] = True
        only = (mask.cpu() & ~named).reshape(B, spec.C, G, G)[:, :, None, :, None, :, None]
        only = only.expand(B, spec.C, p0, G, p1, G, p1).reshape(x.shape)
        assert (got.cpu()[only] == 0).all()


def test_parameter_gradients_unchanged_by_input_gradient():
    """A SimMIM training step's parameter gradients do not depend on whether img requires grad, and the step launches exactly one
    kernel more (the data gradient) when it does."""
    m, spec, _ = _sim(O.HOUSTON, 23, True)
    x = O.synthetic_cube(spec, 4, seed=9).to(DEV)
    np.random.seed(9)
    masks = m.draw_masks(4, DEV)
    L = _lib.lib()

    def step(need_img):
        m.zero_grad(set_to_none=True)
        xi = x.clone().requires_grad_(need_img)
        loss = m(xi, masks=masks)
        n0 = L.msst_launch_count()
        loss.backward()
        torch.cuda.synchronize()
        return {k: p.grad.clone() for k, p in m.named_parameters() if p.grad is not None}, L.msst_launch_count() - n0, xi.grad

    a1, la, ga = step(False)
    b, lb, gb = step(True)
    assert ga is None and gb is not None and lb == la + 1
    # The parameter-gradient kernels flush with float atomics, so a step is bitwise reproducible only up to their order: the bound is
    # that run-to-run spread (~1e-12 here), not a change of arithmetic.
    same = 0
    for k in a1:
        assert b.keys() == a1.keys()
        same += torch.equal(b[k], a1[k])
        assert rel_l2(b[k], a1[k]) <= 1e-6, k
    print(f"{same} of {len(a1)} parameter gradients bitwise equal")


# ---- attribution --------------------------------------------------------------------------------------------------------------------
def _clf(kw, seed=31, precision="fp32"):
    spec = O.Spec(**kw, depth=2)
    m = make_encoder(spec)
    m.load_state_dict(O.synthetic_state_dict(spec, seed=seed), strict=True)
    m.precision = precision
    return m.to(DEV).train(), spec


def _ig64(m, spec, wins, target, steps, base):
    """float64 IG of windows [n, bands, w, w] at alpha_k = ig_alphas(steps) -> (attr, delta) in float64 (CPU)."""
    sd = {k: v.detach().double().cpu() for k, v in m.state_dict().items()}
    x = torch.as_tensor(wins).double()
    b = torch.as_tensor(base).double()[None, :, None, None]
    t = torch.as_tensor(target)
    nc = spec.num_classes
    valid = (t >= 0) & (t < nc)
    oh = torch.nn.functional.one_hot(torch.where(valid, t, 0), nc).permute(0, 3, 1, 2).double() * valid[:, None]
    a = ig_alphas(steps)
    xi = (b[:, None] + a[None, :, None, None, None] * (x[:, None] - b[:, None])).reshape(-1, *x.shape[1:]).requires_grad_(True)
    y = O.encoder_forward(xi, sd, spec)
    (g,) = torch.autograd.grad(y, xi, oh.repeat_interleave(steps, 0))
    attr = (x - b) * g.reshape(x.shape[0], steps, *x.shape[1:]).sum(1) / steps
    with torch.no_grad():
        F = lambda z: (O.encoder_forward(z, sd, spec) * oh).sum((1, 2, 3))
        delta = attr.sum((1, 2, 3)) - (F(x) - F(b.expand_as(x)))
        scale = attr.abs().sum((1, 2, 3)) + F(x).abs() + F(b.expand_as(x)).abs()
    return attr, delta, scale


def test_attribute_windows_vs_float64_ig():
    m, spec = _clf(O.HOUSTON)
    rng = np.random.default_rng(2)
    wins = torch.from_numpy(rng.standard_normal((3, 50, 8, 8)).astype(np.float32))
    target = torch.from_numpy(rng.integers(-1, 20, (3, 8, 8)))
    base = torch.from_numpy(0.3 * rng.standard_normal(50).astype(np.float32))
    attr, delta = attribute_windows(m, wins.to(DEV), target.to(DEV), steps=6, baseline=base)
    want, d64, scale = _ig64(m, spec, wins, target, 6, base)
    err = rel_l2(attr, want)
    print(f"attribute_windows rel-l2 {err:.2e}, delta {delta.tolist()} vs {d64.tolist()}")
    assert attr.dtype == torch.float32 and delta.dtype == torch.float64 and err <= 1e-5
    assert ((delta.cpu() - d64).abs() <= 1e-5 * scale).all()


def _scene_ig64(m, spec, cube, target, steps, stride, weight, base=None):
    cube = np.asarray(cube, dtype=np.float64)
    B, nb, H, W = cube.shape
    w = spec.image_size
    sy, sx = (stride, stride) if isinstance(stride, int) else stride
    ny, nx = scene_windows(H, W, w, (sy, sx))
    oy, ox = _origins(H, w, sy, ny), _origins(W, w, sx, nx)
    tg = np.asarray(target)
    wins = np.stack([cube[b, :, y:y + w, x:x + w] for b in range(B) for y in oy for x in ox])
    tw = np.stack([tg[b, y:y + w, x:x + w] for b in range(B) for y in oy for x in ox])
    base = np.zeros(nb) if base is None else np.asarray(base, dtype=np.float64)
    attr, _, _ = _ig64(m, spec, wins, torch.from_numpy(tw), steps, base)
    attr = attr.numpy().reshape(B, ny, nx, nb, w, w)
    wt = np.ones((w, w)) if weight is None else np.asarray(weight, dtype=np.float64)
    acc, ws = np.zeros((B, nb, H, W)), np.zeros((B, H, W))
    for b in range(B):
        for i, y in enumerate(oy):
            for j, x in enumerate(ox):
                acc[b, :, y:y + w, x:x + w] += wt * attr[b, i, j]
                ws[b, y:y + w, x:x + w] += wt
    return acc / ws[:, None]


SCENE_CASES = {   # name: (model kwargs, scene shape, stride, weight)
    "houston_gauss": (O.HOUSTON, (1, 50, 13, 12), 3, "gauss"),
    "p2x4_stride_3": (P2X4, (1, 48, 12, 13), 3, None),
}


@pytest.mark.parametrize("case", sorted(SCENE_CASES))
def test_attribute_scene_vs_float64_ig(case):
    kw, shape, stride, wkind = SCENE_CASES[case]
    m, spec = _clf(kw)
    rng = np.random.default_rng(7)
    cube = torch.from_numpy(rng.standard_normal(shape).astype(np.float32))
    target = torch.from_numpy(rng.integers(-1, spec.num_classes, (shape[0], *shape[2:])))
    weight = _gauss() if wkind else None
    attr = attribute_scene(m, cube.to(DEV), target.to(DEV), steps=4, stride=stride, weight=weight, batch_samples=4 * 5)
    want = _scene_ig64(m, spec, cube, target, 4, stride, weight)
    err = rel_l2(attr, want)
    print(f"{case}: rel-l2 {err:.2e}")
    assert attr.shape == shape and err <= 1e-5


def test_attribute_scene_raw_tiles_pad_bands_clip():
    means, stds, meta = _stats("houston")
    m, spec = _clf(O.HOUSTON)
    raw = torch.from_numpy(np.random.default_rng(9).integers(-400, 12000, (1, 48, 11, 14)).astype(np.int16)).to(DEV)
    clip = (-1.5, 1.5)
    rt = M.RawTiles(raw, means, stds, image_size=8, pad_bands=meta["pad"], clip=clip)
    target = torch.from_numpy(np.random.default_rng(1).integers(0, 20, (1, 11, 14))).to(DEV)
    attr = attribute_scene(m, rt, target, steps=3, stride=3, batch_samples=10)
    cube = O.input_pipeline(raw.cpu().numpy(), means, stds, 14, pad_bands=meta["pad"], clip=clip)
    want = _scene_ig64(m, spec, cube, target.cpu(), 3, 3, None)
    assert attr.shape == (1, 50, 11, 14) and (attr[:, 48:] == 0).all()
    err = rel_l2(attr, want)
    print(f"raw tiles: rel-l2 {err:.2e}")
    assert err <= 1e-5


def test_attribute_scene_chunking_and_stitching_bitwise():
    m, spec = _clf(O.HOUSTON)
    rng = np.random.default_rng(12)
    cube = torch.from_numpy(rng.standard_normal((2, 50, 16, 24)).astype(np.float32)).to(DEV)
    target = torch.from_numpy(rng.integers(-1, 20, (2, 16, 24))).to(DEV)
    steps = 3
    outs = [attribute_scene(m, cube, target, steps=steps, stride=8, batch_samples=bs) for bs in (steps, 7 * steps, 10 ** 6)]
    assert torch.equal(outs[0], outs[1]) and torch.equal(outs[0], outs[2])
    wins = cube.reshape(2, 50, 2, 8, 3, 8).permute(0, 2, 4, 1, 3, 5).reshape(12, 50, 8, 8)
    tw = target.reshape(2, 2, 8, 3, 8).permute(0, 1, 3, 2, 4).reshape(12, 8, 8)
    attr, _ = attribute_windows(m, wins.contiguous(), tw.contiguous(), steps=steps)
    stitched = attr.reshape(2, 2, 3, 50, 8, 8).permute(0, 3, 1, 4, 2, 5).reshape(2, 50, 16, 24)
    assert torch.equal(stitched, outs[0])
    # overlapping windows with a weight: the same chunk invariance
    o = [attribute_scene(m, cube, target, steps=steps, stride=3, weight=_gauss(), batch_samples=bs) for bs in (steps, 7 * steps)]
    assert torch.equal(o[0], o[1])


def test_scene_attribute_kernel_chunk_invariance_vs_float64():
    rng = np.random.default_rng(4)
    B, nb, H, W, w, steps, stride = 2, 7, 13, 11, 8, 5, (2, 3)
    ny, nx = scene_windows(H, W, w, stride)
    n = B * ny * nx
    grads = torch.from_numpy(rng.standard_normal((n * steps, nb, w, w)).astype(np.float32)).to(DEV)
    weight = torch.from_numpy(_gauss()).to(DEV)
    res = []
    for chunk in (1, 5, n):
        acc = torch.zeros(B, nb, H, W, device=DEV)
        wsum = torch.zeros(B, H, W, device=DEV)
        for first in range(0, n, chunk):
            k = min(chunk, n - first)
            attribute_sum(grads[first * steps:(first + k) * steps].contiguous(), acc, wsum, steps=steps, stride=stride, grid=(ny, nx),
                          first=first, weight=weight)
        res.append((acc, wsum))
    assert all(torch.equal(r[0], res[0][0]) and torch.equal(r[1], res[0][1]) for r in res)
    g = grads.cpu().double().numpy().reshape(B, ny, nx, steps, nb, w, w).sum(3)
    wt = _gauss().astype(np.float64)
    oy, ox = _origins(H, w, stride[0], ny), _origins(W, w, stride[1], nx)
    acc, ws = np.zeros((B, nb, H, W)), np.zeros((B, H, W))
    for b in range(B):
        for i, y in enumerate(oy):
            for j, x in enumerate(ox):
                acc[b, :, y:y + w, x:x + w] += wt * g[b, i, j]
                ws[b, y:y + w, x:x + w] += wt
    assert rel_l2(res[0][0], acc) <= 1e-6 and rel_l2(res[0][1], ws) <= 1e-6


def test_attribution_exact_zeros_side_effects_and_band_importance():
    m, spec = _clf(O.HOUSTON)
    rng = np.random.default_rng(5)
    base = torch.from_numpy(rng.standard_normal(50).astype(np.float32)).to(DEV)
    flat = base[None, :, None, None].expand(1, 50, 10, 9).contiguous()
    target = torch.from_numpy(rng.integers(0, 20, (1, 10, 9))).to(DEV)
    assert (attribute_scene(m, flat, target, steps=2, baseline=base, stride=2) == 0).all()           # baseline = x
    cube = torch.from_numpy(rng.standard_normal((1, 50, 10, 9)).astype(np.float32)).to(DEV)
    assert (attribute_scene(m, cube, torch.full_like(target, -1), steps=2, stride=2) == 0).all()     # nothing counted
    # a FusedAdam gradient arena stays zero; requires_grad and training mode are restored
    m.mlp_head[0].weight.requires_grad_(False)
    opt = FusedAdam(m.parameters(), lr=1e-3)
    opt.zero_grad()
    attr = attribute_scene(m, cube, target, steps=2, stride=2)
    torch.cuda.synchronize()
    assert float(opt.grad_arena.abs().max()) == 0.0
    assert m.training and not m.mlp_head[0].weight.requires_grad
    assert all(p.requires_grad for n, p in m.named_parameters() if n != "mlp_head.0.weight")
    assert all(p.grad is None for p in m.parameters())
    # band profiles on the device equal the host computation
    bi = band_importance(attr, target, num_classes=20)
    a, t = attr.abs().double().cpu(), target.cpu()
    want = torch.stack([a[0][:, t[0] == c].mean(1) if (t == c).any() else torch.full((50,), float("nan"), dtype=torch.float64)
                        for c in range(20)])
    assert torch.allclose(bi.cpu(), want, rtol=1e-12, equal_nan=True)
