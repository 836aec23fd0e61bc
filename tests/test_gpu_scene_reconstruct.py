"""GPU: whole-scene masked reconstruction (maskedsst_b200.inference.reconstruct_scene / reconstruct_windows, msst_scene_reconstruct in
csrc/scene.cu): the SimMIM decoder's predictions of the hidden scene entries, blended from overlapping windows, against a float64
oracle that runs O.simmim_forward on every window and blends in numpy."""
import ctypes

import numpy as np
import pytest
import torch

import maskedsst_b200 as M
from maskedsst_b200 import _lib
from maskedsst_b200.inference import reconstruct_scene, reconstruct_windows, reconstruction_metrics, scene_mask, scene_windows
from oracle import maskedsst_oracle as O
from tests.helpers import gold, rel_l2
from tests.test_gpu_parity import make_encoder

pytestmark = pytest.mark.gpu
DEV = "cuda"
P2X4 = dict(channels=48, num_classes=20, spatial_patch_size=2, spectral_patch_size=4)   # G = 4, C = 12, P = 16


def _sim(kw, seed, blockwise, depth=2, precision="fp32", ratio=0.7, mps=4, tube=True):
    spec = O.Spec(**kw, depth=depth)
    sd = O.synthetic_state_dict(spec, seed=seed, simmim=True, blockwise_decoder=blockwise)
    enc = make_encoder(spec)
    enc.precision = precision
    m = M.SimMIMSpatialSpectral(encoder=enc, masking_ratio=ratio, mask_patch_size=mps, tube_masking=tube,
                                to_pixels_per_spectral_block=blockwise)
    missing, unexpected = m.load_state_dict(sd, strict=False)
    assert not unexpected and all(k.startswith(("to_patch.", "patch_to_emb.")) for k in missing)
    return m.to(DEV).train(), spec, sd


def _gauss(w=8, sigma=2.0):
    yy, xx = np.meshgrid(np.arange(w) - (w - 1) / 2, np.arange(w) - (w - 1) / 2, indexing="ij")
    return np.exp(-(yy ** 2 + xx ** 2) / (2 * sigma ** 2)).astype(np.float32)


def _origins(extent, win, step, n):
    return np.minimum(np.arange(n) * step, extent - win)


def _oracle_recon(cube, mask, sd, spec, stride, weight, blockwise):
    """float64: per window, the token mask from the scene mask ("any" pixel of the patch, numpy loop), O.simmim_forward's embedding,
    mask-token select and encoder with every token decoded, the predictions put back at their pixels and blended over the covering
    windows in numpy.  -> (acc / wsum at the hidden entries, [B, C*p0, H, W] float64; hidden [B, C*p0, H, W] bool)."""
    cube, mask = np.asarray(cube, dtype=np.float64), np.asarray(mask)
    B, nb, H, W = cube.shape
    w, p0, p1, Cb = spec.image_size, spec.spectral_patch_size, spec.spatial_patch_size, spec.C
    G = w // p1
    sy, sx = (stride, stride) if isinstance(stride, int) else stride
    ny, nx = scene_windows(H, W, w, (sy, sx))
    oy, ox = _origins(H, w, sy, ny), _origins(W, w, sx, nx)
    wins, wmask = [], []
    for b in range(B):
        for y in oy:
            for x in ox:
                wins.append(cube[b, :, y:y + w, x:x + w])
                mw = mask[b, :, y:y + w, x:x + w].reshape(Cb, G, p1, G, p1).any(axis=(2, 4))
                wmask.append(mw.reshape(-1))
    wins, wmask = torch.from_numpy(np.stack(wins)), torch.from_numpy(np.stack(wmask))
    n = wins.shape[0]
    idx = torch.arange(spec.T)[None].expand(n, -1)
    sd64 = {k: v.double() for k, v in sd.items()}
    _, _, _, pred = O.simmim_forward(wins, sd64, spec, wmask, idx, blockwise_decoder=blockwise, return_parts=True)   # [n, T, P]
    img = pred.reshape(n, Cb, G, G, p0, p1, p1).permute(0, 1, 4, 2, 5, 3, 6).reshape(n, Cb * p0, w, w).numpy()
    img = img.reshape(B, ny, nx, Cb * p0, w, w)
    wt = np.ones((w, w)) if weight is None else np.asarray(weight, dtype=np.float64)
    acc, ws = np.zeros((B, Cb * p0, H, W)), np.zeros((B, H, W))
    for b in range(B):
        for i, y in enumerate(oy):
            for j, x in enumerate(ox):
                acc[b, :, y:y + w, x:x + w] += wt * img[b, i, j]
                ws[b, y:y + w, x:x + w] += wt
    hidden = np.repeat(mask, p0, axis=1)
    return acc / ws[:, None], hidden


def _stats(tag):
    import json
    g = gold("input_pipeline")
    return g[f"{tag}__means"], g[f"{tag}__stds"], json.loads(str(g[f"{tag}__meta"]))


CASES = {   # name: (model kwargs, blockwise decoder, scene shape, stride, weight, mask kind)
    "houston": (O.HOUSTON, False, (2, 50, 21, 19), 3, None, "scene_mask"),
    "houston_blockwise_gauss": (O.HOUSTON, True, (2, 50, 21, 19), 3, "gauss", "scene_mask"),
    "p2x4": (P2X4, True, (1, 48, 19, 22), 3, None, "sparse"),
    "p2x4_shared_stride_2_5": (P2X4, False, (1, 48, 19, 22), (2, 5), "gauss", "sparse"),
    "stride_window": (O.HOUSTON, True, (1, 50, 24, 21), 8, None, "scene_mask"),
    "spectral_only": (dict(**O.HOUSTON, spectral_only=True), True, (2, 50, 13, 12), 2, None, "per_block"),
}


def _mask(kind, model, shape, seed):
    B, _, H, W = shape
    Cb = model.encoder.num_spectral_patches
    if kind == "sparse":   # single pixels: the "any" rule and the sub-patch position matter
        return torch.from_numpy(np.random.default_rng(seed).random((B, Cb, H, W)) < 0.2).to(DEV)
    if kind == "per_block":
        model.tube_masking = False
    return scene_mask(model, B, H, W, seed=seed, device=DEV)


@pytest.mark.parametrize("case", sorted(CASES))
def test_reconstruct_scene_vs_float64_oracle(case):
    kw, blockwise, shape, stride, wkind, mkind = CASES[case]
    m, spec, sd = _sim(kw, 91, blockwise)
    cube = torch.from_numpy(np.random.default_rng(5).standard_normal(shape).astype(np.float32))
    mask = _mask(mkind, m, shape, 7)
    weight = _gauss() if wkind == "gauss" else None
    recon = reconstruct_scene(m, cube.to(DEV), mask, stride=stride, weight=weight)
    assert m.training and m.encoder.training                              # the training flags are restored
    assert recon.shape == shape and recon.dtype == torch.float32
    want, hidden = _oracle_recon(cube, mask.cpu(), sd, spec, stride, weight, blockwise)
    hidden_t = torch.from_numpy(hidden)
    r = recon.cpu()
    assert torch.equal(r[~hidden_t], cube[~hidden_t])                      # visible entries: the input, bit for bit
    err = rel_l2(r[hidden_t], want[hidden])
    print(f"{case}: {int(hidden.sum())} hidden entries, rel-l2 {err:.2e}")
    assert err <= 1e-5


def test_reconstruct_scene_raw_tiles_vs_oracle():
    """int16 Houston scene with its two zero pad bands and a clip: hidden pad bands are predicted, visible ones stay 0."""
    means, stds, meta = _stats("houston")
    m, spec, sd = _sim(O.HOUSTON, 92, True)
    raw = torch.from_numpy(np.random.default_rng(9).integers(-400, 12000, (1, 48, 17, 23)).astype(np.int16)).to(DEV)
    clip = (-1.5, 1.5)
    rt = M.RawTiles(raw, means, stds, image_size=8, pad_bands=meta["pad"], clip=clip)
    m.tube_masking = False
    mask = scene_mask(m, 1, 17, 23, seed=3, device=DEV)
    recon = reconstruct_scene(m, rt, mask, stride=4, batch_windows=5)
    cube = O.input_pipeline(raw.cpu().numpy(), means, stds, 23, pad_bands=meta["pad"], clip=clip)
    assert cube.shape == (1, 50, 17, 23)
    want, hidden = _oracle_recon(cube, mask.cpu(), sd, spec, 4, None, True)
    hidden_t = torch.from_numpy(hidden)
    r = recon.cpu()
    assert torch.equal(r[~hidden_t], cube[~hidden_t])
    assert hidden[:, 48:].any() and (r[:, 48:][~hidden_t[:, 48:]] == 0).all()
    err = rel_l2(r[hidden_t], want[hidden])
    print(f"raw tiles: rel-l2 {err:.2e}")
    assert err <= 1e-5
    # the metrics' target is the same standardised scene without the pad bands
    got = reconstruction_metrics(recon, rt, mask)
    h48 = hidden[:, :48]
    d = want[:, :48][h48] - cube[:, :48].double().numpy()[h48]
    assert got["count"] == int(h48.sum()) and got["per_band_count"].shape == (48,)
    assert got["l1"] == pytest.approx(np.abs(d).mean(), rel=1e-4)


@pytest.mark.parametrize("case", ["houston", "p2x4"])
def test_reconstruct_scene_chunk_invariant_bitwise(case):
    kw, blockwise, shape, stride, wkind, mkind = CASES[case]
    m, _, _ = _sim(kw, 93, blockwise)
    cube = torch.randn(*shape, device=DEV)
    mask = _mask(mkind, m, shape, 8)
    ny, nx = scene_windows(shape[2], shape[3], 8, stride)
    out = [reconstruct_scene(m, cube, mask, stride=stride, weight=_gauss(), batch_windows=bw) for bw in (1, 7, shape[0] * ny * nx)]
    for r in out[1:]:
        assert torch.equal(r, out[0])


@pytest.mark.parametrize("D,C,p0,p1,n_wb", [(32, 3, 4, 2, 3), (96, 5, 10, 1, 1), (256, 2, 1, 4, 2), (160, 4, 2, 2, 1)])
@pytest.mark.parametrize("stride", [(2, 5), (1, 1)])
def test_reconstruct_windows_chunk_invariant_bitwise(D, C, p0, p1, n_wb, stride):
    B, H, W, w = 2, 21, 19, 8
    G, P = w // p1, p0 * p1 * p1
    ny, nx = scene_windows(H, W, w, stride)
    n = B * ny * nx
    g = torch.Generator(device=DEV).manual_seed(D + p1)
    tokens = torch.randn(n, C * G * G, D, device=DEV, generator=g)
    Wd = torch.randn(n_wb, P, D, device=DEV, generator=g) / D ** 0.5
    bd = torch.randn(n_wb, P, device=DEV, generator=g)
    mask = torch.rand(B, C, H, W, device=DEV, generator=g) < 0.5
    weight = torch.rand(w, w, device=DEV, generator=g) + 0.1
    res = []
    for chunk in (1, 7, n):
        acc = torch.zeros(B, C * p0, H, W, device=DEV)
        wsum = torch.zeros(B, H, W, device=DEV)
        for first in range(0, n, chunk):
            reconstruct_windows(tokens[first:first + chunk], mask, Wd, bd, acc, wsum, C=C, p0=p0, p1=p1, stride=stride, grid=(ny, nx),
                                first=first, weight=weight)
        res.append((acc, wsum))
    for acc, wsum in res[1:]:
        assert torch.equal(acc, res[0][0]) and torch.equal(wsum, res[0][1])
    # float64: decode every token, put the predictions at their pixels, blend the hidden entries
    t64 = tokens.double().reshape(n, C, G * G, D)
    blk = torch.arange(C, device=DEV) if n_wb == C else torch.zeros(C, dtype=torch.long, device=DEV)
    pred = torch.einsum("ncsd,cpd->ncsp", t64, Wd.double()[blk]) + bd.double()[blk][None, :, None, :]
    img = pred.reshape(n, C, G, G, p0, p1, p1).permute(0, 1, 4, 2, 5, 3, 6).reshape(B, ny, nx, C * p0, w, w).cpu().numpy()
    oy, ox = _origins(H, w, stride[0], ny), _origins(W, w, stride[1], nx)
    wt = weight.double().cpu().numpy()
    acc, ws = np.zeros((B, C * p0, H, W)), np.zeros((B, H, W))
    for b in range(B):
        for i, y in enumerate(oy):
            for j, x in enumerate(ox):
                acc[b, :, y:y + w, x:x + w] += wt * img[b, i, j]
                ws[b, y:y + w, x:x + w] += wt
    hidden = np.repeat(mask.cpu().numpy(), p0, axis=1)
    got = res[0][0].cpu().numpy()
    assert (got[~hidden] == 0).all()
    assert rel_l2(got[hidden], acc[hidden]) <= 1e-6 and rel_l2(res[0][1], ws) <= 1e-6


def test_no_leakage_of_hidden_values():
    """Whatever the hidden entries hold (finite garbage, NaN; the int16 sentinel for raw tiles), recon is bitwise the same."""
    m, _, _ = _sim(P2X4, 94, True)
    shape = (1, 48, 19, 22)
    cube = torch.randn(*shape, device=DEV)
    mask = _mask("sparse", m, shape, 9)
    hidden = mask.repeat_interleave(4, 1)
    ref = reconstruct_scene(m, cube, mask, stride=3)
    assert torch.isfinite(ref).all()
    for fill in (lambda t: 1e3 * torch.randn_like(t), lambda t: torch.full_like(t, float("nan"))):
        bad = torch.where(hidden, fill(cube), cube)
        assert torch.equal(reconstruct_scene(m, bad, mask, stride=3), ref)
    means, stds, meta = _stats("houston")
    mh, _, _ = _sim(O.HOUSTON, 95, False)
    raw = torch.from_numpy(np.random.default_rng(10).integers(-400, 12000, (1, 48, 17, 23)).astype(np.int16)).to(DEV)
    mask = scene_mask(mh, 1, 17, 23, seed=4, device=DEV)
    rt = M.RawTiles(raw, means, stds, image_size=8, pad_bands=meta["pad"])
    ref = reconstruct_scene(mh, rt, mask, stride=4)
    bad = torch.where(mask.repeat_interleave(10, 1)[:, :48], torch.full_like(raw, -32768), raw)
    out = reconstruct_scene(mh, M.RawTiles(bad, means, stds, image_size=8, pad_bands=meta["pad"]), mask, stride=4)
    assert torch.isfinite(out).all() and torch.equal(out, ref)


@pytest.mark.parametrize("blockwise", [False, True])
def test_metrics_tie_to_the_training_loss(blockwise):
    """One window, exactly nm hidden (block, pixel) entries: reconstruction_metrics' l1 / nm is SimMIM's loss on that mask."""
    m, spec, _ = _sim(O.HOUSTON, 96, blockwise)
    img = torch.randn(1, 50, 8, 8, device=DEV)
    nm = 157
    sel = torch.from_numpy(np.sort(np.random.default_rng(11).permutation(spec.T)[:nm])).to(DEV)
    wmask = torch.zeros(1, spec.T, dtype=torch.bool, device=DEV)
    wmask[0, sel] = True
    mask = wmask.reshape(1, spec.C, 8, 8)
    with torch.no_grad():
        loss = float(m(img, masks=(wmask, sel[None])))
    got = reconstruction_metrics(reconstruct_scene(m, img, mask), img, mask)
    assert got["count"] == nm * spec.spectral_patch_size
    print(f"l1 / nm = {got['l1'] / nm:.9g}, loss = {loss:.9g}")
    assert got["l1"] / nm == pytest.approx(loss, rel=1e-6)


def test_bf16_close_to_fp32():
    means, stds, _ = _stats("enmap")
    raw = torch.from_numpy(np.random.default_rng(12).integers(-400, 12000, (1, 200, 27, 22)).astype(np.int16)).to(DEV)
    rt = M.RawTiles(raw, means, stds, image_size=8, clip=(-2.0, 2.0))
    m32, _, _ = _sim(O.ENMAP, 97, True)
    m16, _, _ = _sim(O.ENMAP, 97, True, precision="bf16")
    mask = scene_mask(m32, 1, 27, 22, seed=6, device=DEV)
    r32 = reconstruct_scene(m32, rt, mask, stride=4)
    r16 = reconstruct_scene(m16, rt, mask, stride=4, batch_windows=10)
    hidden = mask.repeat_interleave(10, 1)
    assert torch.isfinite(r16).all() and torch.equal(r16[~hidden], r32[~hidden])
    err = rel_l2(r16[hidden], r32[hidden])
    print(f"bf16 vs fp32 rel-l2 {err:.2e}")
    assert err <= 1e-2


def test_c_abi_limits_leave_outputs_untouched():
    L = _lib.lib()
    B, H, W, D, Cb, p0, p1 = 1, 21, 19, 96, 5, 10, 1
    tokens = torch.randn(30, Cb * 64, D, device=DEV)
    mask = torch.ones(B, Cb, H, W, dtype=torch.uint8, device=DEV)
    Wd, bd = torch.randn(Cb, p0, D, device=DEV), torch.randn(Cb, p0, device=DEV)
    acc = torch.full((B, Cb * p0, H, W), 7.0, device=DEV)
    wsum = torch.full((B, H, W), 3.0, device=DEV)
    ok = dict(B=B, D=D, H=H, W=W, win=8, stride_y=3, stride_x=3, win_y=6, win_x=5, win_first=0, n=30, C=Cb, p0=p0, p1=p1, n_wb=Cb)
    stream = torch.cuda.current_stream().cuda_stream
    for kw in (dict(D=80), dict(D=288), dict(p0=17), dict(n_wb=2), dict(p1=3), dict(stride_y=0), dict(win_y=7), dict(n=31),
               dict(C=1000)):
        d = dict(ok)
        d.update(kw)
        dims = _lib.SceneReconstructDims(*[d[k] for k, _ in _lib.SceneReconstructDims._fields_])
        assert L.msst_scene_reconstruct(ctypes.byref(dims), tokens.data_ptr(), mask.data_ptr(), Wd.data_ptr(), bd.data_ptr(), None,
                                        acc.data_ptr(), wsum.data_ptr(), stream) == 1, kw
    dims = _lib.SceneReconstructDims(*ok.values())
    assert L.msst_scene_reconstruct(ctypes.byref(dims), None, mask.data_ptr(), Wd.data_ptr(), bd.data_ptr(), None, acc.data_ptr(),
                                    wsum.data_ptr(), stream) == 1
    torch.cuda.synchronize()
    assert (acc == 7.0).all() and (wsum == 3.0).all()


def test_reconstruct_scene_argument_checks_on_the_device():
    m, _, _ = _sim(O.HOUSTON, 98, False)
    cube = torch.zeros(1, 50, 20, 20, device=DEV)
    mask = torch.zeros(1, 5, 20, 20, dtype=torch.bool, device=DEV)
    with pytest.raises(ValueError, match="mask must be a bool tensor"):
        reconstruct_scene(m, cube, mask.cpu())
    with pytest.raises(ValueError, match="stride"):
        reconstruct_scene(m, cube, mask, stride=9)
    with pytest.raises(ValueError, match="weight"):
        reconstruct_scene(m, cube, mask, weight=torch.ones(4, 4))
    m.eval()
    r = reconstruct_scene(m, cube, mask, stride=4)
    assert not m.training and torch.equal(r, cube)                         # nothing hidden: the input comes back
