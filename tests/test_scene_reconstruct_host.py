"""CPU: the argument checks of msst_scene_reconstruct (MSST_ERR_ARG before any CUDA call), of reconstruct_scene / reconstruct_windows
(ValueError before any device work), scene_mask, the window-mask rule against a numpy loop, and reconstruction_metrics against
term-by-term numpy."""
import ctypes as C
import math

import numpy as np
import pytest
import torch

import maskedsst_b200 as M
from maskedsst_b200 import _lib
from maskedsst_b200.inference import (_patch_any, _window_mask, reconstruct_scene, reconstruct_windows, reconstruction_metrics,
                                      scene_mask, scene_windows)


class _FakeCuda(torch.Tensor):
    """A CPU tensor that claims to live on a CUDA device, so that the checks after the device check can run without one."""
    @property
    def is_cuda(self):
        return True


def _t(*shape, dtype=torch.float32):
    return torch.zeros(*shape, dtype=dtype).as_subclass(_FakeCuda)


def _enc(p1=1, p0=10, channels=50, **kw):
    return M.ViTSpatialSpectral(image_size=8, spatial_patch_size=p1, spectral_patch_size=p0, num_classes=20, dim=96, depth=1, heads=8,
                                mlp_dim=64, channels=channels, spectral_pos_embed=False, **kw)


def _sim(p1=1, p0=10, channels=50, ratio=0.7, mps=4, tube=True, blockwise=False, **kw):
    return M.SimMIMSpatialSpectral(encoder=_enc(p1, p0, channels, **kw), masking_ratio=ratio, mask_patch_size=mps, tube_masking=tube,
                                   to_pixels_per_spectral_block=blockwise)


# ---- msst_scene_reconstruct ------------------------------------------------------------------------------------------------------
_OK = dict(B=1, D=96, H=21, W=19, win=8, stride_y=3, stride_x=3, win_y=6, win_x=5, win_first=0, n=30, C=5, p0=10, p1=1, n_wb=1)


def _rec(**kw):
    d = dict(_OK)
    d.update(kw)
    dims = _lib.SceneReconstructDims(*[d[k] for k, _ in _lib.SceneReconstructDims._fields_])
    return _lib.lib().msst_scene_reconstruct(C.byref(dims), 1, 1, 1, 1, None, 1, 1, None)


@pytest.mark.parametrize("kw, what", [
    (dict(D=80), b"D=80"), (dict(D=288), b"D=288"), (dict(D=16), b"D=16"), (dict(p0=17), b"p0*p1^2 = 17"),
    (dict(p0=5, p1=2), b"p0*p1^2 = 20"), (dict(p0=1, p1=5, win=10), b"p0*p1^2 = 25"), (dict(n_wb=2), b"n_wb=2"),
    (dict(n_wb=6), b"n_wb=6"), (dict(p0=4, p1=2, win=9, H=21), b"multiple"), (dict(C=1000, p0=2), b"shared memory"),
    (dict(win_first=-1), b"outside"), (dict(n=31), b"outside"), (dict(win_first=29, n=2), b"outside"), (dict(n=0), b"outside"),
    (dict(B=2, n=61), b"outside"), (dict(stride_y=0), b"stride"), (dict(stride_x=9), b"stride"), (dict(H=7), b"smaller"),
    (dict(win_y=7), b"grid"), (dict(win_x=6), b"grid"), (dict(B=0), b"bad dims"), (dict(D=0), b"bad dims"), (dict(C=0), b"bad dims"),
    (dict(p0=0), b"bad dims"), (dict(p1=0), b"bad dims"), (dict(n_wb=0), b"bad dims"),
])
def test_scene_reconstruct_argument_checks_without_a_device(kw, what):
    assert _rec(**kw) == 1, kw
    msg = _lib.lib().msst_last_error()
    assert msg.startswith(b"scene_reconstruct:") and what in msg, (kw, msg)


def test_scene_reconstruct_null_pointers_rejected():
    L = _lib.lib()
    dims = _lib.SceneReconstructDims(*_OK.values())
    ptrs = [1, 1, 1, 1, None, 1, 1]
    for i in (0, 1, 2, 3, 5, 6):    # tokens, mask, W, bias, acc, wsum (weight may be NULL)
        args = list(ptrs)
        args[i] = None
        assert L.msst_scene_reconstruct(C.byref(dims), *args, None) == 1
        assert b"must be set" in L.msst_last_error()
    assert L.msst_scene_reconstruct(None, *ptrs, None) == 1
    assert b"bad dims" in L.msst_last_error()
    assert L.msst_version() == 102


# ---- reconstruct_scene / reconstruct_windows -------------------------------------------------------------------------------------
def test_reconstruct_scene_refuses_models_it_cannot_decode():
    cube, mask = _t(1, 50, 10, 10), _t(1, 5, 10, 10, dtype=torch.bool)
    with pytest.raises(ValueError, match="SimMIMSpatialSpectral"):
        reconstruct_scene(_enc(), cube, mask)
    v1 = M.ViTSpatialSpectral_V1(image_size=8, spatial_patch_size=1, spectral_patch_size=10, num_classes=20, dim=96, depth=1, heads=8,
                                 mlp_dim=64, channels=50)
    with pytest.raises(ValueError, match="ViTSpatialSpectral encoder"):
        reconstruct_scene(M.SimMIMSpatialSpectral(encoder=v1, masking_ratio=0.5), cube, mask)
    for blockwise in (False, True):
        with pytest.raises(ValueError, match="blockwise patch embedding"):
            reconstruct_scene(_sim(blockwise_patch_embed=False, blockwise=blockwise), cube, mask)


@pytest.mark.parametrize("scene, mask, match", [
    (torch.zeros(1, 50, 10, 10), torch.zeros(1, 5, 10, 10, dtype=torch.bool), "CUDA"),
    (_t(50, 10, 10), _t(1, 5, 10, 10, dtype=torch.bool), r"\[B, C, H, W\]"),
    (_t(1, 40, 10, 10), _t(1, 4, 10, 10, dtype=torch.bool), "40 bands, the model 50"),
    (_t(1, 50, 10, 10), _t(1, 5, 10, 10, dtype=torch.uint8), "mask must be a bool tensor"),
    (_t(1, 50, 10, 10), _t(1, 50, 10, 10, dtype=torch.bool), "mask must be a bool tensor"),
    (_t(1, 50, 10, 10), _t(2, 5, 10, 10, dtype=torch.bool), "mask must be a bool tensor"),
    (_t(1, 50, 10, 10), _t(1, 5, 10, 9, dtype=torch.bool), "mask must be a bool tensor"),
    (_t(1, 50, 10, 10), torch.zeros(1, 5, 10, 10, dtype=torch.bool, device="meta"), "on cpu"),
    (_t(1, 50, 10, 10), np.zeros((1, 5, 10, 10), dtype=bool), "mask must be a bool tensor"),
])
def test_reconstruct_scene_argument_errors(scene, mask, match):
    with pytest.raises(ValueError, match=match):
        reconstruct_scene(_sim(), scene, mask)


def test_reconstruct_scene_raw_tiles_band_count():
    raw = _t(1, 46, 10, 10, dtype=torch.int16)
    rt = M.RawTiles(raw, np.zeros(46), np.ones(46), image_size=8, pad_bands=2)
    with pytest.raises(ValueError, match="48 bands, the model 50"):
        reconstruct_scene(_sim(), rt, _t(1, 5, 10, 10, dtype=torch.bool))


def _rw(**kw):
    a = dict(tokens=_t(9, 5 * 64, 96), mask=_t(1, 5, 20, 20, dtype=torch.uint8), W=_t(1, 10, 96), bias=_t(1, 10), acc=_t(1, 50, 20, 20),
             wsum=_t(1, 20, 20), C=5, p0=10, p1=1, weight=None)
    a.update(kw)
    reconstruct_windows(a["tokens"], a["mask"], a["W"], a["bias"], a["acc"], a["wsum"], C=a["C"], p0=a["p0"], p1=a["p1"], stride=(8, 8),
                        grid=(3, 3), first=0, weight=a["weight"])


@pytest.mark.parametrize("kw, match", [
    (dict(tokens=torch.zeros(9, 320, 96)), "tokens must be a contiguous fp32 CUDA"),
    (dict(tokens=_t(9, 320, 96, dtype=torch.float64)), "tokens must be"),
    (dict(W=_t(1, 96, 10).transpose(1, 2)), "W must be"),
    (dict(bias=_t(1, 10, dtype=torch.float16)), "bias must be"),
    (dict(acc=torch.zeros(1, 50, 20, 20)), "acc must be"),
    (dict(wsum=None), "wsum must be"),
    (dict(weight=torch.ones(8, 8)), "weight must be"),
    (dict(mask=torch.zeros(1, 5, 20, 20, dtype=torch.uint8)), "mask must be"),
    (dict(mask=_t(1, 5, 20, 20, dtype=torch.int32)), "mask must be"),
    (dict(mask=_t(1, 5, 20, 40, dtype=torch.uint8)[..., ::2]), "mask must be"),
    (dict(tokens=_t(9, 320, 48)), "disagree"),
    (dict(tokens=_t(9, 300, 96)), "disagree"),
    (dict(tokens=_t(320, 96)), r"tokens must be \[n, C\*S, D\]"),
    (dict(C=4), "disagree"),
    (dict(p0=0), r"tokens must be \[n"),
    (dict(acc=_t(1, 48, 20, 20)), "disagree"),
    (dict(mask=_t(1, 50, 20, 20, dtype=torch.uint8)), "disagree"),
    (dict(wsum=_t(20, 20)), "disagree"),
    (dict(W=_t(2, 10, 96), bias=_t(2, 10)), "disagree"),
    (dict(W=_t(1, 16, 96), bias=_t(1, 16)), "disagree"),
    (dict(W=_t(1, 10, 64)), "disagree"),
    (dict(bias=_t(5, 10)), "disagree"),
    (dict(weight=_t(4, 4)), "disagree"),
    (dict(W=_t(10, 96)), r"W \[n_wb, P, D\]"),
])
def test_reconstruct_windows_argument_errors(kw, match):
    with pytest.raises(ValueError, match=match):
        _rw(**kw)


# ---- scene_mask ------------------------------------------------------------------------------------------------------------------
def _cells(mask, mps):
    """[B, C, H, W] -> [B, C, ceil(H / mps), ceil(W / mps)]: each cell's top-left pixel, after checking every cell is uniform."""
    B, Cb, H, W = mask.shape
    cells = mask[:, :, ::mps, ::mps]
    up = cells.repeat_interleave(mps, 2).repeat_interleave(mps, 3)[:, :, :H, :W]
    assert torch.equal(up, mask), "a cell is not uniformly masked"
    return cells


@pytest.mark.parametrize("ratio, mps, tube, H, W", [(0.7, 4, True, 21, 19), (0.7, 4, False, 21, 19), (0.5, 2, True, 8, 8),
                                                    (0.6, 1, False, 5, 7), (0.3, 8, True, 17, 9), (0.75, 4, False, 9, 9)])
def test_scene_mask_counts_cells_and_blocks(ratio, mps, tube, H, W):
    sim = _sim(ratio=ratio, mps=mps, tube=tube)
    B, Cb = 3, sim.encoder.num_spectral_patches
    m = scene_mask(sim, B, H, W, seed=5, device="cpu")
    assert m.shape == (B, Cb, H, W) and m.dtype == torch.bool and m.is_contiguous()
    cells = _cells(m, mps)
    ncells = math.ceil(H / mps) * math.ceil(W / mps)
    assert cells.shape[2] * cells.shape[3] == ncells
    want = int(np.ceil(ncells * ratio))
    assert (cells.reshape(B, Cb, -1).sum(-1) == want).all()
    if tube:
        assert torch.equal(m, m[:, :1].expand_as(m))
    else:
        assert any(not torch.equal(m[b, 0], m[b, c]) for b in range(B) for c in range(1, Cb))
        assert not torch.equal(m[0], m[1])


def test_scene_mask_partial_border_cells():
    """21 x 19 with 4-pixel cells: the last cell row holds one pixel row and the last cell column three columns; both are drawn."""
    sim = _sim(ratio=0.5, mps=4, tube=True)
    seen = torch.zeros(6, 5, dtype=torch.bool)
    for seed in range(20):
        cells = _cells(scene_mask(sim, 1, 21, 19, seed=seed, device="cpu"), 4)[0, 0]
        assert cells.shape == (6, 5)
        seen |= cells
    assert seen[5].any() and seen[:, 4].any() and seen[5, 4]


def test_scene_mask_seed_reproducible_and_documented_draw():
    sim = _sim(ratio=0.7, mps=4, tube=False)
    a = scene_mask(sim, 2, 13, 10, seed=11, device="cpu")
    assert torch.equal(a, scene_mask(sim, 2, 13, 10, seed=11, device="cpu"))
    assert not torch.equal(a, scene_mask(sim, 2, 13, 10, seed=12, device="cpu"))
    # the documented draw: a CPU generator, rows in (scene, block) order, one randperm each
    g = torch.Generator().manual_seed(11)
    ncells = 4 * 3
    for b in range(2):
        for c in range(5):
            want = torch.zeros(ncells, dtype=torch.bool)
            want[torch.randperm(ncells, generator=g)[:9]] = True
            assert torch.equal(a[b, c, ::4, ::4].reshape(-1), want)


@pytest.mark.parametrize("kw, match", [(dict(B=0), "B=0"), (dict(H=-1), "H=-1"), (dict(W=2.0), "W=2.0"), (dict(B=True), "B=True"),
                                       (dict(seed=-1), "seed=-1"), (dict(seed=1.5), "seed=1.5")])
def test_scene_mask_argument_errors(kw, match):
    a = dict(B=1, H=8, W=8, seed=0)
    a.update(kw)
    with pytest.raises(ValueError, match=match):
        scene_mask(_sim(), a["B"], a["H"], a["W"], seed=a["seed"], device="cpu")
    with pytest.raises(ValueError, match="SimMIMSpatialSpectral"):
        scene_mask(_enc(), 1, 8, 8, device="cpu")


# ---- the window-mask rule --------------------------------------------------------------------------------------------------------
def _window_mask_loop(mask, p1, w, stride, first, n):
    """numpy: token (c, s) of window g is masked when any pixel of patch s in that window has block c set in the scene mask."""
    mask = np.asarray(mask)
    B, Cb, H, W = mask.shape
    ny, nx = scene_windows(H, W, w, stride)
    G = w // p1
    out = np.zeros((n, Cb * G * G), dtype=bool)
    for k, g in enumerate(range(first, first + n)):
        b, r = divmod(g, ny * nx)
        oy, ox = min((r // nx) * stride[0], H - w), min((r % nx) * stride[1], W - w)
        for c in range(Cb):
            for h in range(G):
                for v in range(G):
                    y, x = oy + h * p1, ox + v * p1
                    out[k, c * G * G + h * G + v] = mask[b, c, y:y + p1, x:x + p1].any()
    return out


@pytest.mark.parametrize("p1, stride, shape, chunk", [(1, (3, 3), (2, 5, 21, 19), (0, 60)), (2, (3, 3), (2, 12, 19, 22), (7, 30)),
                                                      (2, (2, 5), (1, 12, 13, 30), (3, 11)), (4, (1, 1), (1, 3, 9, 10), (0, 6)),
                                                      (2, (8, 8), (1, 12, 16, 17), (0, 4))])
def test_window_mask_any_rule_against_numpy_loop(p1, stride, shape, chunk):
    rng = np.random.default_rng(p1 * 7 + stride[1])
    mask = torch.from_numpy(rng.random(shape) < 0.15)
    ny, nx = scene_windows(shape[2], shape[3], 8, stride)
    got = _window_mask(_patch_any(mask, p1), p1, 8, stride, (ny, nx), *chunk)
    want = _window_mask_loop(mask, p1, 8, stride, *chunk)
    assert got.dtype == torch.bool and np.array_equal(got.numpy(), want)
    if p1 > 1:   # a sparse mask: "any" differs from "all" and from the patch's top-left pixel alone
        assert want.sum() > _window_mask(mask, 1, 8, stride, (ny, nx), *chunk).reshape(chunk[1], shape[1], 8, 8)[
            :, :, ::p1, ::p1].sum()


# ---- reconstruction_metrics ------------------------------------------------------------------------------------------------------
def _metrics_loop(recon, target, mask, p0):
    recon, target, mask = (np.asarray(a) for a in (recon, target, mask))
    nb = target.shape[1]
    l1, sq, tb, cnt = np.zeros(nb), np.zeros(nb), np.zeros(nb), np.zeros(nb, dtype=np.int64)
    for b, band, y, x in np.ndindex(*target.shape):
        if mask[b, band // p0, y, x]:
            d = float(recon[b, band, y, x]) - float(target[b, band, y, x])
            l1[band] += abs(d)
            sq[band] += d * d
            tb[band] += abs(float(target[b, band, y, x]))
            cnt[band] += 1
    n = cnt.sum()
    return dict(count=n, l1=l1.sum() / n, rmse=math.sqrt(sq.sum() / n), baseline_l1=tb.sum() / n, per_band_count=cnt,
                per_band_l1=l1 / cnt, per_band_rmse=np.sqrt(sq / cnt))


def _check_metrics(got, want):
    assert got["count"] == want["count"]
    for k in ("l1", "rmse", "baseline_l1"):
        assert got[k] == pytest.approx(want[k], rel=1e-12), k
    assert np.array_equal(got["per_band_count"].numpy(), want["per_band_count"])
    for k in ("per_band_l1", "per_band_rmse"):
        assert got[k].dtype == torch.float64
        np.testing.assert_allclose(got[k].numpy(), want[k], rtol=1e-12)


def test_reconstruction_metrics_against_numpy():
    rng = np.random.default_rng(3)
    scene = torch.from_numpy(rng.standard_normal((2, 12, 6, 7)).astype(np.float32))
    recon = scene + torch.from_numpy(rng.standard_normal(scene.shape).astype(np.float32))
    mask = torch.from_numpy(rng.random((2, 3, 6, 7)) < 0.4)
    recon[~mask.repeat_interleave(4, 1)] = float("nan")       # visible entries do not enter
    got = reconstruction_metrics(recon, scene, mask)
    _check_metrics(got, _metrics_loop(recon, scene, mask, 4))
    assert got["per_band_l1"].shape == (12,)


def test_reconstruction_metrics_raw_tiles_leave_out_pad_bands():
    rng = np.random.default_rng(4)
    raw = torch.from_numpy(rng.integers(-400, 12000, (1, 48, 5, 6)).astype(np.int16))
    means, stds = rng.uniform(1000, 3000, 48), rng.uniform(500, 1500, 48)
    rt = M.RawTiles(raw.as_subclass(_FakeCuda), means, stds, image_size=4, pad_bands=2, clip=(-1.0, 1.5))
    target = ((raw.double() - torch.from_numpy(means)[:, None, None]) / torch.from_numpy(stds)[:, None, None]).float().clamp(-1.0, 1.5)
    recon = torch.from_numpy(rng.standard_normal((1, 50, 5, 6)).astype(np.float32))
    mask = torch.from_numpy(rng.random((1, 5, 5, 6)) < 0.5)
    mask[0, 4] = True                                          # the last block holds the two pad bands
    got = reconstruction_metrics(recon, rt, mask)
    want = _metrics_loop(recon[:, :48], target, mask, 10)
    _check_metrics(got, want)
    assert got["per_band_count"].shape == (48,) and int(got["per_band_count"][-1]) == 30


def test_reconstruction_metrics_empty_mask_and_errors():
    scene = torch.randn(1, 50, 4, 4)
    got = reconstruction_metrics(scene, scene, torch.zeros(1, 5, 4, 4, dtype=torch.bool))
    assert got["count"] == 0 and all(math.isnan(got[k]) for k in ("l1", "rmse", "baseline_l1"))
    assert torch.isnan(got["per_band_l1"]).all() and (got["per_band_count"] == 0).all()
    mask = torch.ones(1, 5, 4, 4, dtype=torch.bool)
    for recon, m, match in [(scene[:, :40], mask, "recon has 40 bands"), (scene[0], mask, "recon must be"),
                            (scene, torch.ones(1, 7, 4, 4, dtype=torch.bool), "C dividing"), (scene, mask.to(torch.uint8), "bool"),
                            (scene, mask[:, :, :3], "mask must be a bool tensor")]:
        with pytest.raises(ValueError, match=match):
            reconstruction_metrics(recon, scene, m)
