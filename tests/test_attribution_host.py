"""CPU: the argument checks of msst_patch_embed_bwd_data / msst_scene_attribute (MSST_ERR_ARG before any CUDA call) and of
attribute_windows / attribute_scene (ValueError before any device work), the IG step schedule, the interpolated-window gather against a
numpy loop, and band_importance against brute force."""
import ctypes as C

import numpy as np
import pytest
import torch

import maskedsst_b200 as M
from maskedsst_b200 import _lib
from maskedsst_b200.inference import (_gather_windows, _interpolate, attribute_scene, attribute_windows, band_importance, ig_alphas,
                                      scene_windows)
from tests.test_scene_reconstruct_host import _enc, _sim, _t


# ---- C limits -----------------------------------------------------------------------------------------------------------------------
def _embed_dims(**kw):
    d = dict(B=1, C=5, G=8, p0=10, p1=1, D=96, n_weight_blocks=5, drop_p=0.0, seed=0, seed_dev=None, raw=None)
    d.update(kw)
    return _lib.EmbedDims(*[d[k] for k, _ in _lib.EmbedDims._fields_])


@pytest.mark.parametrize("kw, what", [
    (dict(D=160), b"D=160"), (dict(D=80), b"D=80"), (dict(D=0), b"D=0"), (dict(n_weight_blocks=2), b"n_weight_blocks"),
    (dict(drop_p=1.5), b"drop_p"), (dict(drop_p=float("nan")), b"drop_p"), (dict(C=1, p0=65, n_weight_blocks=1), b"65 > 64"),
    (dict(p1=9, p0=1, C=50, G=1, n_weight_blocks=1), b"81 > 64"), (dict(B=0), b"bad dims"), (dict(G=0), b"bad dims"),
])
def test_patch_embed_bwd_data_argument_checks_without_a_device(kw, what):
    L = _lib.lib()
    assert L.msst_patch_embed_bwd_data(C.byref(_embed_dims(**kw)), *([1] * 8), 1, None, 1, None) == 1, kw
    msg = L.msst_last_error()
    assert msg.startswith(b"patch_embed") and what in msg, (kw, msg)


def test_patch_embed_bwd_data_pointer_checks():
    L = _lib.lib()
    raw = _lib.RawInput()
    assert L.msst_patch_embed_bwd_data(C.byref(_embed_dims(raw=C.pointer(raw))), *([1] * 8), 1, None, 1, None) == 1
    assert b"raw tiles have no gradient" in L.msst_last_error()
    for i in (0, 8, 10):     # img, d_tokens, d_img
        args = [1] * 8 + [1, None, 1]
        args[i] = None
        assert L.msst_patch_embed_bwd_data(C.byref(_embed_dims()), *args, None) == 1
        assert b"must be set" in L.msst_last_error()
    assert L.msst_patch_embed_bwd_data(None, *([1] * 8), 1, None, 1, None) == 1
    assert b"bad dims" in L.msst_last_error()


_OK = dict(B=1, bands=50, H=21, W=19, win=8, stride_y=3, stride_x=3, win_y=6, win_x=5, win_first=0, n=30, steps=4)


def _attr(**kw):
    d = dict(_OK)
    d.update(kw)
    dims = _lib.SceneAttributeDims(*[d[k] for k, _ in _lib.SceneAttributeDims._fields_])
    return _lib.lib().msst_scene_attribute(C.byref(dims), 1, None, 1, 1, None)


@pytest.mark.parametrize("kw, what", [
    (dict(steps=0), b"bad dims"), (dict(bands=0), b"bad dims"), (dict(B=0), b"bad dims"), (dict(win=0), b"bad dims"),
    (dict(win_first=-1), b"outside"), (dict(n=31), b"outside"), (dict(n=0), b"outside"), (dict(B=2, n=61), b"outside"),
    (dict(stride_y=0), b"stride"), (dict(stride_x=9), b"stride"), (dict(H=7), b"smaller"), (dict(win_y=7), b"grid"),
    (dict(win_x=6), b"grid"),
])
def test_scene_attribute_argument_checks_without_a_device(kw, what):
    assert _attr(**kw) == 1, kw
    msg = _lib.lib().msst_last_error()
    assert msg.startswith(b"scene_attribute:") and what in msg, (kw, msg)


def test_scene_attribute_null_pointers_rejected():
    L = _lib.lib()
    dims = _lib.SceneAttributeDims(*_OK.values())
    for i in (0, 2, 3):     # grads, acc, wsum (weight may be NULL)
        args = [1, None, 1, 1]
        args[i] = None
        assert L.msst_scene_attribute(C.byref(dims), *args, None) == 1
        assert b"must be set" in L.msst_last_error()
    assert L.msst_version() == 102


# ---- Python argument errors ---------------------------------------------------------------------------------------------------------
def test_attribution_refuses_models():
    w, tg = _t(2, 50, 8, 8), _t(2, 8, 8, dtype=torch.int64)
    for fn, args in ((attribute_windows, (w, tg)), (attribute_scene, (_t(1, 50, 9, 9), _t(1, 9, 9, dtype=torch.int64)))):
        with pytest.raises(ValueError, match="SimMIM"):
            fn(_sim(), *args)
        with pytest.raises(ValueError, match="pixelwise"):
            fn(_enc(pixelwise=True), *args)
        with pytest.raises(ValueError, match="ViTSpatialSpectral"):
            fn(torch.nn.Linear(2, 2), *args)


@pytest.mark.parametrize("windows, target, kw, match", [
    (torch.zeros(2, 50, 8, 8), torch.zeros(2, 8, 8, dtype=torch.int64), {}, "fp32 CUDA"),
    (_t(2, 50, 8, 8, dtype=torch.float64), _t(2, 8, 8, dtype=torch.int64), {}, "fp32 CUDA"),
    (_t(2, 40, 8, 8), _t(2, 8, 8, dtype=torch.int64), {}, "fp32 CUDA"),
    (_t(2, 50, 7, 7), _t(2, 8, 8, dtype=torch.int64), {}, "fp32 CUDA"),
    (_t(0, 50, 8, 8), _t(0, 8, 8, dtype=torch.int64), {}, "n >= 1"),
    (_t(2, 50, 8, 8), _t(2, 8, 8), {}, "integer tensor"),
    (_t(2, 50, 8, 8), _t(2, 8, 8, dtype=torch.bool), {}, "integer tensor"),
    (_t(2, 50, 8, 8), _t(3, 8, 8, dtype=torch.int64), {}, "integer tensor"),
    (_t(2, 50, 8, 8), np.zeros((2, 8, 8), dtype=np.int64), {}, "integer tensor"),
    (_t(2, 50, 8, 8), _t(2, 8, 8, dtype=torch.int64), dict(steps=0), "steps=0"),
    (_t(2, 50, 8, 8), _t(2, 8, 8, dtype=torch.int64), dict(steps=2.0), "steps=2.0"),
    (_t(2, 50, 8, 8), _t(2, 8, 8, dtype=torch.int64), dict(steps=True), "steps=True"),
    (_t(2, 50, 8, 8), _t(2, 8, 8, dtype=torch.int64), dict(baseline=np.zeros(49)), r"real \[50\] spectrum"),
    (_t(2, 50, 8, 8), _t(2, 8, 8, dtype=torch.int64), dict(baseline=np.zeros((1, 50))), r"real \[50\] spectrum"),
])
def test_attribute_windows_argument_errors(windows, target, kw, match):
    with pytest.raises(ValueError, match=match):
        attribute_windows(_enc(), windows, target, **kw)


@pytest.mark.parametrize("scene, target, kw, match", [
    (torch.zeros(1, 50, 9, 9), torch.zeros(1, 9, 9, dtype=torch.int64), {}, "CUDA device"),
    (_t(50, 9, 9), _t(1, 9, 9, dtype=torch.int64), {}, r"\[B, bands, H, W\]"),
    (_t(1, 50, 9, 9, dtype=torch.float16), _t(1, 9, 9, dtype=torch.int64), {}, "must be fp32"),
    (_t(1, 40, 9, 9), _t(1, 9, 9, dtype=torch.int64), {}, "40 bands, the model 50"),
    (_t(1, 50, 9, 9), _t(1, 9, 8, dtype=torch.int64), {}, "integer tensor"),
    (_t(1, 50, 9, 9), _t(1, 9, 9), {}, "integer tensor"),
    (_t(1, 50, 9, 9), _t(1, 9, 9, dtype=torch.int64), dict(steps=-1), "steps=-1"),
    (_t(1, 50, 9, 9), _t(1, 9, 9, dtype=torch.int64), dict(stride=9), "stride"),
    (_t(1, 50, 7, 9), _t(1, 7, 9, dtype=torch.int64), {}, "smaller than the window"),
    (_t(1, 50, 9, 9), _t(1, 9, 9, dtype=torch.int64), dict(baseline=[0.0] * 48), "spectrum"),
    (_t(1, 50, 9, 9), _t(1, 9, 9, dtype=torch.int64), dict(weight=np.ones((7, 7))), "weight must be"),
    (_t(1, 50, 9, 9), _t(1, 9, 9, dtype=torch.int64), dict(batch_samples=0), "batch_samples=0"),
])
def test_attribute_scene_argument_errors(scene, target, kw, match):
    with pytest.raises(ValueError, match=match):
        attribute_scene(_enc(), scene, target, **kw)


def test_attribute_scene_raw_tiles_checks():
    raw = _t(1, 48, 10, 10, dtype=torch.int16)
    rt = M.RawTiles(raw, np.zeros(48), np.ones(48), image_size=8, pad_bands=2, crop=(1, 0))
    with pytest.raises(ValueError, match="crop"):
        attribute_scene(_enc(), rt, _t(1, 10, 10, dtype=torch.int64))
    rt = M.RawTiles(raw, np.zeros(48), np.ones(48), image_size=8, pad_bands=1)
    with pytest.raises(ValueError, match="49 bands, the model 50"):
        attribute_scene(_enc(), rt, _t(1, 10, 10, dtype=torch.int64))


def test_attribution_refuses_before_touching_training_state():
    m = _enc().train()
    flags = [p.requires_grad for p in m.parameters()]
    with pytest.raises(ValueError):
        attribute_windows(m, _t(1, 50, 8, 8), _t(1, 8, 8, dtype=torch.int64), steps=0)
    assert m.training and [p.requires_grad for p in m.parameters()] == flags


# ---- schedule, gather, band profiles ------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("steps", [1, 2, 7, 32])
def test_ig_alphas_midpoint_rule(steps):
    a = ig_alphas(steps)
    assert a.dtype == torch.float64 and a.shape == (steps,)
    assert torch.equal(a, torch.tensor([(k + 0.5) / steps for k in range(steps)], dtype=torch.float64))
    assert float(a.mean()) == pytest.approx(0.5)


@pytest.mark.parametrize("shape, stride, first, n", [((2, 3, 13, 11), (3, 2), 0, 24), ((2, 3, 13, 11), (3, 2), 5, 9),
                                                     ((1, 2, 8, 8), (8, 8), 0, 1), ((3, 1, 10, 17), (5, 4), 7, 8)])
def test_interpolated_window_gather_against_numpy_loop(shape, stride, first, n):
    B, nb, H, W = shape
    w, steps = 8, 3
    ny, nx = scene_windows(H, W, w, stride)
    n = min(n, B * ny * nx - first)
    rng = np.random.default_rng(0)
    x = rng.standard_normal(shape).astype(np.float32)
    tg = rng.integers(-1, 5, (B, H, W))
    base = rng.standard_normal(nb).astype(np.float32)
    want, want_t = [], []
    for g in range(first, first + n):
        b, k = divmod(g, ny * nx)
        oy, ox = min((k // nx) * stride[0], H - w), min((k % nx) * stride[1], W - w)
        want.append(x[b, :, oy:oy + w, ox:ox + w])
        want_t.append(tg[b, oy:oy + w, ox:ox + w])
    got = _gather_windows(torch.from_numpy(x), w, stride, (ny, nx), first, n)
    assert torch.equal(got, torch.from_numpy(np.stack(want)))
    assert torch.equal(_gather_windows(torch.from_numpy(tg), w, stride, (ny, nx), first, n), torch.from_numpy(np.stack(want_t)))
    xi = _interpolate(got, torch.from_numpy(base), steps).numpy()
    a = ((np.arange(steps) + 0.5) / steps).astype(np.float32)
    b4 = base[None, :, None, None]
    for i in range(n):
        for k in range(steps):
            np.testing.assert_array_equal(xi[i * steps + k], b4[0] + a[k] * (want[i] - b4[0]))


def test_band_importance_against_brute_force():
    rng = np.random.default_rng(3)
    attr = torch.from_numpy(rng.standard_normal((2, 6, 5, 7)).astype(np.float32))
    labels = torch.from_numpy(rng.integers(-2, 6, (2, 5, 7)))
    labels[labels == 3] = 9                                        # class 3 absent; 9 and -2 out of range
    got = band_importance(attr, labels, num_classes=5)
    assert got.dtype == torch.float64 and got.shape == (5, 6)
    a, lab = attr.double().numpy(), labels.numpy()
    for c in range(5):
        pix = [(b, y, x) for b in range(2) for y in range(5) for x in range(7) if lab[b, y, x] == c]
        if not pix:
            assert torch.isnan(got[c]).all()
            continue
        for band in range(6):
            assert float(got[c, band]) == pytest.approx(np.mean([abs(a[b, band, y, x]) for b, y, x in pix]), rel=1e-12)
    ign = band_importance(attr, torch.where(labels == 0, torch.tensor(7), labels), num_classes=8, ignore_index=7)
    assert torch.isnan(ign[7]).all() and torch.isnan(ign[0]).all()


@pytest.mark.parametrize("attr, labels, kw, match", [
    (torch.zeros(2, 3, 4), torch.zeros(2, 3, 4, dtype=torch.int64), dict(num_classes=2), "attr must be"),
    (torch.zeros(1, 3, 4, 5, dtype=torch.int64), torch.zeros(1, 4, 5, dtype=torch.int64), dict(num_classes=2), "attr must be"),
    (torch.zeros(1, 3, 4, 5), torch.zeros(1, 4, 4, dtype=torch.int64), dict(num_classes=2), "labels must be"),
    (torch.zeros(1, 3, 4, 5), torch.zeros(1, 4, 5), dict(num_classes=2), "labels must be"),
    (torch.zeros(1, 3, 4, 5), torch.zeros(1, 4, 5, dtype=torch.int64), dict(num_classes=0), "num_classes=0"),
])
def test_band_importance_argument_errors(attr, labels, kw, match):
    with pytest.raises(ValueError, match=match):
        band_importance(attr, labels, **kw)
