"""CPU: the argument checks of linear_probe_fit / LinearProbe / linear_probe_scene (ValueError before any device work) and of the
msst_linprobe C entry points (MSST_ERR_ARG before any CUDA call)."""
import ctypes

import pytest
import torch

import maskedsst_b200 as M
from maskedsst_b200 import _lib
from maskedsst_b200.inference import LinearProbe, linear_probe_fit, linear_probe_scene


class _FakeCuda(torch.Tensor):
    """A CPU tensor that claims to live on a CUDA device, so that the checks after the device check can run without one."""
    @property
    def is_cuda(self):
        return True


def _t(*shape, dtype=torch.float32):
    return torch.zeros(*shape, dtype=dtype).as_subclass(_FakeCuda)


def _lab(n, v=0):
    return torch.full((n,), v, dtype=torch.int64).as_subclass(_FakeCuda)


@pytest.mark.parametrize("kw, match", [
    (dict(num_classes=0), "num_classes=0"),
    (dict(num_classes=257), "num_classes=257"),
    (dict(num_classes=True), "num_classes=True"),
    (dict(num_classes=5, heads=()), "0 heads"),
    (dict(num_classes=5, heads=[(1e-3, 0.0)] * 17, val=(_t(10, 96), _lab(10))), "17 heads"),
    (dict(num_classes=5, heads=[(1e-3,)]), "pairs"),
    (dict(num_classes=5, heads=[(-1e-3, 0.0)]), "finite and >= 0"),
    (dict(num_classes=5, heads=[(1e-3, float("nan"))]), "finite and >= 0"),
    (dict(num_classes=5, heads=[(float("inf"), 0.0)]), "finite and >= 0"),
    (dict(num_classes=5, epochs=0), "epochs=0"),
    (dict(num_classes=5, epochs=2.0), "epochs=2.0"),
    (dict(num_classes=5, batch_size=0), "batch_size=0"),
    (dict(num_classes=5, seed=-1), "seed=-1"),
    (dict(num_classes=5, heads=[(1e-3, 0.0), (1e-2, 0.0)]), "need val"),
    (dict(num_classes=5, val=_t(10, 96)), "val must be a pair"),
    (dict(num_classes=5, val=(_t(10, 64), _lab(10))), "val rows"),
    (dict(num_classes=5, val=(_t(10, 96), _lab(9))), "labels of val"),
    (dict(num_classes=5, val=(_t(10, 96), _lab(10, 5))), r"labels of val outside \[0, 5\)"),
    (dict(num_classes=5, val=(torch.zeros(10, 96), _lab(10))), "CUDA"),
])
def test_fit_argument_errors(kw, match):
    with pytest.raises(ValueError, match=match):
        linear_probe_fit(_t(100, 96), _lab(100), **kw)


@pytest.mark.parametrize("ref, labels, match", [
    (_t(100, 80), _lab(100), "feature width 80"),
    (_t(100, 288), _lab(100), "feature width 288"),
    (_t(100, 96, dtype=torch.float64), _lab(100), "ref must be a 2-D fp32"),
    (_t(96), _lab(100), "ref must be a 2-D fp32"),
    (torch.zeros(100, 96), _lab(100), "CUDA"),
    (_t(0, 96), _lab(0), "0 rows"),
    (_t(100, 96), _lab(99), "labels of ref"),
    (_t(100, 96), torch.zeros(100).as_subclass(_FakeCuda), "labels of ref"),
    (_t(100, 96), torch.zeros(100, dtype=torch.bool).as_subclass(_FakeCuda), "labels of ref"),
    (_t(100, 96), _lab(100, -1), r"outside \[0, 5\)"),
    (_t(100, 96), _lab(100, 5), r"outside \[0, 5\)"),
])
def test_fit_data_errors(ref, labels, match):
    with pytest.raises(ValueError, match=match):
        linear_probe_fit(ref, labels, num_classes=5)


def _probe(nc=20, D=96, H=2, device_fake=True):
    p = torch.zeros(H, nc * D + nc)
    return LinearProbe(p.as_subclass(_FakeCuda) if device_fake else p, nc, D, [(1e-3, 0.0)] * H)


def test_predict_argument_errors():
    probe = _probe()
    for kw, match in [(dict(head=2), "head=2"), (dict(head=-1), "head=-1"), (dict(head=True), "head=True"), (dict(batch_queries=0), "batch_queries"),
                      (dict(batch_queries=1.5), "batch_queries")]:
        with pytest.raises(ValueError, match=match):
            probe.predict(_t(10, 96), **kw)
    for x, match in [(_t(10, 64), "does not match dim 96"), (torch.zeros(10, 96), "CUDA"), (_t(10, 80), "feature width 80")]:
        with pytest.raises(ValueError, match=match):
            probe.predict(x)


def _vit(**kw):
    args = dict(image_size=8, spatial_patch_size=1, spectral_patch_size=10, num_classes=20, dim=96, depth=1, heads=8, mlp_dim=64,
                channels=50, spectral_pos_embed=False)
    args.update(kw)
    return M.ViTSpatialSpectral(**args)


def test_load_into_refuses_other_heads_and_shapes():
    probe = _probe(device_fake=False)
    for model, match in [(_vit(pixelwise=True), "pixelwise or spectral-MLP"), (_vit(spectral_mlp_head=True), "pixelwise or spectral-MLP"),
                         (M.ViTSpatialSpectral_V1(image_size=8, spatial_patch_size=1, spectral_patch_size=10, num_classes=20, dim=96,
                                                  depth=1, heads=8, mlp_dim=64, channels=50), "ViTSpatialSpectral_V1"),
                         (M.SimMIMSpatialSpectral(encoder=_vit(), masking_ratio=0.5), "SimMIMSpatialSpectral"),
                         (_vit(dim=64), "dim 64"), (_vit(num_classes=8), "num_classes 8")]:
        with pytest.raises(ValueError, match=match):
            probe.load_into(model)
    with pytest.raises(ValueError, match="head=5"):
        probe.load_into(_vit(), head=5)


def test_load_into_writes_the_default_head_in_place():
    """p1 = 2: the Linear's row (pi*p1 + pj)*nc + c is W[c] for every sub-pixel; LayerNorm weight 1, bias 0."""
    nc, D = 20, 96
    params = torch.randn(2, nc * D + nc)
    probe = LinearProbe(params, nc, D, [(1e-3, 0.0)] * 2, best=1)
    m = _vit(spatial_patch_size=2)
    ln, lin = m.mlp_head[0], m.mlp_head[1]
    w_before = lin.weight
    torch.nn.init.normal_(ln.weight)
    probe.load_into(m)
    assert lin.weight is w_before and lin.weight.shape == (4 * nc, D)
    W, b = params[1, :nc * D].reshape(nc, D), params[1, nc * D:]
    for k in range(4):
        assert torch.equal(lin.weight[k * nc:(k + 1) * nc], W) and torch.equal(lin.bias[k * nc:(k + 1) * nc], b)
    assert torch.equal(ln.weight, torch.ones(D)) and torch.equal(ln.bias, torch.zeros(D))


def test_scene_argument_errors():
    m = _vit()
    scene = torch.zeros(1, 50, 12, 13)
    labels = torch.zeros(1, 12, 13, dtype=torch.int64)
    with pytest.raises(ValueError, match="CUDA"):
        linear_probe_scene(m, scene, labels, num_classes=20)
    for bad in (torch.zeros(1, 12, 12, dtype=torch.int64), torch.zeros(1, 12, 13), torch.zeros(12, 13, dtype=torch.int64)):
        with pytest.raises(ValueError, match="train_labels"):
            linear_probe_scene(m, scene, bad, num_classes=20)
    with pytest.raises(ValueError, match="scene"):
        linear_probe_scene(m, torch.zeros(50, 12, 13), labels, num_classes=20)
    fake, flab = scene.as_subclass(_FakeCuda), labels.as_subclass(_FakeCuda)
    for nc in (0, 257):
        with pytest.raises(ValueError, match=f"num_classes={nc}"):
            linear_probe_scene(m, fake, flab, num_classes=nc)
    with pytest.raises(ValueError, match="val_labels"):
        linear_probe_scene(m, fake, flab, num_classes=20, val_labels=torch.zeros(1, 12, 12, dtype=torch.int64).as_subclass(_FakeCuda))
    with pytest.raises(ValueError, match="need val_labels"):
        linear_probe_scene(m, fake, flab, num_classes=20, heads=[(1e-3, 0.0), (1e-2, 0.0)])
    with pytest.raises(ValueError, match="finite and >= 0"):
        linear_probe_scene(m, fake, flab, num_classes=20, heads=[(-1.0, 0.0)])
    with pytest.raises(ValueError, match="labelled pixel"):
        linear_probe_scene(m, fake, torch.full((1, 12, 13), -1, dtype=torch.int64).as_subclass(_FakeCuda), num_classes=20)


def _dims(**kw):
    d = dict(n=1000, dim=96, nc=20, heads=2, batch=300, step=1)
    d.update({k: v for k, v in kw.items() if k in d})
    out = _lib.LinprobeDims(d["n"], d["dim"], d["nc"], d["heads"], d["batch"], d["step"])
    for h in range(16):
        out.lr[h], out.wd[h] = kw.get("lr", 1e-3), kw.get("wd", 0.0)
    return out


def test_c_entry_points_refuse_bad_arguments_without_a_device():
    L = _lib.lib()
    d = _dims()
    assert L.msst_linprobe_workspace(ctypes.byref(d)) == 3 * 2 * (20 * 96 + 20 + 1) * 4
    d = _dims(dim=256, nc=256, heads=16, batch=4096)
    assert L.msst_linprobe_workspace(ctypes.byref(d)) == 32 * 16 * (256 * 257 + 1) * 4
    for kw, what in [(dict(dim=0), b"dim=0"), (dict(dim=48), b"dim=48"), (dict(dim=288), b"dim=288"), (dict(nc=0), b"nc=0"),
                     (dict(nc=257), b"nc=257"), (dict(heads=0), b"heads=0"), (dict(heads=17), b"heads=17"), (dict(n=0), b"n=0"),
                     (dict(n=2 ** 31), b"n=2147483648"), (dict(batch=0), b"batch=0")]:
        d = _dims(**kw)
        assert L.msst_linprobe_grad(ctypes.byref(d), 1, 1, 1, 1, 1, None) == 1, kw
        msg = L.msst_last_error()
        assert msg.startswith(b"linprobe_grad:") and what in msg, (kw, msg)
        assert L.msst_linprobe_update(ctypes.byref(d), 1, 1, 1, 1, 1, None) == 1, kw
        msg = L.msst_last_error()
        assert msg.startswith(b"linprobe_update:") and what in msg, (kw, msg)
        assert L.msst_linprobe_workspace(ctypes.byref(d)) == -1
        assert L.msst_last_error().startswith(b"linprobe_workspace:")
    for kw, what in [(dict(step=0), b"step=0"), (dict(lr=-1.0), b"lr[0]"), (dict(lr=float("nan")), b"lr[0]"),
                     (dict(wd=float("inf")), b"wd[0]"), (dict(wd=-0.5), b"wd[0]")]:
        assert L.msst_linprobe_update(ctypes.byref(_dims(**kw)), 1, 1, 1, 1, 1, None) == 1, kw
        assert what in L.msst_last_error(), (kw, L.msst_last_error())
    d = _dims()
    for i in range(5):
        ptrs = [1] * 5
        ptrs[i] = None
        assert L.msst_linprobe_grad(ctypes.byref(d), *ptrs, None) == 1 and b"must be set" in L.msst_last_error()
        assert L.msst_linprobe_update(ctypes.byref(d), *ptrs, None) == 1 and b"must be set" in L.msst_last_error()
    assert L.msst_linprobe_grad(None, 1, 1, 1, 1, 1, None) == 1 and b"dims" in L.msst_last_error()
    assert L.msst_linprobe_update(None, 1, 1, 1, 1, 1, None) == 1 and b"dims" in L.msst_last_error()
    assert L.msst_linprobe_workspace(None) == -1
    for args, what in [((10, 80, 20), b"dim=80"), ((10, 96, 0), b"nc=0"), ((10, 96, 257), b"nc=257"), ((0, 96, 20), b"n_query=0"),
                       ((2 ** 31, 96, 20), b"n_query=2147483648")]:
        assert L.msst_linprobe_predict(*args, 1, 1, 1, 1, None) == 1, args
        msg = L.msst_last_error()
        assert msg.startswith(b"linprobe_predict:") and what in msg, (args, msg)
    for i in range(4):
        ptrs = [1] * 4
        ptrs[i] = None
        assert L.msst_linprobe_predict(10, 96, 20, *ptrs, None) == 1 and b"must be set" in L.msst_last_error()
