"""CPU: the argument checks of knn_neighbors / knn_classify / knn_scene (ValueError before any device work) and of the C entry points
(MSST_ERR_ARG before any CUDA call)."""
import ctypes

import pytest
import torch

import maskedsst_b200 as M
from maskedsst_b200 import _lib
from maskedsst_b200.inference import knn_classify, knn_neighbors, knn_scene


class _FakeCuda(torch.Tensor):
    """A CPU tensor that claims to live on a CUDA device, so that the checks after the device check can run without one."""
    @property
    def is_cuda(self):
        return True


def _t(*shape, dtype=torch.float32):
    return torch.zeros(*shape, dtype=dtype).as_subclass(_FakeCuda)


@pytest.mark.parametrize("ref, query, k, match", [
    (_t(100, 96), _t(10, 96), 0, "k=0"),
    (_t(100, 96), _t(10, 96), 65, "k=65"),
    (_t(100, 96), _t(10, 96), 2.0, "k=2.0"),
    (_t(100, 96), _t(10, 96), True, "k=True"),
    (_t(19, 96), _t(10, 96), 20, "19 reference rows"),
    (_t(100, 80), _t(10, 80), 5, "feature width 80"),
    (_t(100, 288), _t(10, 288), 5, "feature width 288"),
    (_t(100, 96), _t(10, 64), 5, "disagree"),
    (_t(100, 96, dtype=torch.float64), _t(10, 96), 5, "ref must be a 2-D fp32"),
    (_t(100, 96), _t(10, 96, dtype=torch.bfloat16), 5, "query must be a 2-D fp32"),
    (_t(100, 96, 1), _t(10, 96), 5, "ref must be a 2-D fp32"),
    (_t(96), _t(10, 96), 5, "ref must be a 2-D fp32"),
    (torch.zeros(100, 96), _t(10, 96), 5, "CUDA"),
    (_t(100, 96), torch.zeros(10, 96), 5, "CUDA"),
])
def test_knn_neighbors_argument_errors(ref, query, k, match):
    with pytest.raises(ValueError, match=match):
        knn_neighbors(ref, query, k)


def test_knn_neighbors_batch_queries_must_be_positive():
    for bq in (0, -1, 1.5):
        with pytest.raises(ValueError, match="batch_queries"):
            knn_neighbors(_t(100, 96), _t(10, 96), 5, batch_queries=bq)


def test_knn_classify_argument_errors():
    ref, query = _t(100, 96), _t(10, 96)
    lab = torch.zeros(100, dtype=torch.int64).as_subclass(_FakeCuda)
    for kw, match in [(dict(num_classes=0), "num_classes=0"), (dict(num_classes=257), "num_classes=257"),
                      (dict(num_classes=5, temperature=0.0), "temperature"), (dict(num_classes=5, temperature=-1.0), "temperature"),
                      (dict(num_classes=5, temperature=float("nan")), "temperature"), (dict(num_classes=5, k=0), "k=0"),
                      (dict(num_classes=5, k=65), "k=65")]:
        with pytest.raises(ValueError, match=match):
            knn_classify(ref, lab, query, **kw)
    for bad in (torch.zeros(99, dtype=torch.int64).as_subclass(_FakeCuda), torch.zeros(100).as_subclass(_FakeCuda),
                torch.zeros(100, dtype=torch.bool).as_subclass(_FakeCuda), torch.zeros(100, 1, dtype=torch.int64).as_subclass(_FakeCuda)):
        with pytest.raises(ValueError, match="ref_labels"):
            knn_classify(ref, bad, query, num_classes=5)
    for v in (-1, 5):
        bad = torch.zeros(100, dtype=torch.int64)
        bad[17] = v
        with pytest.raises(ValueError, match=r"outside \[0, 5\)"):
            knn_classify(ref, bad.as_subclass(_FakeCuda), query, num_classes=5)
    with pytest.raises(ValueError, match="CUDA"):
        knn_classify(torch.zeros(100, 96), torch.zeros(100, dtype=torch.int64), torch.zeros(10, 96), num_classes=5)


def test_knn_scene_argument_errors():
    m = M.ViTSpatialSpectral(image_size=8, spatial_patch_size=1, spectral_patch_size=10, num_classes=20, dim=96, depth=1,
                             heads=8, mlp_dim=64, channels=50, spectral_pos_embed=False)
    scene = torch.zeros(1, 50, 12, 13)
    labels = torch.zeros(1, 12, 13, dtype=torch.int64)
    with pytest.raises(ValueError, match="CUDA"):
        knn_scene(m, scene, labels, num_classes=20)
    for bad in (torch.zeros(1, 12, 12, dtype=torch.int64), torch.zeros(1, 12, 13), torch.zeros(12, 13, dtype=torch.int64)):
        with pytest.raises(ValueError, match="train_labels"):
            knn_scene(m, scene, bad, num_classes=20)
    with pytest.raises(ValueError, match="scene"):
        knn_scene(m, torch.zeros(50, 12, 13), labels, num_classes=20)
    fake = scene.as_subclass(_FakeCuda)
    for nc in (0, 257):
        with pytest.raises(ValueError, match=f"num_classes={nc}"):
            knn_scene(m, fake, labels.as_subclass(_FakeCuda), num_classes=nc)


def test_c_entry_points_refuse_bad_arguments_without_a_device():
    L = _lib.lib()

    def topk(N=1000, Q=10, D=96, k=20, ptr=1):
        d = _lib.KnnDims(N, Q, D, k)
        return L.msst_knn_topk(ctypes.byref(d), ptr, 1, 1, 1, None)

    for kw, what in [(dict(k=0), b"k=0"), (dict(k=65), b"k=65"), (dict(N=19), b"n_ref=19"), (dict(N=2 ** 31), b"n_ref=2147483648"),
                     (dict(D=0), b"dim=0"), (dict(D=48), b"dim=48"), (dict(D=288), b"dim=288"), (dict(Q=0), b"n_query=0"),
                     (dict(ptr=None), b"must be set")]:
        assert topk(**kw) == 1, kw
        msg = L.msst_last_error()
        assert msg.startswith(b"knn_topk:") and what in msg, (kw, msg)
    assert L.msst_knn_topk(None, 1, 1, 1, 1, None) == 1 and b"dims" in L.msst_last_error()
    assert L.msst_knn_prepare(1, 10, 100, 1, None) == 1 and b"dim=100" in L.msst_last_error()
    assert L.msst_knn_prepare(1, 0, 96, 1, None) == 1 and b"n=0" in L.msst_last_error()
    assert L.msst_knn_prepare(1, 10, 96, None, None) == 1 and b"must be set" in L.msst_last_error()

    def vote(Q=10, k=20, N=1000, nc=5, T=0.07, ptr=1):
        return L.msst_knn_vote(Q, k, N, 1, 1, ptr, nc, T, 1, 1, None)

    for kw, what in [(dict(nc=0), b"nc=0"), (dict(nc=257), b"nc=257"), (dict(k=0), b"k=0"), (dict(k=65), b"k=65"), (dict(N=5), b"n_ref=5"),
                     (dict(Q=0), b"n_query=0"), (dict(T=0.0), b"temperature"), (dict(T=float("nan")), b"temperature"),
                     (dict(T=-float("inf")), b"temperature"), (dict(ptr=None), b"must be set")]:
        assert vote(**kw) == 1, kw
        msg = L.msst_last_error()
        assert msg.startswith(b"knn_vote:") and what in msg, (kw, msg)
