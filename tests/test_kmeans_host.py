"""CPU: the argument checks of kmeans_fit / KMeans.predict / cluster_scene / clustering_metrics (ValueError before any device work), the
msst_kmeans C entry points (MSST_ERR_ARG before any CUDA call), and clustering_metrics against hand-written float64 formulas and
scipy's assignment solver."""
import ctypes
import itertools
import math

import numpy as np
import pytest
import torch
from scipy.optimize import linear_sum_assignment

import maskedsst_b200 as M
from maskedsst_b200 import _lib
from maskedsst_b200.inference import KMeans, cluster_scene, clustering_metrics, kmeans_fit


class _FakeCuda(torch.Tensor):
    """A CPU tensor that claims to live on a CUDA device, so that the checks after the device check can run without one."""
    @property
    def is_cuda(self):
        return True


def _t(*shape, dtype=torch.float32):
    return torch.zeros(*shape, dtype=dtype).as_subclass(_FakeCuda)


@pytest.mark.parametrize("x, k, kw, match", [
    (_t(100, 80), 5, {}, "feature width 80"),
    (_t(100, 288), 5, {}, "feature width 288"),
    (_t(100, 96, dtype=torch.float64), 5, {}, "x must be a 2-D fp32"),
    (_t(96), 5, {}, "x must be a 2-D fp32"),
    (torch.zeros(100, 96), 5, {}, "CUDA"),
    (_t(4, 96), 5, {}, "4 rows; need num_clusters=5"),
    (_t(100, 96), 0, {}, "num_clusters=0"),
    (_t(300, 96), 257, {}, "num_clusters=257"),
    (_t(100, 96), True, {}, "num_clusters=True"),
    (_t(100, 96), 5.0, {}, "num_clusters=5.0"),
    (_t(300, 96), 171, {}, "exceeds 16384"),
    (_t(300, 256), 65, {}, "exceeds 16384"),
    (_t(100, 96), 5, dict(restarts=0), "restarts=0"),
    (_t(100, 96), 5, dict(restarts=17), "restarts=17"),
    (_t(100, 96), 5, dict(iters=0), "iters=0"),
    (_t(100, 96), 5, dict(iters=2.0), "iters=2.0"),
    (_t(100, 96), 5, dict(seed=-1), "seed=-1"),
    (_t(100, 96), 5, dict(normalize=1), "normalize=1"),
    (_t(100, 96), 5, dict(init=_t(1, 5, 64)), "init must be"),
    (_t(100, 96), 5, dict(restarts=2, init=_t(1, 5, 96)), "init must be"),
    (_t(100, 96), 5, dict(init=_t(1, 5, 96, dtype=torch.float64)), "init must be"),
    (_t(100, 96), 5, dict(init=torch.zeros(1, 5, 96)), "init must be"),
    (_t(100, 96), 5, dict(init=[[0.0] * 96] * 5), "init must be"),
])
def test_fit_argument_errors(x, k, kw, match):
    with pytest.raises(ValueError, match=match):
        kmeans_fit(x, k, **kw)


def _km(R=2, K=5, D=96):
    c = torch.zeros(R, K, D).as_subclass(_FakeCuda)
    return KMeans(c, torch.tensor([2.0, 1.0, 1.0][:R], dtype=torch.float64), torch.ones(R, dtype=torch.int64),
                  torch.ones(R, dtype=torch.bool), True)


def test_kmeans_best_is_the_lowest_inertia_lowest_index_on_ties():
    assert _km(R=2).best == 1
    km = KMeans(torch.zeros(3, 2, 32), torch.tensor([3.0, 1.0, 1.0], dtype=torch.float64), torch.ones(3, dtype=torch.int64),
                torch.ones(3, dtype=torch.bool), False)
    assert km.best == 1 and km.num_clusters == 2


def test_predict_argument_errors():
    km = _km()
    for kw, match in [(dict(restart=2), "restart=2"), (dict(restart=-1), "restart=-1"), (dict(restart=True), "restart=True"),
                      (dict(batch_queries=0), "batch_queries"), (dict(batch_queries=1.5), "batch_queries")]:
        with pytest.raises(ValueError, match=match):
            km.predict(_t(10, 96), **kw)
    for x, match in [(_t(10, 64), "does not match dim 96"), (torch.zeros(10, 96), "CUDA"), (_t(10, 80), "feature width 80")]:
        with pytest.raises(ValueError, match=match):
            km.predict(x)


def _vit(**kw):
    args = dict(image_size=8, spatial_patch_size=1, spectral_patch_size=10, num_classes=20, dim=96, depth=1, heads=8, mlp_dim=64,
                channels=50, spectral_pos_embed=False)
    args.update(kw)
    return M.ViTSpatialSpectral(**args)


def test_scene_argument_errors():
    m = _vit()
    scene = torch.zeros(1, 50, 12, 13)
    with pytest.raises(ValueError, match="CUDA"):
        cluster_scene(m, scene, num_clusters=5)
    with pytest.raises(ValueError, match="scene"):
        cluster_scene(m, torch.zeros(50, 12, 13).as_subclass(_FakeCuda), num_clusters=5)
    fake = scene.as_subclass(_FakeCuda)
    v1 = M.ViTSpatialSpectral_V1(image_size=8, spatial_patch_size=1, spectral_patch_size=10, num_classes=20, dim=96, depth=1, heads=8,
                                 mlp_dim=64, channels=50)
    for model, kw, match in [(v1, {}, "ViTSpatialSpectral encoder"), (m, dict(num_clusters=0), "num_clusters=0"),
                             (m, dict(num_clusters=171), "exceeds 16384"), (m, dict(num_clusters=157), "156 rows"),
                             (m, dict(restarts=17), "restarts=17"), (m, dict(iters=0), "iters=0"), (m, dict(seed=-2), "seed=-2"),
                             (m, dict(normalize=None), "normalize=None"), (m, dict(batch_queries=0), "batch_queries"),
                             (M.SimMIMSpatialSpectral(encoder=_vit(dim=256), masking_ratio=0.5), dict(num_clusters=65), "exceeds"),
                             (_vit(dim=48, heads=4), {}, "feature width 48")]:
        args = dict(num_clusters=5)
        args.update(kw)
        with pytest.raises(ValueError, match=match):
            cluster_scene(model, fake, **args)


def _dims(**kw):
    d = dict(n=10000, dim=96, k=20, restarts=3, normalize=1)
    d.update(kw)
    return _lib.KmeansDims(d["n"], d["dim"], d["k"], d["restarts"], d["normalize"])


def test_c_entry_points_refuse_bad_arguments_without_a_device():
    L = _lib.lib()
    S = 3                                                            # ceil(10000 / 4096)
    assert L.msst_kmeans_workspace(ctypes.byref(_dims())) == 3 * S * (8 + 4 * 20 * 96 + 4 * 20 + 4)
    assert L.msst_kmeans_workspace(ctypes.byref(_dims(n=4096, dim=256, k=64, restarts=16))) == 16 * (8 + 4 * 64 * 256 + 4 * 64 + 4)
    bad = [(dict(dim=0), b"dim=0"), (dict(dim=48), b"dim=48"), (dict(dim=288), b"dim=288"), (dict(k=0), b"k=0"), (dict(k=257), b"k=257"),
           (dict(k=171), b"k*dim=16416"), (dict(dim=256, k=65), b"k*dim=16640"), (dict(restarts=0), b"restarts=0"),
           (dict(restarts=17), b"restarts=17"), (dict(normalize=2), b"normalize=2"), (dict(n=2 ** 31), b"n=2147483648"),
           (dict(n=0), b"n=0")]
    for kw, what in bad:
        d = _dims(**kw)
        for name, call in [("kmeans_seed", lambda: L.msst_kmeans_seed(ctypes.byref(d), 0, 1, 1, 1, 1, 1, 1, None)),
                           ("kmeans_assign", lambda: L.msst_kmeans_assign(ctypes.byref(d), 1, 1, 1, 1, 1, None)),
                           ("kmeans_assign", lambda: L.msst_kmeans_assign(ctypes.byref(d), 1, 1, 1, None, None, None)),
                           ("kmeans_update", lambda: L.msst_kmeans_update(ctypes.byref(d), 1, 1, 1, 1, 1, None))]:
            assert call() == 1, (kw, name)
            msg = L.msst_last_error()
            assert msg.startswith(name.encode() + b":") and what in msg, (kw, msg)
        assert L.msst_kmeans_workspace(ctypes.byref(d)) == -1
        assert L.msst_last_error().startswith(b"kmeans_workspace:")
    d = _dims(n=19)                                                  # K <= n when fitting; prediction needs one row
    assert L.msst_kmeans_seed(ctypes.byref(d), 0, 1, 1, 1, 1, 1, 1, None) == 1 and b"n=19" in L.msst_last_error()
    assert L.msst_kmeans_assign(ctypes.byref(d), 1, 1, 1, 1, 1, None) == 1 and b"n=19" in L.msst_last_error()
    assert L.msst_kmeans_update(ctypes.byref(d), 1, 1, 1, 1, 1, None) == 1 and b"n=19" in L.msst_last_error()
    assert L.msst_kmeans_workspace(ctypes.byref(d)) == -1
    d = _dims()
    for rnd in (-1, 20):
        assert L.msst_kmeans_seed(ctypes.byref(d), rnd, 1, 1, 1, 1, 1, 1, None) == 1 and f"round={rnd}".encode() in L.msst_last_error()
    for i in range(6):
        ptrs = [1] * 6
        ptrs[i] = None
        assert L.msst_kmeans_seed(ctypes.byref(d), 0, *ptrs, None) == 1 and b"must be set" in L.msst_last_error()
    for i in range(3):
        ptrs = [1] * 3
        ptrs[i] = None
        assert L.msst_kmeans_assign(ctypes.byref(d), *ptrs, 1, 1, None) == 1 and b"must be set" in L.msst_last_error()
    for i in range(5):
        ptrs = [1] * 5
        ptrs[i] = None
        assert L.msst_kmeans_update(ctypes.byref(d), *ptrs, None) == 1 and b"must be set" in L.msst_last_error()
    for fn, args in [(L.msst_kmeans_seed, (0, 1, 1, 1, 1, 1, 1, None)), (L.msst_kmeans_assign, (1, 1, 1, 1, 1, None)),
                     (L.msst_kmeans_update, (1, 1, 1, 1, 1, None))]:
        assert fn(None, *args) == 1 and b"dims" in L.msst_last_error()
    assert L.msst_kmeans_workspace(None) == -1


# ---------------------------------------------------------------------------------------------------------------- clustering_metrics

def _metrics64(cont):
    """NMI / ARI / best matching / majority from a contingency [nc, K], by the textbook formulas, written out term by term."""
    nc, K = cont.shape
    N = sum(int(v) for v in cont.flat)
    a = [sum(int(cont[i, j]) for j in range(K)) for i in range(nc)]
    b = [sum(int(cont[i, j]) for i in range(nc)) for j in range(K)]
    mi = 0.0
    for i in range(nc):
        for j in range(K):
            if cont[i, j]:
                mi += cont[i, j] / N * math.log(N * cont[i, j] / (a[i] * b[j]))
    hu = -sum(v / N * math.log(v / N) for v in a if v)
    hv = -sum(v / N * math.log(v / N) for v in b if v)
    one = sum(1 for v in a if v) == 1 and sum(1 for v in b if v) == 1
    nmi = 1.0 if one else mi / ((hu + hv) / 2)
    c2 = lambda v: v * (v - 1) // 2
    idx = sum(c2(int(v)) for v in cont.flat)
    sa, sb = sum(c2(v) for v in a), sum(c2(v) for v in b)
    exp = sa * sb / c2(N) if c2(N) else 0.0
    mx = (sa + sb) / 2
    ari = 1.0 if mx == exp else (idx - exp) / (mx - exp)
    maj = [max(range(nc), key=lambda i: (cont[i, j], -i)) for j in range(K)]
    return nmi, ari, maj, sum(int(cont[maj[j], j]) for j in range(K)) / N


def _from_contingency(cont, rng):
    """(clusters, labels) pixel lists whose contingency is cont, shuffled, with some ignored / out-of-range pixels mixed in."""
    nc, K = cont.shape
    lab = np.concatenate([np.full(int(cont[i, j]), i) for i in range(nc) for j in range(K)] + [np.array([-1, nc, -1], np.int64)])
    cl = np.concatenate([np.full(int(cont[i, j]), j) for i in range(nc) for j in range(K)] + [np.array([K + 3, -7, 0], np.int64)])
    p = rng.permutation(lab.size)
    return torch.from_numpy(cl[p].astype(np.int64)), torch.from_numpy(lab[p].astype(np.int64))


@pytest.mark.parametrize("nc, K", [(5, 3), (6, 6), (3, 7), (20, 20), (12, 30), (40, 9), (1, 4), (4, 1)])
def test_metrics_against_formulas_and_scipy(nc, K):
    rng = np.random.default_rng(nc * 100 + K)
    for trial in range(4):
        if trial == 0:
            cont = rng.integers(0, 30, (nc, K))
        elif trial == 1:
            cont = rng.integers(0, 3, (nc, K)) * 5                  # many exact ties
        elif trial == 2:
            cont = np.zeros((nc, K), np.int64)
            cont[rng.integers(0, nc, 40), rng.integers(0, K, 40)] += rng.integers(1, 50, 40)   # sparse, empty rows / columns
        else:
            cont = np.full((nc, K), 7)                              # every entry tied
        if cont.sum() == 0:
            cont[0, 0] = 1
        cl, lab = _from_contingency(cont, rng)
        m = clustering_metrics(cl, lab, num_clusters=K, num_classes=nc)
        assert torch.equal(m["contingency"], torch.from_numpy(cont.astype(np.int64)))
        nmi, ari, maj, oa_maj = _metrics64(cont)
        assert abs(m["nmi"] - nmi) <= 1e-12 and abs(m["ari"] - ari) <= 1e-12, (trial, m["nmi"], nmi, m["ari"], ari)
        assert m["majority_map"].tolist() == maj and abs(m["oa_majority"] - oa_maj) <= 1e-15
        rows, cols = linear_sum_assignment(cont, maximize=True)
        best = int(cont[rows, cols].sum())
        hmap = m["hungarian_map"].numpy()
        matched = [k for k in range(K) if hmap[k] >= 0]
        assert len(matched) == min(nc, K) and len(set(hmap[matched].tolist())) == len(matched)   # one to one
        assert int(sum(cont[hmap[k], k] for k in matched)) == best, trial
        assert m["oa_hungarian"] == best / cont.sum()


def test_hungarian_brute_force_small():
    rng = np.random.default_rng(3)
    for nc, K in [(3, 3), (2, 4), (4, 2), (4, 4)]:
        for _ in range(20):
            cont = rng.integers(0, 6, (nc, K))
            cont[0, 0] += 1
            if K <= nc:   # every cluster to a distinct class
                want = max(sum(cont[cs[k], k] for k in range(K)) for cs in itertools.permutations(range(nc), K))
            else:         # every class to a distinct cluster
                want = max(sum(cont[c, ks[c]] for c in range(nc)) for ks in itertools.permutations(range(K), nc))
            cl, lab = _from_contingency(cont, rng)
            m = clustering_metrics(cl, lab, num_clusters=K, num_classes=nc)
            assert round(m["oa_hungarian"] * cont.sum()) == want


def test_degenerate_nmi_and_ari():
    one = torch.zeros(50, dtype=torch.int64)
    m = clustering_metrics(one, one, num_clusters=3, num_classes=4)          # both sides one occupied label
    assert m["nmi"] == 1.0 and m["ari"] == 1.0 and m["oa_hungarian"] == 1.0 and m["oa_majority"] == 1.0
    assert m["hungarian_map"][0] == 0 and m["majority_map"].tolist() == [0, 0, 0]
    lab = torch.arange(6) % 3
    m = clustering_metrics(torch.zeros(6, dtype=torch.int64), lab, num_clusters=2, num_classes=3)   # one cluster, three classes
    assert m["nmi"] == 0.0 and m["ari"] == 0.0 and abs(m["oa_hungarian"] - 1 / 3) < 1e-15
    m = clustering_metrics(torch.arange(5), torch.arange(5), num_clusters=5, num_classes=5)          # all singletons, both sides
    assert m["ari"] == 1.0 and abs(m["nmi"] - 1.0) < 1e-12 and m["oa_hungarian"] == 1.0
    m = clustering_metrics(torch.tensor([1]), torch.tensor([2]), num_clusters=2, num_classes=3)     # one pixel
    assert m["nmi"] == 1.0 and m["ari"] == 1.0
    perm = clustering_metrics(torch.tensor([2, 2, 0, 0, 1, 1]), torch.tensor([0, 0, 1, 1, 2, 2]), num_clusters=3, num_classes=3)
    assert abs(perm["nmi"] - 1.0) < 1e-12 and abs(perm["ari"] - 1.0) < 1e-12 and perm["oa_hungarian"] == 1.0
    assert perm["hungarian_map"].tolist() == [1, 2, 0] == perm["majority_map"].tolist()


def test_metrics_maps_feed_confusion_matrix():
    rng = np.random.default_rng(5)
    lab = torch.from_numpy(rng.integers(-1, 4, (2, 9, 7)))
    cl = torch.from_numpy(rng.integers(0, 4, (2, 9, 7)))
    m = clustering_metrics(cl, lab, num_clusters=4, num_classes=4)
    conf = M.inference.confusion_matrix(m["hungarian_map"][cl], lab, 4)
    assert abs(M.inference.classification_metrics(conf)["oa"] - m["oa_hungarian"]) < 1e-15
    conf = M.inference.confusion_matrix(m["majority_map"][cl], lab, 4)
    assert abs(M.inference.classification_metrics(conf)["oa"] - m["oa_majority"]) < 1e-15


def test_metrics_argument_errors():
    z = torch.zeros(10, dtype=torch.int64)
    for kw, match in [(dict(num_clusters=0, num_classes=3), "num_clusters=0"), (dict(num_clusters=3, num_classes=257), "num_classes=257"),
                      (dict(num_clusters=True, num_classes=3), "num_clusters=True")]:
        with pytest.raises(ValueError, match=match):
            clustering_metrics(z, z, **kw)
    with pytest.raises(ValueError, match="clusters must be an integer"):
        clustering_metrics(torch.zeros(10), z, num_clusters=3, num_classes=3)
    with pytest.raises(ValueError, match="labels must be an integer"):
        clustering_metrics(z, torch.zeros(10, dtype=torch.bool), num_clusters=3, num_classes=3)
    with pytest.raises(ValueError, match="9 clusters for 10 labels"):
        clustering_metrics(z[:9], z, num_clusters=3, num_classes=3)
    with pytest.raises(ValueError, match="no labelled pixel"):
        clustering_metrics(z, torch.full((10,), -1), num_clusters=3, num_classes=3)
    with pytest.raises(ValueError, match=r"clusters outside \[0, 3\)"):
        clustering_metrics(torch.full((10,), 3), z, num_clusters=3, num_classes=3)
