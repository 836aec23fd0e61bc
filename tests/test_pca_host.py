"""CPU: the argument checks of pca_fit / PCA / pca_scene / rx_scene / false_colour / anomaly_metrics (ValueError before any device work),
the msst_moments C entry points (MSST_ERR_ARG before any CUDA call), anomaly_metrics against brute-force pair counting and scipy's
Mann-Whitney U, false_colour against numpy quantiles, and the component sign rule."""
import numpy as np
import pytest
import torch
from scipy.stats import mannwhitneyu

import maskedsst_b200 as M
from maskedsst_b200 import _lib
from maskedsst_b200.inference import PCA, _sign_rule, anomaly_metrics, false_colour, pca_fit, pca_scene, rx_scene


class _FakeCuda(torch.Tensor):
    """A CPU tensor that claims to live on a CUDA device, so that the checks after the device check can run without one."""
    @property
    def is_cuda(self):
        return True


def _t(*shape, dtype=torch.float32):
    return torch.zeros(*shape, dtype=dtype).as_subclass(_FakeCuda)


@pytest.mark.parametrize("x, match", [
    (_t(100, 0), "feature width 0"),
    (_t(100, 257), "feature width 257"),
    (_t(100, 8, dtype=torch.float64), "x must be a 2-D fp32"),
    (_t(8), "x must be a 2-D fp32"),
    (torch.zeros(100, 8), "CUDA"),
    ([[1.0, 2.0]], "x must be a 2-D fp32"),
    (_t(1, 8), "1 rows; need at least 2"),
    (_t(0, 8), "0 rows; need at least 2"),
])
def test_fit_argument_errors(x, match):
    with pytest.raises(ValueError, match=match):
        pca_fit(x)


def _pca(dim=8, lam=None):
    lam = torch.arange(dim, 0, -1, dtype=torch.float64) if lam is None else lam
    return PCA(100, torch.zeros(dim, dtype=torch.float64), torch.diag(lam), lam, torch.eye(dim, dtype=torch.float64))


@pytest.mark.parametrize("kw, match", [
    (dict(n_components=0), "n_components=0"),
    (dict(n_components=9), "n_components=9"),
    (dict(n_components=2.0), "n_components=2.0"),
    (dict(n_components=True), "n_components=True"),
    (dict(whiten=1), "whiten=1"),
    (dict(ridge=-1.0), "ridge=-1.0"),
    (dict(ridge=float("nan")), "ridge=nan"),
    (dict(ridge=float("inf")), "ridge=inf"),
    (dict(batch_queries=0), "batch_queries=0"),
    (dict(batch_queries=True), "batch_queries=True"),
])
def test_transform_argument_errors(kw, match):
    with pytest.raises(ValueError, match=match):
        _pca().transform(_t(10, 8), **kw)


def test_projection_argument_errors():
    p = _pca()
    with pytest.raises(ValueError, match="x has 7 features, the fit 8"):
        p.transform(_t(10, 7))
    with pytest.raises(ValueError, match="CUDA"):
        p.mahalanobis(torch.zeros(10, 8))
    with pytest.raises(ValueError, match="ridge=-0.5"):
        p.mahalanobis(_t(10, 8), ridge=-0.5)
    with pytest.raises(ValueError, match="batch_queries=-1"):
        p.mahalanobis(_t(10, 8), batch_queries=-1)
    with pytest.raises(ValueError, match="x on cpu, the fit on"):   # the fit lives on the CPU here: any other device is refused
        PCA(100, torch.zeros(8, dtype=torch.float64, device="meta"), torch.eye(8, dtype=torch.float64, device="meta"),
            torch.ones(8, dtype=torch.float64), torch.eye(8, dtype=torch.float64)).transform(_t(10, 8))
    zero = _pca(lam=torch.zeros(8, dtype=torch.float64))           # trace 0: no ridge can regularise
    with pytest.raises(ValueError, match="zero-variance direction"):
        zero.mahalanobis(_t(10, 8))
    singular = _pca(lam=torch.tensor([2.0, 1.0, 0, 0, 0, 0, 0, 0], dtype=torch.float64))
    with pytest.raises(ValueError, match="zero-variance direction"):
        singular.transform(_t(10, 8), whiten=True, ridge=0.0)


def test_whitening_and_explained_variance_on_the_host():
    lam = torch.tensor([4.0, 1.0, 0.0, -1e-17], dtype=torch.float64)
    p = _pca(4, lam)
    eps = 1e-2 * 5.0 / 4                                            # ridge * trace / dim (the trace of diag(lam))
    W = p._whitening("t", 4, 1e-2)
    want = torch.eye(4, dtype=torch.float64) / torch.sqrt(lam.clamp_min(0) + eps)[:, None]
    assert torch.allclose(W, want, rtol=1e-15, atol=0)
    assert torch.allclose(p.explained_variance_ratio, torch.tensor([0.8, 0.2, 0.0, 0.0], dtype=torch.float64))


def _vit():
    return M.ViTSpatialSpectral(image_size=8, spatial_patch_size=1, spectral_patch_size=10, num_classes=20, dim=96, depth=1, heads=8,
                                mlp_dim=64, channels=50, spectral_pos_embed=False)


def test_scene_argument_errors():
    m, cube = _vit(), _t(1, 50, 12, 12)
    for fn, kw in ((pca_scene, {}), (rx_scene, {})):
        with pytest.raises(ValueError, match="scene must be a"):
            fn(m, torch.zeros(50, 12, 12).as_subclass(_FakeCuda), **kw)
        with pytest.raises(ValueError, match="CUDA device"):
            fn(m, torch.zeros(1, 50, 12, 12), **kw)
        with pytest.raises(ValueError, match="ViTSpatialSpectral encoder"):
            fn(torch.nn.Linear(3, 3), cube, **kw)
        with pytest.raises(ValueError, match="valid must be a bool tensor"):
            fn(m, cube, valid=torch.ones(1, 12, 11, dtype=torch.bool), **kw)
        with pytest.raises(ValueError, match="valid must be a bool tensor"):
            fn(m, cube, valid=torch.ones(1, 12, 12, dtype=torch.uint8), **kw)
        one = torch.zeros(1, 12, 12, dtype=torch.bool)
        one[0, 3, 4] = True
        with pytest.raises(ValueError, match="1 pixels to fit on"):
            fn(m, cube, valid=one, **kw)
    for nc in (0, 97, 2.0, True):
        with pytest.raises(ValueError, match="n_components"):
            pca_scene(m, cube, n_components=nc)
    with pytest.raises(ValueError, match="ViTSpatialSpectral encoder"):
        pca_scene(None, cube)
    with pytest.raises(ValueError, match="ridge=-1"):
        rx_scene(m, cube, ridge=-1)
    with pytest.raises(ValueError, match="feature width 257"):
        rx_scene(None, _t(1, 257, 4, 4))


@pytest.mark.parametrize("kw, match", [
    (dict(maps=torch.zeros(1, 2, 4, 4)), "maps must be"),
    (dict(maps=torch.zeros(3, 4, 4)), "maps must be"),
    (dict(maps=torch.zeros(1, 3, 4, 4, dtype=torch.int32)), "maps must be"),
    (dict(maps=torch.zeros(0, 3, 4, 4)), "empty"),
    (dict(lo=-0.1), "lo=-0.1"),
    (dict(hi=1.5), "hi=1.5"),
    (dict(lo=0.5, hi=0.5), "must be below"),
    (dict(lo=True), "lo=True"),
])
def test_false_colour_argument_errors(kw, match):
    maps = kw.pop("maps", torch.zeros(1, 3, 4, 4))
    with pytest.raises(ValueError, match=match):
        false_colour(maps, **kw)


@pytest.mark.parametrize("lo, hi", [(0.01, 0.99), (0.0, 1.0), (0.25, 0.5), (0.013, 0.987)])
def test_false_colour_against_numpy_quantiles(lo, hi):
    rng = np.random.default_rng(3)
    maps = torch.from_numpy(rng.standard_normal((2, 3, 17, 23)) * np.array([1.0, 5.0, 0.01])[None, :, None, None]).float()
    maps[0, 2, :5] = 7.0                                            # ties at the top of one channel
    out = false_colour(maps, lo=lo, hi=hi)
    assert out.dtype == torch.float32 and out.shape == maps.shape
    v = maps.double().numpy()
    for c in range(3):
        a, b = np.quantile(v[:, c], lo), np.quantile(v[:, c], hi)
        want = (np.clip(v[:, c], a, b) - a) / (b - a)
        assert np.abs(out[:, c].double().numpy() - want).max() <= 1e-6
    assert float(out.min()) >= 0.0 and float(out.max()) <= 1.0
    flat = torch.ones(1, 3, 4, 4)
    assert torch.equal(false_colour(flat), torch.zeros(1, 3, 4, 4))   # equal quantiles: the channel maps to 0


def test_sign_rule():
    v = np.array([[0.1, -0.7, 0.7, 0.0],                           # |max| tie between 1 and 2: index 1 wins, so the row flips
                  [0.5, 0.5, -0.5, 0.5],                           # four-way tie: index 0 is positive already
                  [-0.2, 0.1, 0.3, -0.9],                          # largest is negative: flip
                  [0.0, 0.0, 0.0, 0.0]])                           # all zero: left as is
    out = _sign_rule(v.copy())
    assert np.array_equal(out[0], -v[0]) and np.array_equal(out[1], v[1]) and np.array_equal(out[2], -v[2])
    assert np.array_equal(out[3], v[3])
    for row in out[:3]:
        assert row[np.argmax(np.abs(row))] > 0


def _brute_auc(s, a):
    pos, neg = s[a], s[~a]
    gt = (pos[:, None] > neg[None, :]).sum()
    eq = (pos[:, None] == neg[None, :]).sum()
    return (gt + 0.5 * eq) / (pos.size * neg.size)


@pytest.mark.parametrize("na, nb, levels", [(1, 1, 3), (3, 200, 4), (150, 7, 5), (40, 60, 1000), (1, 500, 2), (25, 25, 1)])
def test_anomaly_auc_against_pair_counting_and_scipy(na, nb, levels):
    rng = np.random.default_rng(na * 1000 + nb + levels)
    s = rng.integers(0, levels, na + nb).astype(np.float64)        # few levels: many ties
    s[:na] += 0.5                                                   # anomalies score somewhat higher
    a = np.zeros(na + nb, bool)
    a[:na] = True
    perm = rng.permutation(na + nb)
    s, a = s[perm], a[perm]
    met = anomaly_metrics(torch.from_numpy(s), torch.from_numpy(a))
    assert met["n_anomalies"] == na and met["n_background"] == nb
    assert abs(met["auc"] - _brute_auc(s, a)) <= 1e-12
    u = mannwhitneyu(s[a], s[~a], alternative="two-sided").statistic
    assert abs(met["auc"] - u / (na * nb)) <= 1e-12
    # the ROC: one point per distinct score, descending, counted by brute force
    t = met["thresholds"].numpy()
    assert np.array_equal(t, np.unique(s)[::-1])
    for i, th in enumerate(t):
        assert met["tpr"][i] == (s[a] >= th).sum() / na and met["fpr"][i] == (s[~a] >= th).sum() / nb
    assert float(met["tpr"][-1]) == 1.0 and float(met["fpr"][-1]) == 1.0


def test_anomaly_argument_errors():
    s, a = torch.zeros(4, 5), torch.zeros(4, 5, dtype=torch.bool)
    a[0, 0] = True
    with pytest.raises(ValueError, match="0 anomalous and 20 background"):
        anomaly_metrics(s, torch.zeros(4, 5, dtype=torch.bool))
    with pytest.raises(ValueError, match="1 anomalous and 0 background"):
        anomaly_metrics(s, a, a)
    with pytest.raises(ValueError, match="anomalies must be a bool tensor"):
        anomaly_metrics(s, a.int())
    with pytest.raises(ValueError, match="anomalies must be a bool tensor"):
        anomaly_metrics(s, a[:3])
    with pytest.raises(ValueError, match="valid must be a bool tensor"):
        anomaly_metrics(s, a, torch.ones(4, 5))
    with pytest.raises(ValueError, match="score must be a real tensor"):
        anomaly_metrics(a, a)
    bad = s.clone()
    bad[1, 1] = float("nan")
    with pytest.raises(ValueError, match="NaN"):
        anomaly_metrics(bad, a)


def test_anomaly_valid_mask_and_shapes():
    rng = np.random.default_rng(5)
    s = torch.from_numpy(rng.standard_normal((2, 9, 11)))
    a = torch.from_numpy(rng.random((2, 9, 11)) < 0.2)
    v = torch.from_numpy(rng.random((2, 9, 11)) < 0.7)
    met = anomaly_metrics(s.float(), a, v)
    s64 = s.float().double().numpy()[v.numpy()]
    assert abs(met["auc"] - _brute_auc(s64, a.numpy()[v.numpy()])) <= 1e-12
    assert met["n_anomalies"] + met["n_background"] == int(v.sum())


def test_c_entry_points_refuse_bad_arguments_without_a_device():
    L = _lib.lib()
    assert L.msst_moments_workspace(100003, 96) == 8 * 7 * 96 * 97
    assert L.msst_moments_workspace(2, 1) == 16
    for n, dim, what in [(100, 0, b"dim=0"), (100, 257, b"dim=257"), (1, 8, b"n=1"), (2 ** 31, 8, b"n=2147483648"), (-5, 8, b"n=-5")]:
        assert L.msst_moments_workspace(n, dim) == -1 and what in L.msst_last_error()
        assert L.msst_moments_mean(n, dim, 1, 1, 1, None) == 1 and what in L.msst_last_error()
        assert L.msst_moments_cov(n, dim, 1, 1, 1, 1, None) == 1 and what in L.msst_last_error()
    for n, dim, k, what in [(100, 0, 1, b"dim=0"), (100, 257, 1, b"dim=257"), (0, 8, 1, b"n=0"), (2 ** 31, 8, 1, b"n=2147483648"),
                            (100, 8, 0, b"k=0"), (100, 8, 9, b"k=9")]:
        assert L.msst_moments_project(n, dim, k, 1, 1, 1, 1, 1, None) == 1 and what in L.msst_last_error(), (n, dim, k)
    for i in range(3):
        ptrs = [1, 1, 1]
        ptrs[i] = None
        assert L.msst_moments_mean(10, 8, *ptrs, None) == 1 and b"must be set" in L.msst_last_error()
    for i in range(4):
        ptrs = [1, 1, 1, 1]
        ptrs[i] = None
        assert L.msst_moments_cov(10, 8, *ptrs, None) == 1 and b"must be set" in L.msst_last_error()
    for i in range(3):
        ptrs = [1, 1, 1]
        ptrs[i] = None
        assert L.msst_moments_project(10, 8, 3, *ptrs, 1, 1, None) == 1 and b"must be set" in L.msst_last_error()
    assert L.msst_moments_project(10, 8, 3, 1, 1, 1, None, None, None) == 1 and b"both NULL" in L.msst_last_error()
    assert L.msst_moments_project(1, 1, 1, 1, 1, 1, None, None, None) == 1    # n = 1 is a valid projection chunk


def test_tpr_at_fpr_boundaries():
    """1000 background pixels at scores 0 .. 999 and anomalies at 999.5 (10), 997.5 (10), 989.5 (10), 899.5 (10) and -1 (10): the
    threshold 999 has FPR exactly 1e-3 and counts, the next one (998) has 2e-3."""
    bg = np.arange(1000, dtype=np.float64)
    an = np.repeat([999.5, 997.5, 989.5, 899.5, -1.0], 10)
    s = np.concatenate([an, bg])
    a = np.arange(s.size) < an.size
    met = anomaly_metrics(torch.from_numpy(s), torch.from_numpy(a))
    assert met["tpr_at_fpr"] == {1e-3: 0.2, 1e-2: 0.6, 1e-1: 0.8}
    # the highest background score (9) is above both anomalies (5): the first threshold already has FPR 0.1 and TPR 0
    only_top = np.concatenate([[5.0, 5.0], np.arange(10, dtype=np.float64)])
    met = anomaly_metrics(torch.from_numpy(only_top), torch.from_numpy(np.arange(12) < 2))
    assert met["tpr_at_fpr"] == {1e-3: 0.0, 1e-2: 0.0, 1e-1: 0.0}
