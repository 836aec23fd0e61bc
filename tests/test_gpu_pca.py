"""GPU: mean, covariance and projection of rows (csrc/moments.cu) and PCA / RX built on them (maskedsst_b200.inference.pca_fit / PCA /
pca_scene / rx_scene) against float64 torch and numpy.  The projection tests feed float64 torch the kernel's own mean and W (teacher
forcing); the order tests build slice partials whose fp64 total depends on the order of addition."""
import json

import numpy as np
import pytest
import torch

import maskedsst_b200 as M
from maskedsst_b200 import _lib
from maskedsst_b200.inference import (_moments_cov, _moments_mean, _moments_project, _pixel_rows, anomaly_metrics, embed_scene, pca_fit,
                                      pca_scene, rx_scene)
from oracle import maskedsst_oracle as O
from tests.helpers import gold, rel_l2
from tests.test_gpu_scene_embed import _oracle_embed
from tests.test_gpu_scene_inference import _model

pytestmark = pytest.mark.gpu
DEV = "cuda"
SLICE = 16384
U32 = 2.0 ** -24
WORST = {}


def _note(key, err):
    WORST[key] = max(WORST.get(key, 0.0), err)
    print(f"{key}: {err:.2e} (worst so far {WORST[key]:.2e})")


def _workspace(n, dim):
    return torch.empty(_lib.lib().msst_moments_workspace(n, dim), device=DEV, dtype=torch.uint8)


def _moments(x):
    n, D = x.shape
    ws = _workspace(n, D)
    mean = torch.full((D,), float("nan"), device=DEV, dtype=torch.float64)
    cov = torch.full((D, D), float("nan"), device=DEV, dtype=torch.float64)
    _moments_mean(x, ws, mean)
    _moments_cov(x, mean, ws, cov)
    return mean, cov, ws


def _rows(n, D, seed, offset=1e3):
    """Correlated rows with column scales spread over 1e-2 .. 1e2, offset from the origin."""
    g = torch.Generator(device=DEV).manual_seed(seed)
    mix = torch.randn(D, D, device=DEV, generator=g) / D ** 0.5 + torch.eye(D, device=DEV)
    scale = torch.logspace(-2, 2, D, device=DEV)
    return ((torch.randn(n, D, device=DEV, generator=g) @ mix) * scale + offset).contiguous()


@pytest.mark.parametrize("D", [1, 7, 32, 50, 96, 129, 200, 256])
def test_mean_and_covariance_vs_fp64(D):
    """Rows offset by 1e3: the two-pass fp64 covariance is within 1e-10 of sum_r |c_ri||c_rj| / (n - 1) of float64 torch (the one-pass
    form lands near 1e-8 there), exactly symmetric, and bitwise reproducible."""
    for n in (2, SLICE - 1, SLICE, SLICE + 1, 100003):
        x = _rows(n, D, seed=D * 7 + n)
        mean, cov, _ = _moments(x)
        x64 = x.double()
        m64 = x64.mean(0)
        c64 = x64 - m64
        cov64 = c64.T @ c64 / (n - 1)
        scale = c64.abs().T @ c64.abs() / (n - 1)
        err_m = float(((mean - m64).abs() / x64.abs().mean(0)).max())
        err_c = float(((cov - cov64).abs() / scale.clamp_min(1e-300)).max())
        _note("mean rel", err_m)
        _note("cov rel to sum|c_i||c_j|/(n-1)", err_c)
        assert err_m <= 1e-11 and err_c <= 1e-10, (n, err_m, err_c)
        assert torch.equal(cov, cov.T)
        mean2, cov2, _ = _moments(x)
        assert torch.equal(mean, mean2) and torch.equal(cov, cov2)


def test_mean_adds_the_slices_in_ascending_order():
    """Column-0 slice sums 1, 2^-53, 2^-53 over three slices: in ascending order the fp64 total is 1 (each 2^-53 is half an ulp of 1 and
    rounds to even), in descending order 1 + 2^-52; divided by n = 3 * 16384 the two totals give different means."""
    n, D = 3 * SLICE, 4
    x = torch.zeros(n, D, device=DEV)
    x[0, 0] = 1.0
    x[SLICE, 0] = 2.0 ** -53
    x[2 * SLICE, 0] = 2.0 ** -53
    mean, _, ws = _moments(x)
    part = ws[:8 * 3 * D].view(torch.float64).view(3, D)
    assert part[:, 0].tolist() == [1.0, 2.0 ** -53, 2.0 ** -53]
    assert 1.0 / n != (1.0 + 2.0 ** -52) / n
    assert float(mean[0]) == 1.0 / n


def test_covariance_adds_the_slices_in_ascending_order():
    """Entry (0, 1) of slice partials 1, 2^-53, 2^-53 (row pairs (a, b), (-a, -b), so every column mean is exactly 0): ascending gives
    1, descending 1 + 2^-52, and cov = total / (n - 1) tells them apart."""
    n, D = 3 * SLICE, 3
    x = torch.zeros(n, D, device=DEV)
    for s, (a, b) in enumerate([(1.0, 0.5), (2.0 ** -27, 2.0 ** -27), (2.0 ** -27, 2.0 ** -27)]):
        x[s * SLICE, :2] = torch.tensor([a, b])
        x[s * SLICE + 1, :2] = torch.tensor([-a, -b])
    mean, cov, ws = _moments(x)
    assert torch.equal(mean, torch.zeros_like(mean))
    part = ws[8 * 3 * D:].view(torch.float64).view(3, D, D)
    assert part[:, 0, 1].tolist() == [1.0, 2.0 ** -53, 2.0 ** -53]
    assert 1.0 / (n - 1) != (1.0 + 2.0 ** -52) / (n - 1)
    assert float(cov[0, 1]) == 1.0 / (n - 1) and float(cov[1, 0]) == 1.0 / (n - 1)


def _check_projection(x, mean, W, key):
    """y and score of the kernel against float64 torch fed the kernel's mean and W:
      |y - y64| <= 2^-24 |y64| + 1e-12 ||c|| ||W_j||
      |score - s64| <= 2^-24 s64 + sum_j (2 |y64_j| e_j + e_j^2) + 1e-12 s64,  e_j = 1e-12 ||c|| ||W_j||   (DESIGN.md §4)."""
    n, k = x.shape[0], W.shape[0]
    y = torch.full((n, k), float("nan"), device=DEV)
    score = torch.full((n,), float("nan"), device=DEV)
    _moments_project(x, mean, W, y=y, score=score)
    c = x.double() - mean
    y64 = c @ W.T
    s64 = (y64 * y64).sum(1)
    e = 1e-12 * c.norm(dim=1)[:, None] * W.norm(dim=1)[None, :]
    err_y = (y.double() - y64).abs()
    tol_y = U32 * y64.abs() + e
    assert bool((err_y <= tol_y).all()), float((err_y / tol_y).max())
    tol_s = U32 * s64 + (2 * y64.abs() * e + e * e).sum(1) + 1e-12 * s64
    err_s = (score.double() - s64).abs()
    assert bool((err_s <= tol_s).all()), float((err_s / tol_s).max())
    _note(f"{key} y err / bound", float((err_y / tol_y).max()))
    _note(f"{key} score err / bound", float((err_s / tol_s).max()))
    y_only = torch.full((n, k), float("nan"), device=DEV)
    s_only = torch.full((n,), float("nan"), device=DEV)
    _moments_project(x, mean, W, y=y_only)
    _moments_project(x, mean, W, score=s_only)
    assert torch.equal(y, y_only) and torch.equal(score, s_only)
    return y, score


@pytest.mark.parametrize("D", [7, 50, 96, 256])
def test_projection_teacher_forced(D):
    """Random W at k = 1, 3, 16 (the 256-row tile), 17 (the 64-row tile) and dim, rows offset by 1e3."""
    x = _rows(20001, D, seed=D)
    mean, _, _ = _moments(x)
    g = torch.Generator(device=DEV).manual_seed(D + 1)
    Wall = torch.randn(D, D, device=DEV, dtype=torch.float64, generator=g)
    ys = {}
    for k in sorted({1, 3, min(16, D), min(17, D), D}):
        ys[k], _ = _check_projection(x, mean, Wall[:k].contiguous(), "projection")
    for k in ys:                                             # a component's y does not depend on k or on the tile shape
        assert torch.equal(ys[k], ys[D][:, :k])


def _conditioned(n, D, kappa, seed, offset=1e3):
    """Gaussian rows with covariance Q diag(logspace(0, -log10 kappa)) Q^T, offset from the origin."""
    g = torch.Generator(device=DEV).manual_seed(seed)
    q, _ = torch.linalg.qr(torch.randn(D, D, device=DEV, dtype=torch.float64, generator=g))
    lam = torch.logspace(0, -np.log10(kappa), D, device=DEV, dtype=torch.float64)
    z = torch.randn(n, D, device=DEV, dtype=torch.float64, generator=g)
    return ((z * lam.sqrt()) @ q.T + offset).float().contiguous()


@pytest.mark.parametrize("D", [32, 96, 256])
def test_whitened_projection_at_condition_1e8(D):
    """The whitening matrix of a covariance of condition 1e8: fp32 staging of W, or an fp32 mean, would be off by orders of magnitude
    more than the bound."""
    x = _conditioned(50000, D, 1e8, seed=D)
    pca = pca_fit(x)
    lam = pca.eigenvalues
    assert float(lam[0] / lam[-1]) > 1e7
    W = pca._whitening("t", D, 0.0)
    _check_projection(x, pca.mean, W, "whitened")


def test_batch_queries_give_the_same_bits():
    x = _rows(3001, 50, seed=3)
    pca = pca_fit(x)
    for whiten in (False, True):
        ref = pca.transform(x, 5, whiten=whiten)
        for b in (1, 1000):
            assert torch.equal(pca.transform(x, 5, whiten=whiten, batch_queries=b), ref)
    ref = pca.mahalanobis(x)
    for b in (1, 1000):
        assert torch.equal(pca.mahalanobis(x, batch_queries=b), ref)


@pytest.mark.parametrize("D", [1, 7, 50, 96, 256])
def test_pca_fit_eigenvalues_and_signs(D):
    x = _rows(30000, D, seed=D + 11)
    pca = pca_fit(x)
    x64 = x.double()
    c64 = x64 - x64.mean(0)
    lam64 = np.linalg.eigh((c64.T @ c64 / (x.shape[0] - 1)).cpu().numpy())[0][::-1]
    err = float(np.abs(pca.eigenvalues.cpu().numpy() - lam64).max() / lam64[0])
    _note("eigenvalues / lambda_max", err)
    assert err <= 1e-9
    assert bool((pca.eigenvalues[:-1] >= pca.eigenvalues[1:]).all())
    V = pca.components
    assert torch.allclose(V @ V.T, torch.eye(D, device=DEV, dtype=torch.float64), atol=1e-12)
    for row in V.cpu().numpy():
        assert row[np.argmax(np.abs(row))] > 0                                 # the sign rule (numpy's argmax: lowest index on ties)
    r = pca.explained_variance_ratio
    assert abs(float(r.sum()) - 1.0) <= 1e-12
    assert pca.n == x.shape[0] and pca.covariance.shape == (D, D) and pca.mean.dtype == torch.float64


def test_zero_variance_column():
    """A constant column: its variance and covariances are exactly 0, its eigenvalue is 0 within rounding, and RX with the default ridge
    stays finite."""
    x = _rows(20000, 16, seed=5)
    x[:, 6] = 3.25
    pca = pca_fit(x)
    assert bool((pca.covariance[6] == 0).all()) and bool((pca.covariance[:, 6] == 0).all())
    assert abs(float(pca.eigenvalues[-1])) <= 1e-12 * float(pca.eigenvalues[0])
    e = pca.components[-1].abs()
    assert float(e[6]) == pytest.approx(1.0, abs=1e-6) and float(pca.components[-1][6]) > 0
    s = pca.mahalanobis(x)
    assert bool(torch.isfinite(s).all())
    y = pca.transform(x, whiten=True)
    assert bool(torch.isfinite(y).all())


def test_rx_of_gaussian_rows_is_chi_square():
    """The mean RX score of n = 10^5 Gaussian rows is dim (n - 1) / n (exactly, for the fitted covariance without ridge) up to the ridge;
    a planted shift of 10 sigma in every feature gives auc = 1."""
    D, n = 50, 100000
    g = torch.Generator(device=DEV).manual_seed(12)
    x = (torch.randn(n, D, device=DEV, generator=g) * torch.linspace(0.5, 3.0, D, device=DEV)).contiguous()
    s = pca_fit(x).mahalanobis(x)
    assert abs(float(s.double().mean()) - D * (n - 1) / n) <= 1e-3 * D
    out = torch.randint(0, n, (50,), device=DEV, generator=g)
    x[out] += 10.0 * torch.linspace(0.5, 3.0, D, device=DEV)
    s = pca_fit(x).mahalanobis(x)
    truth = torch.zeros(n, dtype=torch.bool, device=DEV)
    truth[out] = True
    met = anomaly_metrics(s, truth)
    assert met["auc"] == 1.0 and met["tpr_at_fpr"][1e-3] == 1.0


def _pca64(rows, ridge):
    """float64 PCA / RX reference on numpy rows [n, D]: (mean, eigenvalues descending, components with the sign rule, RX scores)."""
    m = rows.mean(0)
    c = rows - m
    cov = c.T @ c / (rows.shape[0] - 1)
    lam, vec = np.linalg.eigh(cov)
    lam, vec = lam[::-1], vec[:, ::-1].T.copy()
    idx = np.argmax(np.abs(vec), 1)
    vec[vec[np.arange(len(vec)), idx] < 0] *= -1
    eps = ridge * np.trace(cov) / cov.shape[0]
    rx = (((c @ vec.T) ** 2) / (np.maximum(lam, 0) + eps)).sum(1)
    return m, lam, vec, c, rx


def _scene(case):
    m, spec, sd = _model(O.HOUSTON, 2, 81)
    cube = torch.from_numpy(np.random.default_rng(7).standard_normal((2, spec.channels, 21, 19)).astype(np.float32))
    model = M.SimMIMSpatialSpectral(encoder=m, masking_ratio=0.5).to(DEV) if case == "simmim" else m
    return model, spec, sd, cube


@pytest.mark.parametrize("case", ["vit", "simmim"])
def test_pca_and_rx_scene_vs_oracle(case):
    """pca_scene / rx_scene against the float64 scene-embedding oracle followed by float64 PCA / RX (ridge 1e-3 for RX: with ~800 pixels
    of 96 features the smallest eigenvalues are tiny, and RX amplifies the features' fp32 rounding by sqrt(condition))."""
    model, spec, sd, cube = _scene(case)
    B, _, H, W = cube.shape
    maps, pca = pca_scene(model, cube.to(DEV), n_components=3, stride=3)
    assert maps.shape == (B, 3, H, W) and maps.dtype == torch.float32
    feats = _oracle_embed(cube, sd, spec, 3, None)                              # float64 [B, D, H, W]
    rows = feats.transpose(0, 2, 3, 1).reshape(B * H * W, -1)
    _, lam, vec, c, rx = _pca64(rows, 1e-3)
    err_l = float(np.abs(pca.eigenvalues.cpu().numpy() - lam).max() / lam[0])
    want = (c @ vec[:3].T).reshape(B, H, W, 3).transpose(0, 3, 1, 2)
    err_m = rel_l2(maps, want)
    _note(f"pca_scene eigenvalues ({case})", err_l)
    _note(f"pca_scene maps rel-l2 ({case})", err_m)
    assert err_l <= 1e-5 and err_m <= 1e-5
    scores, _ = rx_scene(model, cube.to(DEV), ridge=1e-3, stride=3)
    err_r = rel_l2(scores, rx.reshape(B, H, W))
    _note(f"rx_scene rel-l2 ({case})", err_r)
    assert scores.shape == (B, H, W) and err_r <= 1e-5


def test_rx_on_raw_spectra():
    """model=None: RX on the cube's own spectra, and on int16 RawTiles with pad bands and a clip (rows = standardize(pad=False))."""
    cube = torch.from_numpy(np.random.default_rng(8).standard_normal((2, 48, 23, 17)).astype(np.float32)) * 2 + 5
    scores, pca = rx_scene(None, cube.to(DEV))
    *_, rx = _pca64(cube.double().numpy().transpose(0, 2, 3, 1).reshape(-1, 48), 1e-6)
    err = rel_l2(scores, rx.reshape(2, 23, 17))
    _note("rx raw cube rel-l2", err)
    assert err <= 1e-5 and pca.dim == 48
    g = gold("input_pipeline")
    means, stds, meta = g["houston__means"], g["houston__stds"], json.loads(str(g["houston__meta"]))
    raw = torch.from_numpy(np.random.default_rng(9).integers(-400, 12000, (1, 48, 17, 23)).astype(np.int16)).to(DEV)
    rt = M.RawTiles(raw, means, stds, image_size=8, pad_bands=meta["pad"], clip=(-1.5, 1.5))
    assert meta["pad"] > 0
    scores, pca = rx_scene(None, rt)
    assert pca.dim == 48
    rows = rt.standardize(raw, pad=False).double().cpu().numpy().transpose(0, 2, 3, 1).reshape(-1, 48)
    *_, rx = _pca64(rows, 1e-6)
    err = rel_l2(scores, rx.reshape(1, 17, 23))
    _note("rx raw tiles rel-l2", err)
    assert err <= 1e-5


def test_valid_mask_fits_on_the_gathered_rows():
    model, spec, sd, cube = _scene("vit")
    B, _, H, W = cube.shape
    valid = torch.from_numpy(np.random.default_rng(3).random((B, H, W)) < 0.6).to(DEV)
    flat = _pixel_rows(embed_scene(model, cube.to(DEV), stride=3)).contiguous()
    fit = pca_fit(flat[valid.reshape(-1)])
    maps, pca = pca_scene(model, cube.to(DEV), n_components=4, valid=valid, stride=3)
    assert pca.n == int(valid.sum()) and torch.equal(pca.covariance, fit.covariance) and torch.equal(pca.mean, fit.mean)
    assert torch.equal(maps, fit.transform(flat, 4).reshape(B, H, W, 4).permute(0, 3, 1, 2))
    scores, _ = rx_scene(model, cube.to(DEV), valid=valid, stride=3)
    assert torch.equal(scores, fit.mahalanobis(flat).reshape(B, H, W))


def test_c_abi_limits_leave_outputs_untouched():
    L = _lib.lib()
    n, D = 300, 8
    x = torch.randn(n, D, device=DEV)
    W = torch.randn(D, D, device=DEV, dtype=torch.float64)
    ws = torch.full((1 << 20,), 7, device=DEV, dtype=torch.uint8)
    mean = torch.full((300,), 7.0, device=DEV, dtype=torch.float64)
    cov = torch.full((300 * 300,), 7.0, device=DEV, dtype=torch.float64)
    y = torch.full((n * 300,), 7.0, device=DEV)
    sc = torch.full((n,), 7.0, device=DEV)
    st = None
    for nn, dim in [(n, 0), (n, 257), (1, D), (0, D)]:
        assert L.msst_moments_mean(nn, dim, x.data_ptr(), ws.data_ptr(), mean.data_ptr(), st) == 1
        assert L.msst_moments_cov(nn, dim, x.data_ptr(), mean.data_ptr(), ws.data_ptr(), cov.data_ptr(), st) == 1
    for nn, dim, k in [(n, 0, 1), (n, 257, 1), (0, D, 1), (n, D, 0), (n, D, D + 1)]:
        assert L.msst_moments_project(nn, dim, k, x.data_ptr(), mean.data_ptr(), W.data_ptr(), y.data_ptr(), sc.data_ptr(), st) == 1
    assert L.msst_moments_mean(n, D, None, ws.data_ptr(), mean.data_ptr(), st) == 1
    assert L.msst_moments_mean(n, D, x.data_ptr(), None, mean.data_ptr(), st) == 1
    assert L.msst_moments_cov(n, D, x.data_ptr(), None, ws.data_ptr(), cov.data_ptr(), st) == 1
    assert L.msst_moments_cov(n, D, x.data_ptr(), mean.data_ptr(), ws.data_ptr(), None, st) == 1
    assert L.msst_moments_project(n, D, 3, x.data_ptr(), mean.data_ptr(), None, y.data_ptr(), sc.data_ptr(), st) == 1
    assert L.msst_moments_project(n, D, 3, x.data_ptr(), mean.data_ptr(), W.data_ptr(), None, None, st) == 1
    torch.cuda.synchronize()
    for t in (ws, mean, cov, y, sc):
        assert bool((t == 7).all())
