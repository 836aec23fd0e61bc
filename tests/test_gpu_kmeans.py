"""GPU: k-means clustering (maskedsst_b200.inference.kmeans_fit / KMeans / cluster_scene, csrc/kmeans.cu) against float64 torch.  The
tight tests feed the float64 reference the kernel's own state (teacher forcing): its centroids for the assignment, its labels for the
update, its mindist and uniforms for the seeding, and the workspace partials for the documented summation order."""
import ctypes
import math

import numpy as np
import pytest
import torch
import torch.nn.functional as F

import maskedsst_b200 as M
from maskedsst_b200 import _lib
from maskedsst_b200.inference import (_kmeans_assign, _kmeans_dims, _kmeans_seed, _kmeans_uniforms, _kmeans_update, _pixel_rows,
                                      cluster_scene, clustering_metrics, embed_scene, kmeans_fit)
from oracle import maskedsst_oracle as O
from tests.test_gpu_scene_embed import _oracle_embed
from tests.test_gpu_scene_inference import _model

pytestmark = pytest.mark.gpu
DEV = "cuda"
SLICE = 4096
WORST = {}


def _note(key, err):
    WORST[key] = max(WORST.get(key, 0.0), err)
    print(f"{key}: {err:.2e} (worst so far {WORST[key]:.2e})")


def _rows64(x, normalize):
    x = x.double()
    return F.normalize(x, dim=1, eps=1e-12) if normalize else x


def _d64(y, c):
    """float64 squared distances [n, K] (difference form, in row chunks)."""
    out = torch.empty(y.shape[0], c.shape[0], dtype=torch.float64, device=y.device)
    step = max(1, (1 << 24) // (c.shape[0] * c.shape[1]))
    for a in range(0, y.shape[0], step):
        out[a:a + step] = ((y[a:a + step, None, :] - c[None].double()) ** 2).sum(-1)
    return out


def _tiny(normalize):
    # normalised rows: the reference normalises in float64, the kernel in fp32 (~6e-8 relative per element), which moves a distance
    # d by up to ~2 sqrt(d) 1e-7: that floor is 1e-5 * tiny for d up to 1.  Raw rows are the same bits on both sides.
    return 1e-3 if normalize else 1e-30


class _Ws:
    """Views of a msst_kmeans workspace (include/msst.h): inertia / slice sums [R, S] f64, sums [R, S, K, D] f32, counts, changed."""

    def __init__(self, ws, R, n, K, D):
        S = -(-n // SLICE)
        o = 0
        self.inertia = ws[o:o + 8 * R * S].view(torch.float64).view(R, S)
        o += 8 * R * S
        self.sums = ws[o:o + 4 * R * S * K * D].view(torch.float32).view(R, S, K, D)
        o += 4 * R * S * K * D
        self.counts = ws[o:o + 4 * R * S * K].view(torch.int32).view(R, S, K)
        o += 4 * R * S * K
        self.changed = ws[o:o + 4 * R * S].view(torch.int32).view(R, S)


def _workspace(dims):
    return torch.empty(_lib.lib().msst_kmeans_workspace(ctypes.byref(dims)), device=DEV, dtype=torch.uint8)


def _check_assign(y64, cent, labels, dist, normalize, key):
    """Every row: d64[label] is a minimum within 1e-5 relative, dist is d64[label] within the same bound, and a label is the lowest index
    among bitwise-equal centroids."""
    d64 = _d64(y64, cent)
    lo = d64.min(1).values
    at = d64.gather(1, labels[:, None])[:, 0]
    tol = 1e-5 * (lo + _tiny(normalize))
    assert bool((at <= lo + tol).all()), float(((at - lo) / (lo + _tiny(normalize))).max())
    if dist is not None:
        err = (dist.double() - at).abs()
        assert bool((err <= tol).all()), float((err / (lo + _tiny(normalize))).max())
        _note(f"{key} dist rel", float((err / (lo + _tiny(normalize))).max()))
    K = cent.shape[0]
    eq = (cent[:, None, :] == cent[None, :, :]).all(-1)                         # [K, K] bitwise-equal centroids
    lowest = torch.argmax(eq.int(), 1)                                           # the first equal one
    assert torch.equal(lowest[labels], labels)


def _cap(D):
    return min(256, 16384 // D)


@pytest.mark.parametrize("normalize", [False, True])
@pytest.mark.parametrize("D", [32, 96, 256])
@pytest.mark.parametrize("kk", [1, 7, 20, 64, "cap"])
def test_assign_and_update_vs_fp64(kk, D, normalize):
    K = _cap(D) if kk == "cap" else kk
    g = torch.Generator(device=DEV).manual_seed(D * 1000 + K + normalize)
    for R in (1, 3, 16):
        for n in sorted({K, 4095, 4097, 50000} if R < 16 else {max(K, 4097)}):
            if n < K:
                continue
            x = 2.0 * torch.randn(n, D, device=DEV, generator=g) + 0.5
            cent = x[torch.randint(0, n, (R, K), device=DEV, generator=g)] + 0.3 * torch.randn(R, K, D, device=DEV, generator=g)
            if K >= 3:
                cent[:, K - 1] = cent[:, K // 3]                                 # a duplicate: every tie must go to K // 3, K - 1 stays empty
            if normalize:
                cent = F.normalize(cent, dim=2)
            cent = cent.contiguous()
            prev = torch.randint(-1, K, (R, n), device=DEV, generator=g)
            labels, dist = prev.clone(), torch.full((R, n), -7.0, device=DEV)
            dims = _kmeans_dims(n, D, K, R, normalize)
            ws = _workspace(dims)
            _kmeans_assign(dims, x, cent, labels, dist, ws)
            y64 = _rows64(x, normalize)
            for r in range(R):
                _check_assign(y64, cent[r], labels[r], dist[r], normalize, "assign")
            w = _Ws(ws, R, n, K, D)
            assert torch.equal(w.changed.sum(1).long(), (labels != prev).sum(1))
            for r in range(R):
                assert torch.equal(w.counts[r].sum(0).long(), torch.bincount(labels[r], minlength=K))
            # update: the documented order over the partials, bitwise; and the float64 means of the rows, to 1e-6
            new = cent.clone()
            inertia = torch.empty(R, device=DEV, dtype=torch.float64)
            changed = torch.empty(R, device=DEV, dtype=torch.int32)
            empty = torch.empty(R, device=DEV, dtype=torch.int32)
            _kmeans_update(dims, ws, new, inertia, changed, empty)
            acc = torch.zeros(R, K, D, device=DEV, dtype=torch.float64)
            ins = torch.zeros(R, device=DEV, dtype=torch.float64)
            for s in range(w.sums.shape[1]):                                     # ascending slices, one rounding per add
                acc = acc + w.sums[:, s].double()
                ins = ins + w.inertia[:, s]
            cnt = w.counts.sum(1).long()
            want = torch.where(cnt[..., None] > 0, (acc / cnt[..., None].clamp_min(1)).float(), cent)
            assert torch.equal(new, want)
            assert torch.equal(inertia, ins)
            assert torch.equal(changed.long(), (labels != prev).sum(1).int().long())
            assert torch.equal(empty.long(), (cnt == 0).sum(1))
            for r in range(R):
                lab = labels[r]
                c64 = torch.zeros(K, D, device=DEV, dtype=torch.float64).index_add_(0, lab, y64)
                a64 = torch.zeros(K, D, device=DEV, dtype=torch.float64).index_add_(0, lab, y64.abs())
                k = cnt[r] > 0
                mean = c64[k] / cnt[r][k, None]
                err = (new[r][k].double() - mean).abs()
                assert bool((err <= 1e-6 * (a64[k] / cnt[r][k, None]) + 1e-6 * mean.abs()).all())
                _note("update rel", float((err / (a64[k] / cnt[r][k, None])).max()))
                assert torch.equal(new[r][~k], cent[r][~k])                    # empty: kept bit for bit
                i64 = _d64(y64, cent[r]).gather(1, lab[:, None]).sum()
                assert abs(float(inertia[r]) - float(i64)) <= 1e-5 * float(i64) + 1e-30
                if K >= 3:
                    assert int(cnt[r, K - 1]) == 0
            # prediction mode: no workspace, labels not read; the same bits as the fit-mode launch, any n >= 1
            for q in sorted({1, min(33, n)}):
                pl = torch.full((1, q), 5, device=DEV, dtype=torch.int64)
                pd = torch.empty(1, q, device=DEV)
                _kmeans_assign(_kmeans_dims(q, D, K, 1, normalize), x[:q], cent[R - 1].contiguous(), pl, pd)
                assert torch.equal(pl[0], labels[R - 1, :q]) and torch.equal(pd[0], dist[R - 1, :q])


def test_update_adds_the_slices_in_ascending_order():
    """Slice inertias 1, 2^-53, 2^-53 (three 4096-row slices, one cluster at the origin): in ascending order the fp64 total is 1 (each
    2^-53 is half an ulp of 1 and rounds away), in any other order the two small partials meet first and the total is 1 + 2^-52.
    (Partials of fp32 rows of similar magnitude add exactly in fp64, so only such a spread can tell the orders apart.)"""
    n, D = 3 * SLICE, 32
    x = torch.zeros(n, D, device=DEV)
    x[0, 0] = 1.0
    x[SLICE:SLICE + 2, 0] = 2.0 ** -27                                           # each row's distance 2^-54, the slice's 2^-53
    x[2 * SLICE:2 * SLICE + 2, 0] = 2.0 ** -27
    cent = torch.zeros(1, 1, D, device=DEV)
    dims = _kmeans_dims(n, D, 1, 1, False)
    ws = _workspace(dims)
    labels = torch.full((1, n), -1, device=DEV, dtype=torch.int64)
    _kmeans_assign(dims, x, cent, labels, workspace=ws)
    w = _Ws(ws, 1, n, 1, D)
    assert w.inertia[0].tolist() == [1.0, 2.0 ** -53, 2.0 ** -53]
    inertia, changed, empty = (torch.empty(1, device=DEV, dtype=t) for t in (torch.float64, torch.int32, torch.int32))
    _kmeans_update(dims, ws, cent, inertia, changed, empty)
    assert float(inertia[0]) == 1.0 and int(changed[0]) == n and int(empty[0]) == 0
    assert float(cent[0, 0, 0]) == float(np.float32((1.0 + 4 * 2.0 ** -27) / n))


def test_update_adds_the_centroid_sums_in_ascending_order():
    """One cluster's feature-0 slice sums 1, 2^-53, 2^-53, 2^-24 over four rows (one per slice): in ascending order the fp64 total is
    1 + 2^-24 (each 2^-53 rounds away against 1), whose quarter 0.25 + 2^-26 is an fp32 midpoint and rounds to even, 0.25; in descending
    order the total is 1 + 2^-24 + 2^-52 and the centroid rounds up to 0.25 + 2^-25.  The other rows form cluster 1."""
    n, D = 4 * SLICE, 32
    x = torch.zeros(n, D, device=DEV)
    x[:, 1] = 5.0
    for s_, v in enumerate([1.0, 2.0 ** -53, 2.0 ** -53, 2.0 ** -24]):
        x[s_ * SLICE, 0], x[s_ * SLICE, 1] = v, 0.0
    cent = torch.zeros(1, 2, D, device=DEV)
    cent[0, 1, 1] = 5.0
    dims = _kmeans_dims(n, D, 2, 1, False)
    ws = _workspace(dims)
    labels = torch.full((1, n), -1, device=DEV, dtype=torch.int64)
    _kmeans_assign(dims, x, cent, labels, workspace=ws)
    assert int((labels == 0).sum()) == 4 and all(int(labels[0, s_ * SLICE]) == 0 for s_ in range(4))
    inertia, changed, empty = (torch.empty(1, device=DEV, dtype=t) for t in (torch.float64, torch.int32, torch.int32))
    _kmeans_update(dims, ws, cent, inertia, changed, empty)
    assert float(cent[0, 0, 0]) == 0.25 and float(cent[0, 1, 1]) == 5.0


def test_offset_rows_need_the_difference_form():
    """Rows offset by 1e3 with unit spread: |y|^2 ~ 1e8, where fp32 |y|^2 - 2 y.c + |c|^2 is off by tens, far above the gaps between
    the distances (~200)."""
    g = torch.Generator(device=DEV).manual_seed(4)
    n, D, K = 20000, 96, 20
    x = 1e3 + torch.randn(n, D, device=DEV, generator=g)
    cent = (1e3 + 0.5 * torch.randn(1, K, D, device=DEV, generator=g)).contiguous()
    labels = torch.empty(1, n, device=DEV, dtype=torch.int64)
    dist = torch.empty(1, n, device=DEV)
    _kmeans_assign(_kmeans_dims(n, D, K, 1, False), x, cent, labels, dist)
    _check_assign(x.double(), cent[0], labels[0], dist[0], False, "offset")
    want = _d64(x.double(), cent[0]).argmin(1)
    assert float((labels[0] == want).double().mean()) == 1.0


def _replay_pick(md, u, n, j):
    """float64 replay of k-means++ round j > 0 from the kernel's mindist [n] (fp32) and u: -> row, or None for the T == 0 rule."""
    S = -(-n // SLICE)
    m = md.double().cpu().numpy()
    sums = [np.cumsum(m[s * SLICE:(s + 1) * SLICE])[-1] for s in range(S)]      # sequential, as the kernel adds
    T = 0.0
    for v in sums:
        T += v
    if not T > 0:
        return None, sums
    t = u * T
    P = 0.0
    for s, v in enumerate(sums):
        if P + v > t:
            L = np.cumsum(m[s * SLICE:(s + 1) * SLICE])
            return s * SLICE + int(np.argmax(P + L > t)), sums
        P = P + v
    raise AssertionError("no slice crosses the threshold")


@pytest.mark.parametrize("normalize", [False, True])
@pytest.mark.parametrize("case", ["random", "duplicates", "identical"])
def test_seeding_replayed_round_by_round(case, normalize):
    g = torch.Generator(device=DEV).manual_seed(7 + normalize)
    n, D, K, R = 9000, 64, 12, 3
    if case == "identical":
        x = torch.randn(1, D, device=DEV, generator=g).repeat(n, 1)
    else:
        x = torch.randn(n, D, device=DEV, generator=g) + 1.0
        if case == "duplicates":
            x[4000:8200] = x[5]                                                  # most mass on one repeated row
    u = torch.rand(R, K, device=DEV, dtype=torch.float64, generator=g)
    u[0, :2] = 0.0                                                               # row 0 first, then the threshold t = 0
    u[1, 3] = 0.0
    dims = _kmeans_dims(n, D, K, R, normalize)
    ws = _workspace(dims)
    w = _Ws(ws, R, n, K, D)
    cent = torch.empty(R, K, D, device=DEV)
    index = torch.empty(R, K, device=DEV, dtype=torch.int64)
    mindist = torch.empty(R, n, device=DEV)
    y64 = _rows64(x, normalize)
    fallbacks = 0
    for j in range(K):
        before = mindist.clone()
        _kmeans_seed(dims, j, x, u, cent, index, mindist, ws)
        for r in range(R):
            ur = float(u[r, j])
            want = None
            if j > 0:
                want, sums = _replay_pick(before[r], ur, n, j)
            if want is None:
                want = min(math.floor(ur * n), n - 1)
                fallbacks += j > 0
            assert int(index[r, j]) == want, (case, r, j, int(index[r, j]), want)
            if normalize:
                assert (cent[r, j].double() - y64[want]).abs().max().item() <= 1e-6
            else:
                assert torch.equal(cent[r, j], x[want])
            if j + 1 < K:                                                        # mindist and its slice sums after the round
                d = _d64(y64, cent[r, :j + 1]).min(1).values
                assert bool(((mindist[r].double() - d).abs() <= 1e-5 * (d + _tiny(normalize))).all())
                m = mindist[r].double().cpu().numpy()
                for s in range(w.inertia.shape[1]):
                    assert float(w.inertia[r, s]) == np.cumsum(m[s * SLICE:(s + 1) * SLICE])[-1]
    if case == "identical":
        assert fallbacks == R * (K - 1)                                          # T == 0 every round
    else:
        assert fallbacks == 0
        assert int(index[0, 0]) == 0 and int(index[0, 1]) != 0                  # t = 0 takes the first row of positive mindist


def _blobs(n, D, K, seed, sep=10.0):
    g = torch.Generator(device=DEV).manual_seed(seed)
    means = sep * torch.randn(K, D, device=DEV, generator=g)
    y = torch.randint(0, K, (n,), device=DEV, generator=g)
    return means[y] + torch.randn(n, D, device=DEV, generator=g), y


def test_separated_blobs_give_ari_one():
    x, y = _blobs(20000, 32, 8, seed=1)
    km = kmeans_fit(x, 8, restarts=4, seed=3, normalize=False)
    pred, _ = km.predict(x)
    m = clustering_metrics(pred, y, num_clusters=8, num_classes=8)
    assert m["ari"] == 1.0 and m["oa_hungarian"] == 1.0 and abs(m["nmi"] - 1.0) < 1e-12, m
    assert bool(km.converged[km.best])


def _lloyd64(y64, c64, iters):
    """float64 Lloyd from c64 [K, D]: -> labels of every iteration (empty clusters keep their centroid)."""
    out = []
    for _ in range(iters):
        lab = _d64(y64, c64).argmin(1)
        out.append(lab)
        cnt = torch.bincount(lab, minlength=c64.shape[0])
        s = torch.zeros_like(c64).index_add_(0, lab, y64)
        c64 = torch.where(cnt[:, None] > 0, s / cnt[:, None].clamp_min(1), c64)
    return out


@pytest.mark.parametrize("normalize", [False, True])
def test_fit_follows_fp64_lloyd_every_iteration(normalize):
    """Started from one row of each of 12 blobs (so no cluster boundary runs through a blob, where fp32 and float64 could part on a
    near-equidistant row), the kernel's labels equal float64 Lloyd's at every iteration."""
    x, y = _blobs(30000, 96, 12, seed=2, sep=1.5)
    K, R, iters = 12, 2, 8
    g = torch.Generator(device=DEV).manual_seed(5)
    init = torch.stack([x[torch.stack([torch.nonzero(y == k)[torch.randint(0, int((y == k).sum()), (1,), device=DEV, generator=g)][0, 0]
                                       for k in torch.randperm(K, device=DEV, generator=g).tolist()])] for _ in range(R)])
    if normalize:
        init = F.normalize(init, dim=2)
    init = init.contiguous()
    dims = _kmeans_dims(x.shape[0], 96, K, R, normalize)
    ws = _workspace(dims)
    cent = init.clone()
    labels = torch.full((R, x.shape[0]), -1, device=DEV, dtype=torch.int64)
    inertia, changed, empty = (torch.empty(R, device=DEV, dtype=t) for t in (torch.float64, torch.int32, torch.int32))
    y64 = _rows64(x, normalize)
    want = [_lloyd64(y64, init[r].double(), iters) for r in range(R)]
    for it in range(iters):
        _kmeans_assign(dims, x, cent, labels, workspace=ws)
        _kmeans_update(dims, ws, cent, inertia, changed, empty)
        for r in range(R):
            assert torch.equal(labels[r], want[r][it]), (r, it, int((labels[r] != want[r][it]).sum()))
    km = kmeans_fit(x, K, restarts=R, iters=iters, normalize=normalize, init=init)
    assert torch.equal(km.centroids, cent)                                       # a converged restart stays at its fixed point
    assert torch.equal(km.inertia, inertia.cpu()) and bool(km.converged.all()) and bool((km.iterations <= iters).all())


def test_fits_are_bitwise_reproducible_and_restarts_independent():
    x, _ = _blobs(12000, 96, 20, seed=3, sep=0.7)
    kw = dict(iters=30, seed=11)
    a = kmeans_fit(x, 20, restarts=4, **kw)
    b = kmeans_fit(x, 20, restarts=4, **kw)
    assert torch.equal(a.centroids, b.centroids) and torch.equal(a.inertia, b.inertia) and torch.equal(a.iterations, b.iterations)
    assert torch.equal(a.seed_index, b.seed_index)
    q = torch.randn(3000, 96, device=DEV)
    for r in range(4):
        alone = kmeans_fit(x, 20, restarts=1, iters=30, seed=11 + r)
        assert torch.equal(alone.centroids[0], a.centroids[r]) and torch.equal(alone.inertia[0], a.inertia[r]), r
        assert torch.equal(alone.seed_index[0], a.seed_index[r]) and torch.equal(alone.iterations[0], a.iterations[r])
        la, da = a.predict(x, restart=r)
        lb, db = alone.predict(x)
        assert torch.equal(la, lb) and torch.equal(da, db)
    assert a.best == int(torch.argmin(a.inertia))
    l0, d0 = a.predict(q)
    for bq in (1, 7, 3000):
        n = 200 if bq == 1 else 3000
        l, d = a.predict(q[:n], batch_queries=bq)
        assert torch.equal(l, l0[:n]) and torch.equal(d, d0[:n]), bq
    u = _kmeans_uniforms(11, 4, 20, x.device)
    for r in range(4):
        g = torch.Generator(device=DEV).manual_seed(11 + r)
        assert torch.equal(u[r], torch.rand(20, generator=g, device=DEV, dtype=torch.float64))


def test_empty_cluster_keeps_its_centroid_in_a_fit():
    x, _ = _blobs(5000, 32, 4, seed=6)
    init = torch.cat([x[:4], torch.full((1, 32), 1e3, device=DEV)])[None].contiguous()   # centroid 4 far from every row: always empty
    km = kmeans_fit(x, 5, init=init, normalize=False)
    assert torch.equal(km.centroids[0, 4], init[0, 4])
    labels, _ = km.predict(x)
    assert int((labels == 4).sum()) == 0


def _scene(case):
    m, spec, sd = _model(O.HOUSTON, 2, 81)
    cube = torch.from_numpy(np.random.default_rng(7).standard_normal((1, spec.channels, 19, 22)).astype(np.float32))
    model = M.SimMIMSpatialSpectral(encoder=m, masking_ratio=0.5).to(DEV) if case == "simmim" else m
    return model, spec, sd, cube


@pytest.mark.parametrize("case", ["vit", "simmim"])
def test_cluster_scene_vs_oracle(case):
    """The kernel's clusters and centroids against the float64 scene-embedding oracle: the assignment with the fit's centroids, the
    centroids as float64 means of the oracle features of their clusters, and a fit from the best restart's k-means++ rows against a
    float64 Lloyd on the oracle features from the same rows (labels and centroids at convergence)."""
    model, spec, sd, cube = _scene(case)
    B, _, H, W = cube.shape
    K = 5
    clusters, km = cluster_scene(model, cube.to(DEV), num_clusters=K, restarts=3, seed=4, stride=3)
    assert clusters.shape == (B, H, W) and km.centroids.shape == (3, K, spec.dim)
    assert bool(km.converged[km.best])
    feats = torch.from_numpy(_oracle_embed(cube, sd, spec, 3, None)).to(DEV)       # float64 [B, D, H, W]
    y64 = F.normalize(feats.permute(0, 2, 3, 1).reshape(B * H * W, -1), dim=1)
    c = km.centroids[km.best]
    d64 = _d64(y64, c)
    top2 = torch.topk(d64, 2, 1, largest=False).values
    clear = top2[:, 1] - top2[:, 0] > 1e-6
    lab = clusters.reshape(-1)
    assert torch.equal(lab[clear], d64.argmin(1)[clear]) and float(clear.double().mean()) >= 0.99
    for k in range(K):
        sel = lab == k
        assert bool(sel.any())
        _note(f"scene centroid abs ({case})", float((c[k].double() - y64[sel].mean(0)).abs().max()))
        assert (c[k].double() - y64[sel].mean(0)).abs().max().item() <= 1e-5
    rows = km.seed_index[km.best].to(DEV)
    flat = _pixel_rows(embed_scene(model, cube.to(DEV), stride=3))
    again = kmeans_fit(flat, K, init=F.normalize(flat[rows], dim=1)[None].contiguous())
    assert bool(again.converged[0])
    lab_k, _ = again.predict(flat)
    c64 = y64[rows]
    for _ in range(100):                                                         # float64 Lloyd to its fixed point
        lab64 = _d64(y64, c64).argmin(1)
        cnt = torch.bincount(lab64, minlength=K)
        nxt = torch.where(cnt[:, None] > 0, torch.zeros_like(c64).index_add_(0, lab64, y64) / cnt[:, None].clamp_min(1), c64)
        if torch.equal(_d64(y64, nxt).argmin(1), lab64):
            c64 = nxt
            break
        c64 = nxt
    assert torch.equal(lab_k, lab64), int((lab_k != lab64).sum())
    _note(f"scene lloyd centroid abs ({case})", float((again.centroids[0].double() - c64).abs().max()))
    assert (again.centroids[0].double() - c64).abs().max().item() <= 1e-5


def test_cluster_scene_separable_classes_score_oa_one():
    """Four 16 x 16 class quadrants, one spectrum each, tiled by 8 x 8 windows.  A pixel's feature depends on its class and its place in
    the window; the class partition is the least-inertia one (float64 Lloyd from k-means++ seeds reaches it from about 4 seeds in 5),
    so the best of 8 restarts recovers the classes."""
    m, spec, sd = _model(O.HOUSTON, 2, 81)
    B, H, W = 1, 32, 32
    g = torch.Generator().manual_seed(8)
    truth = torch.zeros(B, H, W, dtype=torch.int64)
    truth[:, :16, 16:] = 1
    truth[:, 16:, :16] = 2
    truth[:, 16:, 16:] = 3
    cube = (3.0 * torch.randn(4, spec.channels, generator=g))[truth].permute(0, 3, 1, 2).contiguous()
    clusters, km = cluster_scene(m, cube.to(DEV), num_clusters=4, restarts=8, stride=8)
    met = clustering_metrics(clusters, truth.to(DEV), num_clusters=4, num_classes=4)
    assert met["oa_hungarian"] == 1.0 and met["ari"] == 1.0 and met["oa_majority"] == 1.0, met
    conf = M.inference.confusion_matrix(met["hungarian_map"].to(DEV)[clusters], truth.to(DEV), 4)
    assert M.inference.classification_metrics(conf)["kappa"] == 1.0
    assert bool(km.converged[km.best])


def test_c_abi_limits_leave_outputs_untouched():
    L = _lib.lib()
    n, D = 300, 96
    x = torch.randn(n, D, device=DEV)
    u = torch.full((16, 256), 0.5, device=DEV, dtype=torch.float64)
    cent = torch.full((16, 256 * 256), 7.0, device=DEV)
    index = torch.full((16, 256), 7, device=DEV, dtype=torch.int64)
    md = torch.full((16, n), 7.0, device=DEV)
    labels = torch.full((16, n), 7, device=DEV, dtype=torch.int64)
    dist = torch.full((16, n), 7.0, device=DEV)
    ws = torch.full((1 << 24,), 7, device=DEV, dtype=torch.uint8)
    inertia = torch.full((16,), 7.0, device=DEV, dtype=torch.float64)
    ch = torch.full((16,), 7, device=DEV, dtype=torch.int32)
    em = ch.clone()
    st = None
    bad = [(dict(dim=80), b"dim=80"), (dict(k=0), b"k=0"), (dict(k=257), b"k=257"), (dict(k=171), b"k*dim"), (dict(restarts=17), b"restarts"),
           (dict(normalize=3), b"normalize"), (dict(n=0), b"n=0"), (dict(n=2 ** 31), b"n=2147483648"), (dict(k=301), b"k=301")]
    for kw, what in bad:
        d = dict(n=n, dim=D, k=20, restarts=2, normalize=1)
        d.update(kw)
        d = _lib.KmeansDims(d["n"], d["dim"], d["k"], d["restarts"], d["normalize"])
        assert L.msst_kmeans_seed(ctypes.byref(d), 0, x.data_ptr(), u.data_ptr(), cent.data_ptr(), index.data_ptr(), md.data_ptr(),
                                  ws.data_ptr(), st) == 1
        assert what in L.msst_last_error(), (kw, L.msst_last_error())
        assert L.msst_kmeans_assign(ctypes.byref(d), x.data_ptr(), cent.data_ptr(), labels.data_ptr(), dist.data_ptr(), ws.data_ptr(), st) == 1
        assert L.msst_kmeans_update(ctypes.byref(d), ws.data_ptr(), cent.data_ptr(), inertia.data_ptr(), ch.data_ptr(), em.data_ptr(), st) == 1
    d = _lib.KmeansDims(n, D, 20, 2, 1)
    assert L.msst_kmeans_seed(ctypes.byref(d), 20, x.data_ptr(), u.data_ptr(), cent.data_ptr(), index.data_ptr(), md.data_ptr(),
                              ws.data_ptr(), st) == 1
    assert L.msst_kmeans_seed(ctypes.byref(d), 0, x.data_ptr(), None, cent.data_ptr(), index.data_ptr(), md.data_ptr(), ws.data_ptr(), st) == 1
    assert L.msst_kmeans_assign(ctypes.byref(d), x.data_ptr(), cent.data_ptr(), None, dist.data_ptr(), ws.data_ptr(), st) == 1
    assert L.msst_kmeans_update(ctypes.byref(d), ws.data_ptr(), cent.data_ptr(), inertia.data_ptr(), None, em.data_ptr(), st) == 1
    torch.cuda.synchronize()
    for t in (cent, index, md, labels, dist, ws, inertia, ch, em):
        assert bool((t == 7).all())
