"""GPU: k-nearest-neighbour probing (maskedsst_b200.inference.knn_neighbors / knn_classify / knn_scene, csrc/knn.cu) against a float64
torch oracle: normalise, q @ r.T, stable sort by (-score, index), weighted vote."""
import ctypes

import numpy as np
import pytest
import torch
import torch.nn.functional as F

import maskedsst_b200 as M
from maskedsst_b200 import _lib
from maskedsst_b200.inference import classification_metrics, confusion_matrix, knn_classify, knn_neighbors, knn_scene
from oracle import maskedsst_oracle as O
from tests.test_gpu_scene_embed import _oracle_embed
from tests.test_gpu_scene_inference import _model

pytestmark = pytest.mark.gpu
DEV = "cuda"
SCORE_TOL = 1e-5     # |kernel score - float64 cosine|
GAP = 1e-4           # index sets are compared where the oracle's k-th and (k+1)-th scores differ by more than this


def _oracle_sims(ref, query):
    r = F.normalize(ref.double().cpu(), dim=1, eps=1e-12)
    q = F.normalize(query.double().cpu(), dim=1, eps=1e-12)
    return q @ r.T


def _oracle_topk(sims, k):
    """(scores [Q, k + 1], index [Q, k + 1]) ordered by (score descending, index ascending); k + 1 columns where N > k."""
    n = sims.shape[1]
    order = torch.sort(-sims, dim=1, stable=True).indices[:, :min(k + 1, n)]
    return torch.gather(sims, 1, order), order


def _check_selection(scores, index, sims, k):
    want_s, want_i = _oracle_topk(sims, k)
    scores, index = scores.cpu(), index.cpu()
    assert scores.shape == (sims.shape[0], k) and index.shape == (sims.shape[0], k) and index.dtype == torch.int64
    err = (scores.double() - want_s[:, :k]).abs().max().item()
    assert err <= SCORE_TOL, err
    # the returned indices really have the returned scores (to the score tolerance), and each row is ordered
    got = torch.gather(sims, 1, index)
    assert (got - scores.double()).abs().max().item() <= SCORE_TOL
    assert bool((scores[:, 1:] <= scores[:, :-1]).all())
    if want_s.shape[1] > k:
        sep = (want_s[:, k - 1] - want_s[:, k]) > GAP
    else:
        sep = torch.ones(sims.shape[0], dtype=torch.bool)
    same = torch.sort(index, 1).values == torch.sort(want_i[:, :k], 1).values
    assert bool(same[sep].all()), int((~same.all(1) & sep).sum())
    return err


def _data(N, Q, D, seed):
    g = torch.Generator().manual_seed(seed)
    return torch.randn(N, D, generator=g), torch.randn(Q, D, generator=g)


@pytest.mark.parametrize("D", [32, 96, 128, 256])
@pytest.mark.parametrize("k", [1, 5, 20, 64])
@pytest.mark.parametrize("N", ["k", 127, 129, 4099, 100003])
def test_selection_vs_fp64(D, k, N):
    N = k if N == "k" else N
    Q = 300 if N < 10000 else 131
    ref, query = _data(N, Q, D, seed=D * 1000 + k * 7 + N)
    scores, index = knn_neighbors(ref.to(DEV), query.to(DEV), k)
    err = _check_selection(scores, index, _oracle_sims(ref, query), k)
    print(f"D={D} k={k} N={N}: max score error {err:.2e}")


def test_duplicated_references_come_back_in_ascending_index_order():
    D, k = 96, 8
    g = torch.Generator().manual_seed(3)
    base = torch.randn(50, D, generator=g)
    ref = base.repeat(4, 1)                      # row r and r + 50, r + 100, r + 150 are identical
    query = base[:7] + 1e-3 * torch.randn(7, D, generator=g)
    scores, index = knn_neighbors(ref.to(DEV), query.to(DEV), k)
    _check_selection(scores, index, _oracle_sims(ref, query), k)
    scores, index = scores.cpu(), index.cpu()
    for q in range(7):
        for j in range(k - 1):
            if scores[q, j] == scores[q, j + 1]:
                assert index[q, j] < index[q, j + 1], (q, index[q])
        assert index[q, 0] == q and index[q, 1] == q + 50 and index[q, 2] == q + 100 and index[q, 3] == q + 150, index[q]


@pytest.mark.parametrize("k", [1, 20, 64])
def test_all_identical_references_return_the_first_k(k):
    ref = torch.randn(1, 64).repeat(1000, 1)
    query = torch.randn(33, 64)
    scores, index = knn_neighbors(ref.to(DEV), query.to(DEV), k)
    assert torch.equal(index.cpu(), torch.arange(k).expand(33, k))
    assert bool((scores == scores[:, :1]).all())


def test_zero_vectors_follow_the_eps_rule():
    ref, query = _data(300, 40, 64, seed=9)
    ref[5] = 0
    query[3] = 0
    scores, index = knn_neighbors(ref.to(DEV), query.to(DEV), 10)
    assert bool(torch.isfinite(scores).all())
    assert torch.equal(scores[3].cpu(), torch.zeros(10)) and torch.equal(index[3].cpu(), torch.arange(10))   # all ties at 0
    _check_selection(scores, index, _oracle_sims(ref, query), 10)


@pytest.mark.parametrize("D", [32, 256])
def test_near_duplicates_keep_fp32_accurate_scores(D):
    """Adjacent pixels of overlapping windows: references 1e-4 .. 1e-6 apart.  bf16-rounded scores (error ~2^-9) fail here."""
    g = torch.Generator().manual_seed(D)
    centre = torch.randn(4, D, generator=g)
    eps = torch.tensor([1e-4, 3e-5, 1e-5, 3e-6, 1e-6]).repeat_interleave(40)
    ref = (centre.repeat_interleave(200, 0) + eps.repeat(4)[:, None] * torch.randn(800, D, generator=g))
    query = centre + 1e-5 * torch.randn(4, D, generator=g)
    for k in (20, 64):
        scores, index = knn_neighbors(ref.to(DEV), query.to(DEV), k)
        err = _check_selection(scores, index, _oracle_sims(ref, query), k)
        print(f"D={D} k={k}: near-duplicate max score error {err:.2e}")


def test_scores_track_fp64_far_below_bf16_resolution():
    """Self-similarity of unit vectors: every score must be within 2e-6 of float64 (bf16 products alone are off by ~4e-3)."""
    ref, _ = _data(2000, 1, 256, seed=11)
    scores, index = knn_neighbors(ref.to(DEV), ref[:500].to(DEV), 5)
    sims = _oracle_sims(ref, ref[:500])
    err = (scores.cpu().double() - _oracle_topk(sims, 5)[0][:, :5]).abs().max().item()
    assert err <= 2e-6, err
    assert torch.equal(index[:, 0].cpu(), torch.arange(500))


def test_results_bitwise_independent_of_query_chunking_and_runs():
    ref, query = _data(5000, 2500, 96, seed=13)
    ref, query = ref.to(DEV), query.to(DEV)
    s0, i0 = knn_neighbors(ref, query, 20)
    s_again, i_again = knn_neighbors(ref, query, 20)
    assert torch.equal(s0, s_again) and torch.equal(i0, i_again)
    for bq in (1, 1000, 2500):
        s, i = knn_neighbors(ref, query[:300] if bq == 1 else query, 20, batch_queries=bq)
        n = s.shape[0]
        assert torch.equal(s, s0[:n]) and torch.equal(i, i0[:n]), bq
    # a query's result does not depend on the other queries of its chunk or its row inside the 128-query tile
    s, i = knn_neighbors(ref, query[77:1077].flip(0), 20)
    assert torch.equal(s.flip(0), s0[77:1077]) and torch.equal(i.flip(0), i0[77:1077])


def _votes64(scores, index, labels, nc, T):
    s = scores.double().cpu()
    w = torch.exp((s - s[:, :1]) / T) if T != float("inf") else torch.ones_like(s)
    lab = labels.cpu()[index.cpu()]
    p = torch.zeros(s.shape[0], nc, dtype=torch.float64).scatter_add_(1, lab, w)
    return p / w.sum(1, keepdim=True)


def _pred_where_clear(probs64, pred):
    top2 = torch.topk(probs64, min(2, probs64.shape[1]), dim=1)
    clear = (top2.values[:, 0] - top2.values[:, -1] > 1e-4) if probs64.shape[1] > 1 else torch.ones(probs64.shape[0], dtype=torch.bool)
    assert torch.equal(pred.cpu()[clear], top2.indices[:, 0][clear])


@pytest.mark.parametrize("nc", [1, 2, 20, 256])
@pytest.mark.parametrize("T", [0.07, 1.0, float("inf")])
def test_votes_vs_fp64(nc, T):
    N, Q, D, k = 3000, 700, 96, 20
    ref, query = _data(N, Q, D, seed=nc * 13 + int(T * 100 if T < 10 else 999))
    labels = torch.randint(0, nc, (N,), generator=torch.Generator().manual_seed(nc))
    probs, pred = knn_classify(ref.to(DEV), labels.to(DEV), query.to(DEV), num_classes=nc, k=k, temperature=T)
    assert probs.shape == (Q, nc) and pred.shape == (Q,) and pred.dtype == torch.int64
    scores, index = knn_neighbors(ref.to(DEV), query.to(DEV), k)
    own = _votes64(scores, index, labels, nc, T)
    assert (probs.cpu().double() - own).abs().max().item() <= 1e-6
    _pred_where_clear(own, pred)
    # against the full oracle on the queries whose k-th neighbour is separated from the (k+1)-th
    sims = _oracle_sims(ref, query)
    ws, wi = _oracle_topk(sims, k)
    sep = (ws[:, k - 1] - ws[:, k]) > GAP
    full = _votes64(ws[:, :k], wi[:, :k], labels, nc, T)
    assert (probs.cpu().double() - full)[sep].abs().max().item() <= 1e-4
    _pred_where_clear(full[sep], pred[sep.to(DEV)])


def test_vote_keeps_exp_in_range_at_small_temperature():
    """exp(s / T) overflows fp32 at T = 0.005; exp((s - s_0) / T) does not."""
    ref, query = _data(2000, 300, 64, seed=21)
    query = ref[:300] + 0.01 * query                  # top scores close to 1
    labels = torch.randint(0, 5, (2000,), generator=torch.Generator().manual_seed(2))
    probs, pred = knn_classify(ref.to(DEV), labels.to(DEV), query.to(DEV), num_classes=5, k=10, temperature=0.005)
    assert bool(torch.isfinite(probs).all())
    scores, index = knn_neighbors(ref.to(DEV), query.to(DEV), 10)
    assert (probs.cpu().double() - _votes64(scores, index, labels, 5, 0.005)).abs().max().item() <= 1e-6


def _scene_case(case):
    kw = O.HOUSTON
    m, spec, sd = _model(kw, 2, 81)
    cube = torch.from_numpy(np.random.default_rng(7).standard_normal((1, spec.channels, 19, 22)).astype(np.float32))
    model = M.SimMIMSpatialSpectral(encoder=m, masking_ratio=0.5).to(DEV) if case == "simmim" else m
    return model, spec, sd, cube


@pytest.mark.parametrize("case", ["vit", "simmim"])
def test_knn_scene_vs_oracle(case):
    model, spec, sd, cube = _scene_case(case)
    B, _, H, W = cube.shape
    nc = spec.num_classes
    g = torch.Generator().manual_seed(5)
    labels = torch.randint(0, nc, (B, H, W), generator=g)
    labels[torch.rand(B, H, W, generator=g) < 0.6] = -1          # 40 % labelled training pixels
    labels[0, 0, :3] = nc + 2                                      # out of range: not a reference
    probs, pred = knn_scene(model, cube.to(DEV), labels.to(DEV), num_classes=nc, k=10, temperature=0.07, stride=3)
    assert probs.shape == (B, nc, H, W) and pred.shape == (B, H, W)
    feats = torch.from_numpy(_oracle_embed(cube, sd, spec, 3, None))       # float64 [B, D, H, W]
    flat = feats.permute(0, 2, 3, 1).reshape(B * H * W, -1)
    lab = labels.reshape(-1)
    valid = (lab >= 0) & (lab < nc)
    sims = _oracle_sims(flat[valid], flat)
    ws, wi = _oracle_topk(sims, 10)
    sep = (ws[:, 9] - ws[:, 10]) > GAP
    full = _votes64(ws[:, :10], wi[:, :10], lab[valid], nc, 0.07)
    got = probs.permute(0, 2, 3, 1).reshape(B * H * W, nc).cpu().double()
    err = (got - full)[sep].abs().max().item()
    print(f"{case}: {int(sep.sum())} of {sep.numel()} pixels separated, max prob error {err:.2e}")
    assert sep.float().mean() > 0.5 and err <= 1e-4
    _pred_where_clear(full[sep], pred.reshape(-1)[sep.to(DEV)])


def test_knn_scene_separable_clusters_score_oa_one():
    """Four 16 x 16 class quadrants, one spectrum each, tiled by 8 x 8 windows: every window lies inside one class, so a held-out
    window's pixels have exact feature copies in the labelled windows of their class (and features of other classes are far)."""
    m, spec, sd = _model(O.HOUSTON, 2, 81)
    B, H, W = 1, 32, 32
    g = torch.Generator().manual_seed(8)
    truth = torch.zeros(B, H, W, dtype=torch.int64)
    truth[:, :16, 16:] = 1
    truth[:, 16:, :16] = 2
    truth[:, 16:, 16:] = 3
    spectra = 3.0 * torch.randn(4, spec.channels, generator=g)
    cube = spectra[truth].permute(0, 3, 1, 2).contiguous()
    labelled = torch.zeros(B, H, W, dtype=torch.bool)
    for y in (0, 16):
        for x in (0, 16):
            labelled[:, y:y + 8, x:x + 8] = True             # top-left and bottom-right window of each quadrant
            labelled[:, y + 8:y + 16, x + 8:x + 16] = True
    train = torch.where(labelled, truth, torch.full_like(truth, -1))
    held_out = torch.where(labelled, torch.full_like(truth, -1), truth)
    probs, pred = knn_scene(m, cube.to(DEV), train.to(DEV), num_classes=4, k=2, stride=8)
    metrics = classification_metrics(confusion_matrix(pred, held_out.to(DEV), 4))
    assert metrics["oa"] == 1.0 and metrics["aa"] == 1.0 and metrics["kappa"] == 1.0, metrics


def _topk_c(dims, ref=1, query=1, scores=1, index=1):
    return _lib.lib().msst_knn_topk(ctypes.byref(dims) if dims is not None else None, ref, query, scores, index, None)


def test_c_abi_limits_leave_outputs_untouched():
    L = _lib.lib()
    ref = torch.zeros(200, 3 * 96, device=DEV, dtype=torch.bfloat16)
    qry = torch.zeros(10, 3 * 96, device=DEV, dtype=torch.bfloat16)
    scores = torch.full((10, 64), 7.0, device=DEV)
    index = torch.full((10, 64), 7, device=DEV, dtype=torch.int64)
    ptrs = dict(ref=ref.data_ptr(), query=qry.data_ptr(), scores=scores.data_ptr(), index=index.data_ptr())
    for (N, Q, D, k), what in [((200, 10, 96, 0), b"k=0"), ((200, 10, 96, 65), b"k=65"), ((19, 10, 96, 20), b"n_ref=19"),
                               ((200, 10, 80, 20), b"dim=80"), ((200, 10, 288, 20), b"dim=288"), ((200, 10, 0, 20), b"dim=0"),
                               ((2 ** 31, 10, 96, 20), b"n_ref="), ((200, 0, 96, 20), b"n_query=0")]:
        assert _topk_c(_lib.KnnDims(N, Q, D, k), **ptrs) == 1, (N, Q, D, k)
        assert what in L.msst_last_error(), L.msst_last_error()
    assert _topk_c(_lib.KnnDims(200, 10, 96, 20), **dict(ptrs, index=None)) == 1 and b"must be set" in L.msst_last_error()
    assert _topk_c(None) == 1 and b"dims" in L.msst_last_error()
    x = torch.full((4, 96), 3.0, device=DEV)
    assert L.msst_knn_prepare(x.data_ptr(), 4, 100, ref.data_ptr(), None) == 1 and b"dim=100" in L.msst_last_error()
    assert L.msst_knn_prepare(None, 4, 96, ref.data_ptr(), None) == 1 and b"must be set" in L.msst_last_error()
    probs = torch.full((10, 256), 7.0, device=DEV)
    pred = torch.full((10,), 7, device=DEV, dtype=torch.int64)
    labels = torch.zeros(200, device=DEV, dtype=torch.int64)
    vote = lambda k=20, n_ref=200, nc=5, T=0.07, lab=labels.data_ptr(): L.msst_knn_vote(10, k, n_ref, scores.data_ptr(), index.data_ptr(),
                                                                                       lab, nc, T, probs.data_ptr(), pred.data_ptr(), None)
    for kw, what in [(dict(nc=0), b"nc=0"), (dict(nc=257), b"nc=257"), (dict(k=65), b"k=65"), (dict(k=0), b"k=0"), (dict(n_ref=19), b"n_ref=19"),
                     (dict(T=0.0), b"temperature"), (dict(T=-1.0), b"temperature"), (dict(T=float("nan")), b"temperature"),
                     (dict(lab=None), b"must be set")]:
        assert vote(**kw) == 1, kw
        assert what in L.msst_last_error(), (kw, L.msst_last_error())
    torch.cuda.synchronize()
    assert bool((scores == 7).all()) and bool((index == 7).all()) and bool((probs == 7).all()) and bool((pred == 7).all())
    assert bool((ref == 0).all())
