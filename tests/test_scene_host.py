"""CPU: whole-scene inference host logic -- the window grid, the confusion matrix and OA / AA / kappa, and the argument checks of
msst_scene_blend and of the strided raw-input reader, which run before any CUDA call."""
import ctypes as C

import numpy as np
import pytest
import torch

from maskedsst_b200 import _lib
from maskedsst_b200.inference import classification_metrics, confusion_matrix, scene_windows


def _origins(extent, win, step, n):
    return np.minimum(np.arange(n) * step, extent - win)   # the origin rule of csrc/pixel_source.cuh (window_origin)


@pytest.mark.parametrize("H,W,win,stride", [(601, 2384, 8, 8), (601, 2384, 8, (4, 2)), (21, 19, 8, 3), (8, 8, 8, 1),
                                            (1024, 1024, 8, 8), (9, 15, 8, 8), (100, 37, 8, 5)])
def test_scene_windows_cover_every_pixel_flush_with_the_border(H, W, win, stride):
    ny, nx = scene_windows(H, W, win, stride)
    sy, sx = (stride, stride) if isinstance(stride, int) else stride
    for extent, n, step in ((H, ny, sy), (W, nx, sx)):
        o = _origins(extent, win, step, n)
        cov = np.zeros(extent, dtype=int)
        for a in o:
            cov[a:a + win] += 1
        assert (cov > 0).all()
        assert o[-1] + win == extent                       # the last window ends on the border
        assert (np.diff(o) > 0).all()                      # no duplicate window
        assert (np.diff(o)[:-1] == step).all()             # only the last step may be shortened by the snap
        assert n == 1 or o[-2] + win < extent              # one window fewer would leave the border uncovered


def test_scene_windows_at_stride_window_is_the_tile_grid():
    for H, W in ((64, 64), (24, 16), (8, 8), (1024, 512)):
        assert scene_windows(H, W, 8, 8) == (H // 8, W // 8)


def test_scene_windows_argument_checks():
    with pytest.raises(ValueError):
        scene_windows(21, 19, 8, 0)
    with pytest.raises(ValueError):
        scene_windows(21, 19, 8, 9)
    with pytest.raises(ValueError):
        scene_windows(7, 19, 8, 4)


def test_confusion_matrix_matches_numpy_with_ignored_and_out_of_range_labels():
    rng = np.random.default_rng(3)
    nc = 6
    labels = rng.integers(-2, nc + 2, (3, 17, 23))         # -1 ignored; -2, nc, nc+1 outside [0, nc)
    pred = rng.integers(0, nc, labels.shape)
    want = np.zeros((nc, nc), dtype=np.int64)
    for t, p in zip(labels.ravel(), pred.ravel()):
        if t != -1 and 0 <= t < nc:
            want[t, p] += 1
    got = confusion_matrix(torch.from_numpy(pred), torch.from_numpy(labels), nc)
    assert got.dtype == torch.int64 and np.array_equal(got.numpy(), want)
    # another ignore index: -1 is then simply out of range, 3 is skipped
    want3 = want.copy()
    want3[3] = 0
    assert np.array_equal(confusion_matrix(torch.from_numpy(pred), torch.from_numpy(labels), nc, ignore_index=3).numpy(), want3)
    with pytest.raises(ValueError):
        confusion_matrix(torch.full((4,), nc), torch.zeros(4, dtype=torch.int64), nc)


def test_oa_aa_kappa_textbook_values():
    # a 4-class accuracy-assessment matrix, rows = true class, columns = predicted class
    conf = np.array([[65, 4, 22, 24], [6, 81, 5, 8], [0, 11, 85, 19], [4, 7, 3, 90]], dtype=np.int64)
    m = classification_metrics(torch.from_numpy(conf))
    n = conf.sum()
    po = np.trace(conf) / n
    pe = (conf.sum(1) * conf.sum(0)).sum() / n ** 2
    assert m["oa"] == pytest.approx(321 / 434, rel=1e-15)
    assert m["oa"] == pytest.approx(po, rel=1e-15)
    assert m["aa"] == pytest.approx(np.mean([65 / 115, 81 / 100, 85 / 115, 90 / 104]), rel=1e-15)
    assert m["kappa"] == pytest.approx((po - pe) / (1 - pe), rel=1e-14)
    assert m["kappa"] == pytest.approx(0.6535, abs=5e-5)
    assert np.allclose(m["per_class_acc"].numpy(), np.diag(conf) / conf.sum(1))
    # perfect map: everything 1; chance-level map (rows proportional to the column totals): kappa 0
    p = classification_metrics(torch.diag(torch.tensor([5, 7, 9])))
    assert p["oa"] == 1.0 and p["aa"] == 1.0 and p["kappa"] == 1.0
    c = classification_metrics(torch.tensor([[2, 2], [2, 2]]))
    assert c["oa"] == 0.5 and c["aa"] == 0.5 and c["kappa"] == pytest.approx(0.0, abs=1e-15)


def test_aa_leaves_out_classes_absent_from_the_labels():
    conf = torch.tensor([[3, 1, 0], [0, 0, 0], [1, 0, 1]])   # class 1 never occurs in the labels (but is predicted once)
    m = classification_metrics(conf)
    assert m["aa"] == pytest.approx((3 / 4 + 1 / 2) / 2)
    assert np.isnan(m["per_class_acc"][1].item())
    assert m["oa"] == pytest.approx(4 / 6)
    assert np.isnan(classification_metrics(torch.tensor([[5, 0], [0, 0]]))["kappa"])   # pe == 1: kappa undefined


def _blend(**kw):
    d = dict(B=1, nc=20, H=21, W=19, win=8, stride_y=3, stride_x=3, win_y=6, win_x=5, win_first=0, n=30)
    d.update(kw)
    dims = _lib.SceneDims(*[d[k] for k, _ in _lib.SceneDims._fields_])
    return _lib.lib().msst_scene_blend(C.byref(dims), 1, None, 1, 1, None)


def test_scene_blend_argument_checks_without_a_device():
    L = _lib.lib()
    for kw, what in [(dict(stride_y=0), b"stride"), (dict(stride_x=0), b"stride"), (dict(stride_y=9), b"stride"),
                     (dict(H=7), b"smaller"), (dict(W=5), b"smaller"), (dict(win_y=7), b"grid"), (dict(win_x=6), b"grid"),
                     (dict(win_first=-1), b"outside"), (dict(n=31), b"outside"), (dict(win_first=29, n=2), b"outside"),
                     (dict(n=0), b"outside"), (dict(nc=257), b"nc"), (dict(B=0), b"bad dims")]:
        assert _blend(**kw) == 1, kw
        assert what in L.msst_last_error(), (kw, L.msst_last_error())


def _embed_raw(**kw):
    """msst_patch_embed_fwd on a Houston-shaped model (50 bands, 8 x 8 windows) reading raw tiles; the pixel reader's checks fail
    before any pointer is touched."""
    r = dict(tiles=1, dtype=_lib.RAW_I16, raw_bands=48, tile_h=21, tile_w=19, y0=0, x0=0, mean=1, std=1, clip=0, clip_lo=0.0,
             clip_hi=0.0, win_y=6, win_x=5, stride_y=3, stride_x=3, win_first=0)
    r.update(kw)
    raw = _lib.RawInput(*[r[k] for k, _ in _lib.RawInput._fields_])
    dims = _lib.EmbedDims(30, 5, 8, 10, 1, 96, 5, 0.0, 0, None, C.pointer(raw))
    return _lib.lib().msst_patch_embed_fwd(C.byref(dims), *([None] * 12), None)


def test_strided_raw_input_argument_checks_without_a_device():
    L = _lib.lib()
    for kw in [dict(stride_y=9), dict(stride_x=9), dict(stride_y=-1), dict(win_first=-1), dict(tile_h=7), dict(tile_w=7),
               dict(y0=14), dict(x0=12)]:
        assert _embed_raw(**kw) == 1, kw
        assert b"raw input" in L.msst_last_error(), kw
