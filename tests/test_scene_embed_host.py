"""CPU: the argument checks of msst_scene_embed, which run before any CUDA call."""
import ctypes as C

from maskedsst_b200 import _lib


def _embed(**kw):
    d = dict(B=1, D=96, H=21, W=19, win=8, stride_y=3, stride_x=3, win_y=6, win_x=5, win_first=0, n=30, C=5, p1=1)
    d.update(kw)
    dims = _lib.SceneEmbedDims(*[d[k] for k, _ in _lib.SceneEmbedDims._fields_])
    return _lib.lib().msst_scene_embed(C.byref(dims), 1, None, 1, 1, None)


def test_scene_embed_argument_checks_without_a_device():
    L = _lib.lib()
    assert L.msst_version() == 102
    for kw, what in [(dict(p1=3), b"multiple"), (dict(win=12, p1=8, win_y=4, win_x=3), b"multiple"), (dict(D=257), b"D=257"),
                     (dict(D=1024), b"D=1024"), (dict(win_first=-1), b"outside"), (dict(n=31), b"outside"),
                     (dict(win_first=29, n=2), b"outside"), (dict(n=0), b"outside"), (dict(B=2, n=61), b"outside"),
                     (dict(stride_y=0), b"stride"), (dict(stride_x=0), b"stride"), (dict(stride_x=9), b"stride"),
                     (dict(H=7), b"smaller"), (dict(win_y=7), b"grid"), (dict(win_x=6), b"grid"),
                     (dict(B=0), b"bad dims"), (dict(D=0), b"bad dims"), (dict(C=0), b"bad dims"), (dict(p1=0), b"bad dims")]:
        assert _embed(**kw) == 1, kw
        msg = L.msst_last_error()
        assert msg.startswith(b"scene_embed:") and what in msg, (kw, msg)


def test_scene_embed_null_pointers_rejected():
    dims = _lib.SceneEmbedDims(1, 96, 21, 19, 8, 3, 3, 6, 5, 0, 30, 5, 1)
    L = _lib.lib()
    assert L.msst_scene_embed(C.byref(dims), None, None, 1, 1, None) == 1
    assert b"must be set" in L.msst_last_error()
    assert L.msst_scene_embed(None, 1, None, 1, 1, None) == 1
    assert b"bad dims" in L.msst_last_error()
