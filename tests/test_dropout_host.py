"""CPU: the dropout-probability checks (p outside [0, 1] or NaN is refused before any launch, in Python and at every C entry
point), and the host mask model of tests/dropout_ref.py against a plain-integer restatement of csrc/common.cuh."""
import ctypes as C
import math

import numpy as np
import pytest
import torch

from maskedsst_b200 import _lib, ops
from maskedsst_b200._lib import PREC_FP32, PREC_BF16
from tests import dropout_ref as R

BAD_P = [float("nan"), -0.1, 1.5]
FAKE = 256   # a non-null pointer that must never be dereferenced: the checks return before any CUDA call


def _c_calls(p):
    L = _lib.lib()
    ad = _lib.AttnDims(4, 64, 1, 2, 64, p, 1, 0, PREC_FP32, None)
    ab = _lib.AttnDims(4, 64, 1, 2, 64, p, 1, 0, PREC_BF16, None)
    ld = _lib.LinearDims(8, 16, 16, 0, p, 1, 3, PREC_FP32, None, 1)
    ed = _lib.EmbedDims(1, 5, 8, 10, 1, 96, 5, p, 1, None, None)
    td = _lib.TfDims(4, 64, 1, 96, 2, 64, 64, 1, p, 1, 16, PREC_FP32, 1, None)
    lp = (_lib.LayerPtrs * 1)(_lib.LayerPtrs(*[FAKE] * 11))
    return {
        "dropout_apply": lambda: L.msst_dropout_apply(FAKE, FAKE, 4, p, 1, 3, None, None),
        "attention": lambda: L.msst_attention_fwd(C.byref(ad), FAKE, FAKE, FAKE, None),
        "attention_bwd": lambda: L.msst_attention_bwd(C.byref(ab), FAKE, FAKE, FAKE, FAKE, FAKE, None),
        "attn_block": lambda: L.msst_attn_block_fwd(C.byref(ab), 96, FAKE, FAKE, FAKE, FAKE, None),
        "linear_fwd": lambda: L.msst_linear_fwd(C.byref(ld), FAKE, FAKE, None, None, FAKE, None, None),
        "linear_bwd_data": lambda: L.msst_linear_bwd_data(C.byref(ld), FAKE, FAKE, FAKE, None, FAKE, None),
        "patch_embed": lambda: L.msst_patch_embed_fwd(C.byref(ed), *[FAKE] * 8, None, None, FAKE, None, None),
        "patch_embed_bwd": lambda: L.msst_patch_embed_bwd(C.byref(ed), *[FAKE] * 7, None, FAKE, None, *[FAKE] * 7, None, None),
        "mlp_block": lambda: L.msst_mlp_block_fwd(*[FAKE] * 9, None, None, None, None, 64, 96, 64, p, 1, 18, 19, None, None),
        "mlp_block_bwd": lambda: L.msst_mlp_block_bwd(*[FAKE] * 10, 64, 96, 64, p, 1, 18, None, None),
        "transformer": lambda: L.msst_transformer_fwd(C.byref(td), lp, FAKE, FAKE, FAKE, None),
        "workspace": lambda: L.msst_transformer_workspace_bytes(C.byref(td)),
    }


@pytest.mark.parametrize("p", BAD_P)
def test_c_entry_points_reject_bad_dropout_probability(p):
    for name, call in _c_calls(p).items():
        rc = call()
        if name == "workspace":
            assert rc == -1, name
            continue
        assert rc == 1, (name, rc)
        assert b"outside [0, 1]" in _lib.lib().msst_last_error(), (name, _lib.lib().msst_last_error())


@pytest.mark.parametrize("p", BAD_P)
def test_ops_reject_bad_dropout_probability(p):
    x = torch.zeros(64, 96)
    with pytest.raises(ValueError, match="dropout probability"):
        ops.transformer_stack(x, [[x] * 11], n_seq=1, N=64, inner=1, heads=2, dim_head=64, mlp_dim=64, drop_p=p, seed=1)
    with pytest.raises(ValueError, match="dropout probability"):
        ops.attention(x, n_seq=1, N=64, heads=1, dim_head=32, drop_p=p)
    with pytest.raises(ValueError, match="dropout probability"):
        ops.patch_embed(x, *[x] * 7, geom=(1, 1, 8, 1, 96), drop_p=p, seed=1)


def _bits_int(seed, site, q):
    M = 0xFFFFFFFF

    def mix(x):
        x ^= x >> 16; x = (x * 0x7FEB352D) & M; x ^= x >> 15; x = (x * 0x846CA68B) & M; x ^= x >> 16
        return x
    x = ((((q & M) + (seed >> 32)) & M) * 0x9E3779B1 & M) ^ (((q >> 32) * 0x85EBCA77) & M) ^ (seed & M) ^ ((site * 0xC2B2AE3D) & M)
    a = mix(x)
    return a, mix((a + 0x9E3779B9) & M)


def test_host_model_matches_integer_restatement():
    for seed in (5, 0xFFFFFFFF, 1 << 32, 0xFFFFFFFFFFFFFFFF):
        for site in (1, 19, 0xFFFFFFF0):
            qs = [0, 1, 77, (1 << 32) + 5, (1 << 40) + 3]
            a, b = R.drop_bits64(seed, site, np.array(qs, dtype=np.uint64))
            assert [(int(x), int(y)) for x, y in zip(a, b)] == [_bits_int(seed, site, q) for q in qs]
    # element convention: quad e >> 2, word a / b by e & 2, low / high half by e & 1
    p, seed, site, n = 0.5, 123, 17, 1001
    t16 = R.drop_params(p)[0] >> 16
    want = []
    for e in range(n):
        a, b = _bits_int(seed, site, e >> 2)
        w = b if e & 2 else a
        want.append(2.0 if ((w >> 16) if e & 1 else (w & 0xFFFF)) >= t16 else 0.0)
    assert np.array_equal(R.elem_mask(p, seed, site, n), np.array(want, dtype=np.float32))


def test_make_drop_edges():
    assert R.drop_params(0.0) == (0, 1.0)
    assert R.drop_params(1.0) == (0xFFFFFFFF, 0.0)                     # p = 1: every factor 0, never inf
    assert R.drop_params(2.0 ** -40)[0] == 1                            # thresh 0 would disable dropout: clamped to 1
    assert R.drop_params(2.0 ** -17)[0] >> 16 == 0                      # below 2^-16 nothing is dropped ...
    assert R.drop_params(2.0 ** -17)[1] == np.float32(1) / np.float32(1 - 2.0 ** -17)   # ... but it still scales
    assert not (R.elem_mask(1.0, 3, 4, 1 << 18) != 0).any()
    m = R.elem_mask(0.1, 3, 4, 1 << 20)
    assert abs((m != 0).mean() - 0.9) < 3e-3 and math.isclose(float(m.max()), 1 / 0.9, rel_tol=1e-6)


def test_attention_pair_masks_are_consistent():
    """N <= 64 packing: a key pair shares one hash word; N > 64: tile indices.  Both give each (seq, h, q, k) one factor and
    the mask of a sequence does not depend on how many sequences follow it."""
    a = R.attn_mask_bf16(0.3, 9, 16, 6, 22, 2, 4)
    b = R.attn_mask_bf16(0.3, 9, 16, 12, 22, 2, 4)
    assert np.array_equal(a, b[:6])
    a = R.attn_mask_bf16(0.3, 9, 16, 2, 130, 1, 2)
    assert a.shape == (2, 2, 130, 130) and abs((a != 0).mean() - 0.7) < 0.01
