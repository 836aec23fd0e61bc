"""GPU: every dropout-carrying kernel, the transformer stack and whole training steps with dropout ON, against float64
references that apply the kernels' own masks (rebuilt on the host by tests/dropout_ref.py).

The masks are a pure function of (seed, site, index), so nothing here is statistical: the host model is first pinned to the
device bit for bit (msst_dropout_apply; every attention kernel through a probe that reads its mask back), then each kernel and
step is compared with float64 at the tolerances of the p = 0 parity tests (fp32 1e-5 / 2e-5 or 1e-4 for whole steps; bf16 as in
the neighbouring bf16 files).  A mask at the wrong point (dropped probabilities in the softmax denominator or in lse), a wrong
scale, a site id wired to the wrong layer, a wrong device seed offset, or an indexing error shared by twin kernels all fail."""
import ctypes as C
import os
import subprocess
import sys

import numpy as np
import pytest
import torch

import maskedsst_b200 as M
from maskedsst_b200 import _lib, ops
from maskedsst_b200._lib import check, PREC_FP32, PREC_BF16
from oracle import maskedsst_oracle as O
from tests import dropout_ref as R
from tests.helpers import rel_l2
from tests.test_gpu_kernel_edges import _run_embed
from tests.test_gpu_parity import make_encoder

pytestmark = pytest.mark.gpu
DEV = "cuda"
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _st():
    return torch.cuda.current_stream().cuda_stream


def _t(a):
    return torch.from_numpy(np.ascontiguousarray(a)).double()


def _in_env(env, call):
    """Runs `call` (a Python expression over this module, imported as t) in a fresh process with `env` set: the kernel
    switches are read once per process."""
    code = f"import sys; sys.path.insert(0, '.'); import tests.test_gpu_dropout_exact as t; {call}"
    r = subprocess.run([sys.executable, "-c", code], cwd=ROOT, env=dict(os.environ, **env), capture_output=True, text=True, timeout=1200)
    assert r.returncode == 0, f"{env}: {call}\n{r.stdout[-4000:]}\n{r.stderr[-4000:]}"
    print(r.stdout)


# ---------------------------------------------------------------------------------------------------------------------
# 1. the host model against the device, bit for bit
# ---------------------------------------------------------------------------------------------------------------------
P_EDGE = [0.1, 0.5, 0.9, 2.0 ** -17, 1 - 2.0 ** -17]


@pytest.mark.parametrize("p", P_EDGE)
def test_dropout_apply_equals_host_model(p):
    n = 4 * 12345
    x = torch.ones(n, device=DEV)
    for seed in (7, 0xFFFFFFFF, 1 << 32, 0x9E3779B97F4A7C15):
        for site in (1, 16, 19, 16 + 8 * 7 + 3):
            y = torch.empty_like(x)
            check(_lib.lib().msst_dropout_apply(x.data_ptr(), y.data_ptr(), n, p, seed, site, None, _st()))
            want = R.elem_mask(p, seed, site, n)
            assert np.array_equal(y.cpu().numpy().view(np.uint32), want.view(np.uint32)), (p, seed, site)
    if p == 2.0 ** -17:   # below the 2^-16 resolution: nothing dropped, everything scaled by 1/(1-p)
        assert (want == np.float32(1) / np.float32(1 - p)).all()


def test_dropout_apply_device_seed_offset_and_ragged_n():
    """seed_dev is added to the seed (what a CUDA-graph replay relies on); n % 4 != 0 is refused (the ragged tail of an
    element-indexed site is exercised through the GEMM epilogues at N = 13 below)."""
    n = 4096
    x = torch.ones(n, device=DEV)
    off = torch.tensor(5 + (3 << 32), dtype=torch.int64, device=DEV)
    y = torch.empty_like(x)
    check(_lib.lib().msst_dropout_apply(x.data_ptr(), y.data_ptr(), n, 0.3, 11, 17, off.data_ptr(), _st()))
    assert np.array_equal(y.cpu().numpy(), R.elem_mask(0.3, 11 + 5 + (3 << 32), 17, n))
    assert _lib.lib().msst_dropout_apply(x.data_ptr(), y.data_ptr(), 4095, 0.3, 11, 17, None, _st()) == 1   # MSST_ERR_ARG


# attention geometries (n_seq, N, inner, H): spatial, Houston / EnMAP spectral, ragged packing, long sequences
PROBE_GEOMS = [(3, 64, 1, 8), (128, 5, 64, 8), (128, 20, 64, 8), (6, 22, 2, 4), (3, 65, 1, 2), (2, 130, 1, 2), (4, 200, 2, 2),
               (1, 1000, 1, 2)]


def _rows(n_seq, N, inner):
    seq = torch.arange(n_seq)[:, None]
    return (seq // inner) * N * inner + seq % inner + torch.arange(N)[None, :] * inner   # [n_seq, N]


def probe_attention_mask(n_seq, N, inner, H, prec, p=0.1, seed=0x1234567890AB, site=21):
    """Reads an attention kernel's mask back: Q = 0 makes every probability 1/N, and V = one-hot rows over key block b
    (keys b*64 .. b*64+63) gives O[q, j] = f(q, b*64 + j) / N.  Checks the kept set against the host model exactly and the
    kept values against scale / N."""
    dh, I = 64, H * 64
    Rn = n_seq * N
    dt = torch.bfloat16 if prec == PREC_BF16 else torch.float32
    rows = _rows(n_seq, N, inner)
    want = (R.attn_mask_bf16 if prec == PREC_BF16 else R.attn_mask_f32)(p, seed, site, n_seq, N, inner, H)
    _, scale = R.drop_params(p)
    got = np.zeros_like(want)
    for b in range((N + 63) // 64):
        qkv = torch.zeros(Rn, 3 * I)
        qkv[:, I:2 * I] = torch.randn(Rn, I)                     # K: irrelevant once Q = 0
        pos = torch.arange(N)
        v = torch.zeros(N, dh)
        sel = (pos // 64) == b
        v[pos[sel], pos[sel] % 64] = 1.0
        for h in range(H):
            qkv[rows.reshape(-1), 2 * I + h * dh: 2 * I + (h + 1) * dh] = v.repeat(n_seq, 1)
        qkv = qkv.to(DEV, dt)
        out = torch.full((Rn, I), float("nan"), device=DEV, dtype=dt)
        lse = torch.full((Rn, H), float("nan"), device=DEV)
        dims = _lib.AttnDims(n_seq, N, inner, H, dh, p, seed, site, prec, None)
        check(_lib.lib().msst_attention_fwd(C.byref(dims), qkv.data_ptr(), out.data_ptr(), lse.data_ptr(), _st()))
        o = out.float().cpu()[rows.reshape(-1)].reshape(n_seq, N, H, dh).permute(0, 2, 1, 3).numpy()   # [n_seq, H, q, j]
        kb = pos[sel].numpy()
        got[:, :, :, kb] = o[:, :, :, kb % 64] * N
        assert np.allclose(lse.cpu().numpy(), np.log(N), rtol=0, atol=1e-5)   # the undropped log-sum-exp
    keep_err = int(((got != 0) != (want != 0)).sum())
    assert keep_err == 0, f"{keep_err} of {want.size} mask bits differ ({n_seq}, {N}, {inner}, {H}, prec {prec})"
    kept = want != 0
    tol = 1e-6 if prec == PREC_FP32 else 8e-3
    assert np.allclose(got[kept], scale, rtol=tol, atol=0), float(np.abs(got[kept] / scale - 1).max())
    print(f"probe prec={prec} {(n_seq, N, inner, H)}: {want.size} bits equal")


def probe_all(prec, geoms):
    for g in geoms:
        probe_attention_mask(*g, prec=prec)


def test_attention_mask_probe_fp32():
    probe_all(PREC_FP32, PROBE_GEOMS)


def test_attention_mask_probe_bf16_default():
    """tcgen05 for N <= 64, mma.sync long kernel for 64 < N < 512, tcgen05 long forward from 512."""
    probe_all(PREC_BF16, PROBE_GEOMS)


@pytest.mark.parametrize("env,which", [({"MSST_ATTN_TC": "0"}, "short"),          # mma.sync, N <= 64
                                       ({"MSST_ATTN_TC_LONG": "1"}, "long"),      # tcgen05 long forward at every N > 64
                                       ({"MSST_ATTN_TC_LONG": "0"}, "long")])     # mma.sync long kernel at N = 1000 too
def test_attention_mask_probe_bf16_switched(env, which):
    geoms = [g for g in PROBE_GEOMS if (g[1] <= 64) == (which == "short")]
    _in_env(env, f"t.probe_all(t.PREC_BF16, {geoms!r})")


# ---------------------------------------------------------------------------------------------------------------------
# 2. kernels against float64 with the exact masks
# ---------------------------------------------------------------------------------------------------------------------
def ref_attention_masked(qkv, n_seq, N, inner, H, dh, mask):
    """fp64 softmax(q k^T dh^-0.5) * mask @ v over the strided row layout; also lse of the undropped scores [R, H]."""
    I = H * dh
    rows = _rows(n_seq, N, inner).reshape(-1)
    inv = torch.argsort(rows)
    q, k, v = qkv.double().split(I, dim=-1)
    g = lambda t: t[rows].reshape(n_seq, N, H, dh).permute(0, 2, 1, 3)
    s = g(q) @ g(k).transpose(-1, -2) * dh ** -0.5
    pr = torch.softmax(s, dim=-1)
    if mask is not None:
        pr = pr * mask
    o = (pr @ g(v)).permute(0, 2, 1, 3).reshape(n_seq * N, I)[inv]
    lse = torch.logsumexp(s, dim=-1).permute(0, 2, 1).reshape(n_seq * N, H)[inv]
    return o, lse


def attention_vs_fp64(n_seq, N, inner, H, dh, prec, p, seed=77, site=40):
    torch.manual_seed(N * 7 + H)
    Rn, I = n_seq * N, H * dh
    dt = torch.bfloat16 if prec == PREC_BF16 else torch.float32
    qkv = torch.randn(Rn, 3 * I).to(dt)
    w = torch.randn(Rn, I).to(dt)
    mask = _t((R.attn_mask_bf16 if prec == PREC_BF16 else R.attn_mask_f32)(p, seed, site, n_seq, N, inner, H))
    a = qkv.double().requires_grad_(True)
    want, lse_want = ref_attention_masked(a, n_seq, N, inner, H, dh, mask)
    (want * w.double()).sum().backward()
    dims = _lib.AttnDims(n_seq, N, inner, H, dh, p, seed, site, prec, None)
    qd = qkv.to(DEV)
    out = torch.full((Rn, I), float("nan"), device=DEV, dtype=dt)
    lse = torch.full((Rn, H), float("nan"), device=DEV)
    check(_lib.lib().msst_attention_fwd(C.byref(dims), qd.data_ptr(), out.data_ptr(), lse.data_ptr(), _st()))
    dq = torch.full((Rn, 3 * I), float("nan"), device=DEV, dtype=dt)
    wd = w.to(DEV)
    check(_lib.lib().msst_attention_bwd(C.byref(dims), qd.data_ptr(), out.data_ptr(), lse.data_ptr(), wd.data_ptr(), dq.data_ptr(), _st()))
    torch.cuda.synchronize()
    eo, eg, el = rel_l2(out, want), rel_l2(dq, a.grad), float((lse.cpu().double() - lse_want).abs().max())
    tol = (1e-5, 2e-5, 1e-5) if prec == PREC_FP32 else (6e-3, 1.5e-2, 2e-3)
    print(f"attention prec={prec} {(n_seq, N, inner, H, dh)} p={p}: out {eo:.2e} dqkv {eg:.2e} lse {el:.2e}")
    assert eo < tol[0] and eg < tol[1] and el < tol[2], (eo, eg, el)


ATTN_GEOMS = [(4, 64, 1, 8), (128, 5, 64, 8), (128, 20, 64, 8), (6, 22, 2, 4), (3, 65, 1, 2), (3, 200, 1, 2), (2, 256, 2, 2),
              (1, 1000, 1, 2)]


@pytest.mark.parametrize("dh", [32, 64, 128])
@pytest.mark.parametrize("p", [0.1, 0.3])
def test_attention_fp32_vs_fp64(dh, p):
    for g in ATTN_GEOMS:
        attention_vs_fp64(*g, dh=dh, prec=PREC_FP32, p=p)


def attention_bf16_all(p):
    for g in ATTN_GEOMS:
        attention_vs_fp64(*g, dh=64, prec=PREC_BF16, p=p)


@pytest.mark.parametrize("p", [0.1, 0.3])
def test_attention_bf16_vs_fp64(p):
    attention_bf16_all(p)


@pytest.mark.parametrize("env", [{"MSST_ATTN_TC": "0", "MSST_ATTN_BWD_TC": "0"},       # mma.sync forward and backward
                                 {"MSST_ATTN_TC_LONG": "1", "MSST_ATTN_BWD_TC_LONG": "65"},   # tcgen05 long forward + backward
                                 {"MSST_ATTN_TC_LONG": "0", "MSST_ATTN_BWD_TC_LONG": "0"}])   # mma.sync long kernels only
def test_attention_bf16_switched_vs_fp64(env):
    _in_env(env, "t.attention_bf16_all(0.1); t.attention_bf16_all(0.3)")


def _gelu(x):
    return 0.5 * x * (1.0 + torch.erf(x / 2 ** 0.5))


@pytest.mark.parametrize("prec", [PREC_FP32, PREC_BF16])
@pytest.mark.parametrize("N", [10, 13, 40, 96, 1536])
@pytest.mark.parametrize("p", [0.1, 0.3])
def test_linear_epilogue_dropout(prec, N, p):
    """y = dropout(act(x W^T + b)) + residual with GELU and without, and the act-2 data-gradient epilogue
    dx = (dy W) * GELU'(pre_act) * mask: the ragged drop_factor tail runs at N = 10 / 13."""
    torch.manual_seed(N)
    Mr, K = 77, 96
    bf = prec == PREC_BF16
    dt = torch.bfloat16 if bf else torch.float32
    x, W = torch.randn(Mr, K).to(dt), (torch.randn(N, K) * K ** -0.5).to(dt)
    b, res = torch.randn(N), torch.randn(Mr, N)
    seed, site = 0x5EED0000DEADBEEF, 18
    mask = _t(R.elem_mask(p, seed, site, Mr * N).reshape(Mr, N))
    for act in (0, 1):
        t = x.double() @ W.double().t() + b.double()
        want = (_gelu(t) if act else t) * mask + res.double()
        y = torch.full((Mr, N), float("nan"), device=DEV)
        pre = torch.full((Mr, N), float("nan"), device=DEV, dtype=dt) if act else None
        dims = _lib.LinearDims(Mr, N, K, act, p, seed, site, prec, None, 1)
        xd, Wd, bd, rd = (t.to(DEV) for t in (x, W, b, res))
        check(_lib.lib().msst_linear_fwd(C.byref(dims), xd.data_ptr(), Wd.data_ptr(), bd.data_ptr(), rd.data_ptr(), y.data_ptr(),
                                         None if pre is None else pre.data_ptr(), _st()))
        torch.cuda.synchronize()
        e = rel_l2(y, want)
        assert e < (1e-5 if not bf else 4e-3), (act, e)
    # the act-2 data-gradient epilogue: the backward of g = dropout(gelu(u)) [Mr, N] through the layer that consumed g
    # (W2 [K2, N]): dx = (dy W2) * gelu'(u) * mask + dx_add, same (seed, site) and element index as the forward's hidden output
    K2 = 64
    dy, W2, u = torch.randn(Mr, K2).to(dt), (torch.randn(K2, N) * 0.2).to(dt), torch.randn(Mr, N).to(dt)
    add = torch.randn(Mr, N)
    want = (dy.double() @ W2.double()) * (0.5 * (1 + torch.erf(u.double() / 2 ** 0.5)) + u.double() * torch.exp(-0.5 * u.double() ** 2) / (2 * np.pi) ** 0.5) * mask + add.double()
    dx = torch.full((Mr, N), float("nan"), device=DEV)
    dims = _lib.LinearDims(Mr, K2, N, 0, p, seed, site, prec, None, 1)    # dx[M, K] = dy[M, N] . W ; here "N" = K2, "K" = N
    Wt = (W2.t().contiguous() if bf else W2).to(DEV)     # bf16 mode takes the transposed copy W2^T [N, K2]
    dyd, ud, addd = dy.to(DEV), u.to(DEV), add.to(DEV)
    check(_lib.lib().msst_linear_bwd_data(C.byref(dims), dyd.data_ptr(), Wt.data_ptr(), ud.data_ptr(), addd.data_ptr(), dx.data_ptr(),
                                          _st()))
    torch.cuda.synchronize()
    e = rel_l2(dx, want)
    assert e < (2e-5 if not bf else 8e-3), e


@pytest.mark.parametrize("D,p0,p1", [(32, 10, 1), (96, 10, 1), (32, 4, 2), (96, 4, 2)])
@pytest.mark.parametrize("p", [0.1, 0.3])
def test_patch_embed_emb_dropout(D, p0, p1, p):
    """msst_patch_embed_fwd / _bwd with emb-dropout (site 1) at P = 10 / 16, against float64 with the host mask; gradients
    accumulate into non-zero buffers.  B = 30 with 20 blocks makes each backward CTA loop over 2-3 samples."""
    _run_embed(B=3, C_=3, G=8 // p1, p0=p0, p1=p1, D=D, nwb=3, mask_mode="some", with_ln=False, drop_p=p, seed=0xABCDEF0123)
    _run_embed(B=30, C_=20, G=9, p0=p0, p1=p1, D=D, nwb=20, mask_mode="none", with_ln=False, drop_p=p, seed=(1 << 40) + 3)


# ---------------------------------------------------------------------------------------------------------------------
# 3. the transformer stack, depth 2: site = base + 8 * layer + k in both precisions and every kernel configuration
# ---------------------------------------------------------------------------------------------------------------------
def ref_stack(x, layers, n_seq, N, inner, H, dh, p, seed, bf16, base=16):
    """fp64 restatement of the stack over rows [R, D] with the kernels' masks."""
    Rn, D = x.shape
    amask = R.attn_mask_bf16 if bf16 else R.attn_mask_f32
    em = lambda site, w: _t(R.elem_mask(p, seed, site, Rn * w).reshape(Rn, w))
    for l, (l1w, l1b, wqkv, wo, bo, l2w, l2b, w1, b1, w2, b2) in enumerate(layers):
        site = base + 8 * l
        h = torch.nn.functional.layer_norm(x, (D,), l1w, l1b)
        o, _ = ref_attention_masked(h @ wqkv.t(), n_seq, N, inner, H, dh, _t(amask(p, seed, site, n_seq, N, inner, H)))
        xm = x + (o @ wo.t() + bo) * em(site + 1, D)
        h2 = torch.nn.functional.layer_norm(xm, (D,), l2w, l2b)
        g = _gelu(h2 @ w1.t() + b1) * em(site + 2, w1.shape[0])
        x = xm + (g @ w2.t() + b2) * em(site + 3, D)
    return x


def stack_vs_fp64(prec, D=96, n_seq=6, N=64, inner=1, Mh=64, p=0.1, seed=0x0123456789ABCDEF):
    torch.manual_seed(D + N)
    H, dh, L = 2, 64, 2
    Rn, I = n_seq * N, H * dh
    mk = lambda *s, sc=1.0: torch.randn(*s) * sc
    layers = [[1 + 0.1 * mk(D), 0.1 * mk(D), mk(3 * I, D, sc=D ** -0.5), mk(D, I, sc=I ** -0.5), 0.1 * mk(D), 1 + 0.1 * mk(D),
               0.1 * mk(D), mk(Mh, D, sc=D ** -0.5), 0.1 * mk(Mh), mk(D, Mh, sc=Mh ** -0.5), 0.1 * mk(D)] for _ in range(L)]
    x = torch.randn(Rn, D)
    wgt = torch.randn(Rn, D)
    ref = [[t.double().requires_grad_(True) for t in lp] for lp in layers]
    xr = x.double().requires_grad_(True)
    want = ref_stack(xr, ref, n_seq, N, inner, H, dh, p, seed, prec == PREC_BF16)
    (want * wgt.double()).sum().backward()
    dev = [[t.to(DEV).requires_grad_(True) for t in lp] for lp in layers]
    xd = x.to(DEV).requires_grad_(True)
    got = ops.transformer_stack(xd, dev, n_seq=n_seq, N=N, inner=inner, heads=H, dim_head=dh, mlp_dim=Mh, drop_p=p, seed=seed,
                                prec=prec)
    (got * wgt.to(DEV)).sum().backward()
    torch.cuda.synchronize()
    tol = (1e-5, 1e-4) if prec == PREC_FP32 else (1e-2, 5e-2)
    errs = {"y": rel_l2(got, want), "dx": rel_l2(xd.grad, xr.grad)}
    for l in range(L):
        for k, name in enumerate(ops._LAYER_FIELDS):
            errs[f"{l}.{name}"] = rel_l2(dev[l][k].grad, ref[l][k].grad)
    worst = max(errs.values())
    print(f"stack prec={prec} D={D} geom={(n_seq, N, inner)} M={Mh} {os.environ.get('MSST_CFG', '')}: worst {worst:.2e} "
          f"({max(errs, key=errs.get)})")
    assert errs["y"] < tol[0], errs
    bad = {k: v for k, v in errs.items() if k != "y" and v >= tol[1]}
    assert not bad, bad


def stack_all(prec):
    stack_vs_fp64(prec)                                      # spatial geometry
    stack_vs_fp64(prec, n_seq=40, N=5, inner=8)             # packed spectral geometry
    stack_vs_fp64(prec, n_seq=3, N=130, inner=1)            # long sequences
    stack_vs_fp64(prec, D=64, Mh=128)                       # unfused FeedForward (mlp_dim != 64)
    stack_vs_fp64(prec, D=192)                               # D > 128: cast_rows second pass with its dropout
    stack_vs_fp64(prec, p=0.3, n_seq=24, N=20, inner=4)


@pytest.mark.parametrize("prec", [PREC_FP32, PREC_BF16])
def test_transformer_stack_vs_fp64(prec):
    stack_all(prec)


@pytest.mark.parametrize("env", [{"MSST_ATTN_FUSED": "0"}, {"MSST_MLP_FUSED": "0"}, {"MSST_ATTN_OUT_FUSED": "0"},
                                 {"MSST_GEMM_LNB": "1"}, {"MSST_GEMM_LNB": "1", "MSST_ATTN_FUSED": "0"}])
def test_transformer_stack_bf16_switched_vs_fp64(env):
    _in_env(dict(env, MSST_CFG=str(env)), "t.stack_all(t.PREC_BF16)")


# ---------------------------------------------------------------------------------------------------------------------
# 4. whole training steps against the oracle with the same masks
# ---------------------------------------------------------------------------------------------------------------------
class SeedRecorder:
    """Replaces ops.next_seed by a deterministic sequence and records it (one seed per embedding call and per stack)."""

    def __init__(self, monkeypatch, start=0x243F6A8885A308D3):
        self.seeds, self.next = [], start
        monkeypatch.setattr(ops, "next_seed", self)

    def __call__(self):
        s = self.next
        self.next = (self.next * 6364136223846793005 + 1442695040888963407) & 0xFFFFFFFFFFFFFFFF
        self.seeds.append(s)
        return s


def oracle_drop(p, seeds, spec, B, bf16, offset=0):
    """The callable the oracle takes: layout "emb" [B, T, D]; stack "spatial" [B*C, S, *] / "spectral" [B*S, C, *]
    (attention probabilities [n, H, N, N]) -> t * the kernels' mask, rows mapped to the kernels' token order t = c*S + s."""
    Cb, S = spec.C, spec.S
    amask = R.attn_mask_bf16 if bf16 else R.attn_mask_f32

    def fn(t, site, layout):
        seed = (seeds[layout] + offset) & 0xFFFFFFFFFFFFFFFF
        if t.dim() == 4:
            n, H, N, _ = t.shape
            inner = 1 if layout == "spatial" else S
            return t * _t(amask(p, seed, site, n, N, inner, H))
        m = _t(R.elem_mask(p, seed, site, t.numel()))
        if layout == "spectral":   # oracle rows (b*S + s, c), kernel rows b*T + c*S + s
            m = m.reshape(B, Cb, S, -1).permute(0, 2, 1, 3)
        return t * m.reshape(t.shape)
    return fn


def _finetune(spec, B, prec, monkeypatch, p=0.1):
    rec = SeedRecorder(monkeypatch)
    sd = O.synthetic_state_dict(spec, seed=9)
    m = make_encoder(spec, dropout=p)
    m.load_state_dict(sd)
    m.precision = prec
    m.to(DEV).train()
    x = O.synthetic_cube(spec, B, seed=9)
    rng = np.random.Generator(np.random.PCG64(9))
    hw = (B, spec.image_size, spec.image_size)
    labels = torch.from_numpy(np.where(rng.random(hw) < 0.2, -1, rng.integers(0, spec.num_classes, hw)).astype(np.int64))
    logits = m(x.to(DEV))
    loss = M.cross_entropy(logits, labels.to(DEV), ignore_index=-1)
    loss.backward()
    assert len(rec.seeds) == 3                               # emb-dropout, spatial stack, spectral stack
    seeds = dict(zip(("emb", "spatial", "spectral"), rec.seeds))
    ref = {k: v.double().clone().requires_grad_(True) for k, v in sd.items()}
    drop = oracle_drop(p, seeds, spec, B, prec == "bf16")
    tok = drop(O.encoder_tokens(x.double(), ref, spec), O.SITE_EMB, "emb")
    want_logits = O.head(O.transformer_forward(tok, ref, spec, drop=drop), ref, spec)
    want = O.cross_entropy(want_logits, labels)
    want.backward()
    return m, ref, rel_l2(logits, want_logits), abs(loss.item() - want.item()) / abs(want.item())


def _grads(m, ref, tol):
    worst, n = 0.0, 0
    for k, v in m.named_parameters():
        if k in ref and ref[k].grad is not None:
            e = rel_l2(v.grad, ref[k].grad)
            assert e < tol, (k, e)
            worst, n = max(worst, e), n + 1
    assert n > 20
    return worst


@pytest.mark.parametrize("prec", ["fp32", "bf16"])
@pytest.mark.parametrize("shape", ["houston", "enmap"])
def test_finetune_step_with_dropout_vs_oracle(shape, prec, monkeypatch):
    spec = O.Spec(**(O.HOUSTON if shape == "houston" else O.ENMAP), depth=2)
    m, ref, el, eloss = _finetune(spec, 2, prec, monkeypatch)
    tol = (1e-5, 1e-4) if prec == "fp32" else (1e-2, 5e-2)
    worst = _grads(m, ref, tol[1])
    print(f"finetune {shape} {prec}: logits {el:.2e} loss {eloss:.2e} grads {worst:.2e}")
    assert el < tol[0] and eloss < tol[0]


@pytest.mark.parametrize("prec", ["fp32", "bf16"])
def test_simmim_step_with_dropout_vs_oracle(prec, monkeypatch):
    rec = SeedRecorder(monkeypatch)
    spec = O.Spec(**O.HOUSTON, depth=2)
    B, p = 4, 0.1
    sd = O.synthetic_state_dict(spec, seed=13, simmim=True)
    if prec == "bf16":   # keep every L1 residual away from zero (see test_gpu_shape_sweep): shift the decoder bias
        for k in sd:
            if k.startswith("to_pixels") and k.endswith("bias"):
                sd[k] = sd[k] + 3.0
    enc = M.ViTSpatialSpectral(image_size=8, spatial_patch_size=1, spectral_patch_size=10, num_classes=20, dim=96, depth=2, heads=8,
                               mlp_dim=64, channels=50, spectral_pos_embed=False, dropout=p, emb_dropout=p)
    model = M.SimMIMSpatialSpectral(encoder=enc, masking_ratio=0.7, mask_patch_size=4, tube_masking=True,
                                    to_pixels_per_spectral_block=True)
    model.load_state_dict(sd)
    enc.precision = prec
    model.to(DEV).train()
    x = O.synthetic_cube(spec, B, seed=13)
    rng = np.random.Generator(np.random.PCG64(13))
    mask = torch.from_numpy(rng.random((B, spec.T)) < 0.6)
    idx = torch.from_numpy(rng.integers(0, spec.T, (B, 40)).astype(np.int64))
    loss = model(x.to(DEV), masks=(mask.to(DEV), idx.to(DEV)))
    loss.backward()
    assert len(rec.seeds) == 2, rec.seeds                   # the SimMIM path applies no emb-dropout (C5): stacks only
    ref = {k: v.double().clone().requires_grad_(True) for k, v in sd.items()}
    want = O.simmim_forward(x.double(), ref, spec, mask, idx, drop=oracle_drop(p, dict(zip(("spatial", "spectral"), rec.seeds)),
                                                                           spec, B, prec == "bf16"))
    want.backward()
    e = abs(loss.item() - want.item()) / abs(want.item())
    tol = (1e-5, 1e-4) if prec == "fp32" else (1e-2, 5e-2)
    worst = _grads(model, ref, tol[1])
    print(f"simmim {prec}: loss {e:.2e} grads {worst:.2e}")
    assert e < tol[0]


def test_graphed_step_replays_with_device_seed(monkeypatch):
    """A captured step draws its masks at (captured seed + seed_t): the loss of each replay equals the oracle's at that seed."""
    from maskedsst_b200.graph import GraphedStep
    from maskedsst_b200.optim import FusedAdam
    rec = SeedRecorder(monkeypatch)
    spec = O.Spec(**O.HOUSTON, depth=1)
    B, p = 2, 0.1
    sd = O.synthetic_state_dict(spec, seed=17)
    m = M.ViTSpatialSpectral(image_size=8, spatial_patch_size=1, spectral_patch_size=10, num_classes=20, dim=96, depth=1, heads=8,
                             mlp_dim=64, channels=50, spectral_pos_embed=False, dropout=p, emb_dropout=p)
    m.load_state_dict(sd)
    m.to(DEV).train()
    opt = FusedAdam(m.parameters(), lr=0.0, weight_decay=0.0, capturable=True)   # lr 0: parameters frozen, only masks change
    x = O.synthetic_cube(spec, B, seed=17)
    labels = torch.from_numpy(np.random.Generator(np.random.PCG64(17)).integers(0, 20, (B, 8, 8)).astype(np.int64))
    loss_fn = lambda mm, xi, yi: M.cross_entropy(mm(xi), yi, ignore_index=-1)
    g = GraphedStep(m, opt, (x.to(DEV), labels.to(DEV)), loss_fn=loss_fn, warmup=1)
    seeds = dict(zip(("emb", "spatial", "spectral"), rec.seeds[-3:]))        # the ones baked into the captured graph
    ref = {k: v.double() for k, v in sd.items()}
    for _ in range(2):
        loss = float(g(x.to(DEV), labels.to(DEV)))
        off = int(g.seed_t)
        assert off > 0
        drop = oracle_drop(p, seeds, spec, B, False, offset=off)
        tok = drop(O.encoder_tokens(x.double(), ref, spec), O.SITE_EMB, "emb")
        want = float(O.cross_entropy(O.head(O.transformer_forward(tok, ref, spec, drop=drop), ref, spec), labels))
        print(f"graph replay seed_t={off}: loss {loss:.6f} oracle {want:.6f}")
        assert abs(loss - want) < 1e-5 * abs(want), (off, loss, want)


# ---------------------------------------------------------------------------------------------------------------------
# 5. p = 1: the dropped branches are exactly zero, gradients finite (nn.Dropout(1.0) returns zeros)
# ---------------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("prec", [PREC_FP32, PREC_BF16])
def test_p_one_zeroes_every_site(prec):
    torch.manual_seed(3)
    D, H, Mh, n_seq, N = 96, 2, 64, 6, 64
    layers = [[(torch.randn(*s) * 0.2).to(DEV).requires_grad_(True) for s in
               [(D,), (D,), (3 * H * 64, D), (D, H * 64), (D,), (D,), (D,), (Mh, D), (Mh,), (D, Mh), (D,)]] for _ in range(2)]
    x = torch.randn(n_seq * N, D, device=DEV, requires_grad=True)
    y = ops.transformer_stack(x, layers, n_seq=n_seq, N=N, inner=1, heads=H, dim_head=64, mlp_dim=Mh, drop_p=1.0, seed=5, prec=prec)
    assert torch.equal(y, x)                                 # both residual branches dropped entirely, in every layer
    dy = torch.randn_like(y)
    y.backward(dy)
    assert torch.equal(x.grad, dy)
    for lp in layers:
        for t in lp:
            assert t.grad is not None and torch.isfinite(t.grad).all()
        assert float(lp[4].grad.abs().max()) == 0.0 and float(lp[10].grad.abs().max()) == 0.0   # b_out, b2
    # attention probabilities and the embedding
    qkv = torch.randn(n_seq * N, 3 * H * 64, device=DEV, dtype=torch.bfloat16 if prec == PREC_BF16 else torch.float32,
                      requires_grad=True)
    o = ops.attention(qkv, n_seq=n_seq, N=N, heads=H, dim_head=64, drop_p=1.0, seed=5, site=2)
    assert float(o.float().abs().max()) == 0.0
    o.float().sum().backward()
    assert float(qkv.grad.float().abs().max()) == 0.0
    xo = torch.ones(1024, device=DEV)
    yo = torch.empty_like(xo)
    check(_lib.lib().msst_dropout_apply(xo.data_ptr(), yo.data_ptr(), 1024, 1.0, 5, 3, None, _st()))
    assert float(yo.abs().max()) == 0.0
