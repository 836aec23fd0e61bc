"""GPU: linear probing (maskedsst_b200.inference.linear_probe_fit / LinearProbe / linear_probe_scene, csrc/linprobe.cu) against float64
torch.  The tight tests feed the float64 reference the kernel's own state (teacher forcing): Adam's early steps are close to
lr * sign(g), so a gradient element within fp32 rounding of 0 may legitimately move a parameter by up to 2 lr, and whole fp32 fits are
only compared loosely with whole float64 fits."""
import ctypes

import numpy as np
import pytest
import torch
import torch.nn.functional as F

import maskedsst_b200 as M
from maskedsst_b200 import _lib
from maskedsst_b200.inference import (LinearProbe, _linprobe_dims, _linprobe_grad, _linprobe_update, _pixel_rows, classification_metrics,
                                      confusion_matrix, embed_scene, linear_probe_fit, linear_probe_scene, predict_tiles)
from oracle import maskedsst_oracle as O
from tests.test_gpu_scene_embed import P2X4, _oracle_embed
from tests.test_gpu_scene_inference import _model

pytestmark = pytest.mark.gpu
DEV = "cuda"
WORST = {}


def _note(key, err):
    WORST[key] = max(WORST.get(key, 0.0), err)
    print(f"{key}: {err:.2e} (worst so far {WORST[key]:.2e})")


def _split(params, nc, D):
    H = params.shape[0]
    return params[:, :nc * D].reshape(H, nc, D), params[:, nc * D:]


def _grad64(x, labels, idx, params, nc):
    """float64 (mean gradient [H, P], loss sums [H]) of the minibatch x[idx] at params."""
    D = x.shape[1]
    z = F.layer_norm(x[idx].double(), (D,))
    y = labels[idx]
    W, b = _split(params.double(), nc, D)
    logp = torch.log_softmax(torch.einsum("rd,hcd->hrc", z, W) + b[:, None], -1)
    rows = torch.arange(idx.numel(), device=x.device)
    G = logp.exp()
    G[:, rows, y] -= 1
    gW = torch.einsum("hrc,rd->hcd", G, z) / idx.numel()
    gb = G.sum(1) / idx.numel()
    return torch.cat([gW.reshape(W.shape[0], -1), gb], 1), -logp[:, rows, y].sum(1)


def _adamw64(p, m, v, g, heads, step):
    lr = torch.tensor([h[0] for h in heads], dtype=torch.float64, device=p.device)[:, None]
    wd = torch.tensor([h[1] for h in heads], dtype=torch.float64, device=p.device)[:, None]
    p, m, v, g = p.double(), m.double(), v.double(), g.double()
    p = p * (1 - lr * wd)
    m = 0.9 * m + 0.1 * g
    v = 0.999 * v + 0.001 * g * g
    p = p - lr / (1 - 0.9 ** step) * m / (v.sqrt() / (1 - 0.999 ** step) ** 0.5 + 1e-8)
    return p, m, v


def _kernel_grad(ws, H, P, B):
    """The kernel's mean gradient [H, P] and loss sums [H] from the workspace partials (float64 sum of the fp32 slice partials)."""
    part = ws[:-(-B // 128) * H * (P + 1)].view(-1, H, P + 1).double().sum(0)
    return part[:, :P] / B, part[:, P]


class _Run:
    """The state of a fit driven launch by launch, as linear_probe_fit drives it."""

    def __init__(self, x, labels, nc, heads, batch, params=None, m=None, v=None):
        N, D = x.shape
        self.x, self.labels, self.nc, self.heads = x, labels, nc, heads
        P = nc * D + nc
        self.P = P
        z = lambda: torch.zeros(len(heads), P, device=DEV)
        self.params = params if params is not None else z()
        self.m = m if m is not None else z()
        self.v = v if v is not None else z()
        self.dims = _linprobe_dims(N, D, nc, heads, batch=batch)
        self.ws = torch.empty(_lib.lib().msst_linprobe_workspace(ctypes.byref(self.dims)) // 4, device=DEV)
        self.loss = torch.empty(len(heads), device=DEV)

    def grad(self, idx):
        self.dims.batch = idx.numel()
        _linprobe_grad(self.dims, self.x, self.labels, idx, self.params, self.ws)
        return _kernel_grad(self.ws, len(self.heads), self.P, idx.numel())

    def update(self, step):
        self.dims.step = step
        _linprobe_update(self.dims, self.ws, self.params, self.m, self.v, self.loss)


def _rel(a, b):
    return ((a.double() - b.double()).abs().max() / b.double().abs().max().clamp_min(1e-30)).item()


@pytest.mark.parametrize("D", [32, 96, 256])
@pytest.mark.parametrize("nc", [1, 2, 20, 256])
@pytest.mark.parametrize("H", [1, 3, 16])
def test_grad_and_update_vs_fp64(D, nc, H):
    g = torch.Generator(device=DEV).manual_seed(D * 1000 + nc * 17 + H)
    N = 4200
    x = 2.0 * torch.randn(N, D, device=DEV, generator=g) + 0.5
    labels = torch.randint(0, nc, (N,), device=DEV, generator=g)
    heads = [(10 ** -(1 + h % 3), 0.05 * (h % 2)) for h in range(H)]
    for B in (1, 127, 128, 129, 4099):
        idx = torch.randperm(N, device=DEV, generator=g)[:B]           # gathered, unsorted
        P = nc * D + nc
        params = 0.1 * torch.randn(H, P, device=DEV, generator=g)
        moments = nc > 1                                                 # nc = 1: zero moments, so only the decay moves the parameters
        m = 1e-2 * torch.randn(H, P, device=DEV, generator=g) if moments else torch.zeros(H, P, device=DEV)
        v = 1e-4 * (0.5 + torch.rand(H, P, device=DEV, generator=g)) if moments else torch.zeros(H, P, device=DEV)
        run = _Run(x, labels, nc, heads, B, params.clone(), m.clone(), v.clone())
        gk, lk = run.grad(idx)
        run.update(5)
        want_g, want_l = _grad64(x, labels, idx, params, nc)
        if nc == 1:
            assert torch.equal(gk, torch.zeros_like(gk)) and torch.equal(run.loss, torch.zeros_like(run.loss))
        else:
            eg, el = _rel(gk, want_g), _rel(run.loss, want_l)
            assert eg <= 1e-5 and el <= 1e-5, (B, eg, el)
            _note("gradient rel", eg)
            _note("loss rel", el)
            assert _rel(lk, want_l) <= 1e-5
        p64, m64, v64 = _adamw64(params, m, v, gk, heads, 5)
        ep = (run.params.double() - p64).abs().max().item()
        assert ep <= 1e-6, (B, ep)
        assert _rel(run.m, m64) <= 1e-6 and (run.v.double() - v64).abs().max().item() <= 1e-6 * v64.abs().max().item() + 1e-30
        _note("adamw abs", ep)


def _replay_steps(x, labels, nc, heads, epochs, bs, seed, check):
    """Replays linear_probe_fit launch by launch with the documented permutation draw; check(run, idx, step, state before)."""
    N, bs = x.shape[0], min(bs, x.shape[0])
    run = _Run(x, labels, nc, heads, bs)
    gen = torch.Generator(device=DEV).manual_seed(seed)
    step, sums = 0, []
    for _ in range(epochs):
        perm = torch.randperm(N, generator=gen, device=DEV)
        for first in range(0, N, bs):
            idx = perm[first:first + bs]
            step += 1
            before = (run.params.clone(), run.m.clone(), run.v.clone())
            gk, _ = run.grad(idx)
            run.update(step)
            sums.append(run.loss.clone())
            if check:
                check(run, idx, step, before, gk)
    return run, torch.stack(sums)


def _blobs(N, D, nc, seed, sep=3.0):
    g = torch.Generator(device=DEV).manual_seed(seed)
    means = sep * torch.randn(nc, D, device=DEV, generator=g)
    y = torch.randint(0, nc, (N,), device=DEV, generator=g)
    return means[y] + torch.randn(N, D, device=DEV, generator=g), y


def test_short_fit_replayed_step_by_step():
    x, y = _blobs(700, 64, 5, seed=1)
    heads = [(1e-2, 0.05), (3e-3, 0.0)]
    probe = linear_probe_fit(x, y, num_classes=5, heads=heads, epochs=3, batch_size=256, seed=4, val=(x[:100], y[:100]))

    def check(run, idx, step, before, gk):
        want_g, want_l = _grad64(x, y, idx, before[0], 5)
        _note("stepped gradient rel", _rel(gk, want_g))
        assert _rel(gk, want_g) <= 1e-5 and _rel(run.loss, want_l) <= 1e-5
        p64, _, _ = _adamw64(*before, gk, heads, step)
        ep = (run.params.double() - p64).abs().max().item()
        _note("stepped adamw abs", ep)
        assert ep <= 1e-6

    run, sums = _replay_steps(x, y, 5, heads, 3, 256, 4, check)
    assert torch.equal(run.params, probe.params)                       # the documented draw is the one the fit uses
    want = sums.cpu().double().reshape(3, 3, 2).sum(1) / 700
    assert probe.train_loss.shape == (3, 2) and (probe.train_loss - want).abs().max().item() <= 1e-12


def _fit64(x, y, nc, heads, epochs, bs, seed):
    """The whole fit in float64 (same permutations, AdamW in float64); -> params [H, P] float64."""
    N, D = x.shape
    H = len(heads)
    p = torch.zeros(H, nc * D + nc, dtype=torch.float64, device=DEV)
    m, v = torch.zeros_like(p), torch.zeros_like(p)
    gen = torch.Generator(device=DEV).manual_seed(seed)
    step = 0
    for _ in range(epochs):
        perm = torch.randperm(N, generator=gen, device=DEV)
        for first in range(0, N, min(bs, N)):
            idx = perm[first:first + min(bs, N)]
            step += 1
            g, _ = _grad64(x, y, idx, p, nc)
            p, m, v = _adamw64(p, m, v, g, heads, step)
    return p


def _probs64(x, params64, nc):
    W, b = _split(params64, nc, x.shape[1])
    return torch.softmax(F.layer_norm(x.double(), (x.shape[1],)) @ W[0].T + b[0], -1)


def _loose(probs, pred, want, tol=1e-3):
    err = (probs.double() - want).abs().max().item()
    top2 = torch.topk(want, min(2, want.shape[1]), 1)
    clear = top2.values[:, 0] - top2.values[:, -1] > 1e-3
    assert torch.equal(pred[clear], top2.indices[clear, 0])
    assert err <= tol, err
    return err


def test_whole_fit_close_to_fp64_fit():
    x, y = _blobs(2000, 32, 4, seed=2)
    heads = [(1e-2, 1e-2)]
    probe = linear_probe_fit(x, y, num_classes=4, heads=heads, epochs=20, batch_size=256, seed=7)
    want = _probs64(x, _fit64(x, y, 4, heads, 20, 256, 7), 4)
    probs, pred = probe.predict(x)
    _note("whole fit probs abs", _loose(probs, pred, want))
    assert float((pred == y).double().mean()) > 0.95


def test_fits_are_bitwise_reproducible_and_heads_independent():
    x, y = _blobs(1500, 96, 20, seed=3, sep=0.5)
    heads = [(10 ** -(2 + h % 3), 0.02 * (h % 4)) for h in range(8)]
    kw = dict(num_classes=20, epochs=3, batch_size=300, seed=11, val=(x[:200], y[:200]))
    a = linear_probe_fit(x, y, heads=heads, **kw)
    b = linear_probe_fit(x, y, heads=heads, **kw)
    assert torch.equal(a.params, b.params) and torch.equal(a.train_loss, b.train_loss)
    for h, hp in enumerate(heads):
        alone = linear_probe_fit(x, y, heads=[hp], **kw)
        assert torch.equal(alone.params[0], a.params[h]), h
        assert torch.equal(alone.train_loss[:, 0], a.train_loss[:, h]), h
    assert a.best == int(torch.argmax(a.val_acc))
    q = torch.randn(2500, 96, device=DEV)
    p0, i0 = a.predict(q, head=3)
    for bq in (1, 1000, 2500):
        n = 300 if bq == 1 else 2500
        p, i = a.predict(q[:n], head=3, batch_queries=bq)
        assert torch.equal(p, p0[:n]) and torch.equal(i, i0[:n]), bq


@pytest.mark.parametrize("D", [32, 256])
@pytest.mark.parametrize("nc", [1, 20, 256])
def test_predict_vs_fp64(D, nc):
    g = torch.Generator(device=DEV).manual_seed(D + nc)
    # W ~ N(0, 1/D) as a fitted probe's scale: logits of order 1 (at |logit| ~ 20 the fp32 ulp alone would be 2e-6 of a probability)
    params = torch.randn(1, nc * D + nc, device=DEV, generator=g) * 0.3
    params[:, :nc * D] *= D ** -0.5
    probe = LinearProbe(params, nc, D, [(0.0, 0.0)])
    x = 3.0 * torch.randn(1000, D, device=DEV, generator=g) - 1.0
    x[5] = 0
    x[6] = 2.5                                                    # constant rows normalise to 0: logits = b
    probs, pred = probe.predict(x)
    want = _probs64(x, params.double(), nc)
    err = (probs.double() - want).abs().max().item()
    _note("predict probs abs", err)
    assert err <= 1e-6
    _, b = _split(params, nc, D)
    sb = torch.softmax(b[0].double(), -1)
    assert (probs[5:7].double() - sb).abs().max().item() <= 1e-6
    assert torch.equal(probs[5], probs[6])
    clear = torch.topk(want, min(2, nc), 1).values
    clear = clear[:, 0] - clear[:, -1] > 1e-6 if nc > 1 else torch.ones(1000, dtype=torch.bool, device=DEV)
    assert torch.equal(pred[clear], want.argmax(1)[clear])


def test_predict_ties_go_to_the_lowest_class():
    D, nc = 64, 6
    g = torch.Generator(device=DEV).manual_seed(9)
    W = 0.1 * torch.randn(nc, D, device=DEV, generator=g)
    b = torch.zeros(nc, device=DEV)
    W[4], W[1] = 3 * W[0], 3 * W[0]                               # classes 1 and 4 identical and dominant on rows along W[0]
    b[1] = b[4] = 1.0
    probe = LinearProbe(torch.cat([W.reshape(-1), b])[None].contiguous(), nc, D, [(0.0, 0.0)])
    x = W[0][None].repeat(50, 1) * torch.rand(50, 1, device=DEV, generator=g) * 10 + 0.01 * torch.randn(50, D, device=DEV, generator=g)
    probs, pred = probe.predict(x)
    assert torch.equal(probs[:, 1], probs[:, 4])
    top = probs.max(1).values
    assert bool((probs[:, 1] == top).all()) and bool((pred == 1).all())
    zero = probe.predict(torch.zeros(3, D, device=DEV))             # z = 0: logits = b, classes 1 and 4 tie again
    assert bool((zero[1] == 1).all())


@pytest.mark.parametrize("kw", [O.HOUSTON, P2X4], ids=["p1=1", "p1=2"])
def test_load_into_default_head_matches_probe(kw):
    m, spec, sd = _model(kw, 2, 81)
    nc, D = spec.num_classes, spec.dim
    g = torch.Generator(device=DEV).manual_seed(12)
    probe = LinearProbe(0.5 * torch.randn(2, nc * D + nc, device=DEV, generator=g), nc, D, [(0.0, 0.0)] * 2, best=1)
    scene = torch.from_numpy(np.random.default_rng(3).standard_normal((2, spec.channels, 16, 24)).astype(np.float32)).to(DEV)
    w = spec.image_size
    lin_w = m.mlp_head[1].weight
    probe.load_into(m)
    assert m.mlp_head[1].weight is lin_w                            # in place
    got = torch.softmax(predict_tiles(m, scene), 1)                # [B, nc, H, W]
    feats = embed_scene(m, scene, stride=w)
    probs, _ = probe.predict(_pixel_rows(feats))                   # best head
    want = probs.reshape(2, 16, 24, nc).permute(0, 3, 1, 2)
    err = (got - want).abs().max().item()
    _note("export probs abs", err)
    assert err <= 1e-5


def _scene(case):
    m, spec, sd = _model(O.HOUSTON, 2, 81)
    cube = torch.from_numpy(np.random.default_rng(7).standard_normal((1, spec.channels, 19, 22)).astype(np.float32))
    model = M.SimMIMSpatialSpectral(encoder=m, masking_ratio=0.5).to(DEV) if case == "simmim" else m
    return model, spec, sd, cube


@pytest.mark.parametrize("case", ["vit", "simmim"])
def test_linear_probe_scene_vs_oracle(case):
    model, spec, sd, cube = _scene(case)
    B, _, H, W = cube.shape
    nc = spec.num_classes
    g = torch.Generator().manual_seed(5)
    labels = torch.randint(0, nc, (B, H, W), generator=g)
    labels[torch.rand(B, H, W, generator=g) < 0.5] = -1
    labels[0, 0, :3] = nc + 2                                      # out of range: not a training row
    val = torch.randint(0, nc, (B, H, W), generator=g)
    heads = [(1e-2, 0.0), (1e-3, 0.01), (3e-2, 0.0)]
    probs, pred, probe = linear_probe_scene(model, cube.to(DEV), labels.to(DEV), num_classes=nc, val_labels=val.to(DEV), heads=heads,
                                            epochs=15, batch_size=64, seed=2, stride=3)
    assert probs.shape == (B, nc, H, W) and pred.shape == (B, H, W) and probe.val_acc.shape == (3,)
    feats = torch.from_numpy(_oracle_embed(cube, sd, spec, 3, None)).to(DEV)        # float64 [B, D, H, W]
    flat = feats.permute(0, 2, 3, 1).reshape(B * H * W, -1)
    lab = labels.reshape(-1).to(DEV)
    ok = (lab >= 0) & (lab < nc)
    got = probs.permute(0, 2, 3, 1).reshape(B * H * W, nc)
    for h in range(3):
        p64 = _fit64(flat[ok], lab[ok], nc, [heads[h]], 15, 64, 2)
        want = _probs64(flat, p64, nc)
        ph, ih = probe.predict(_pixel_rows(embed_scene(model, cube.to(DEV), stride=3)), head=h)
        _note(f"scene probs abs ({case})", _loose(ph, ih, want))
        assert abs(probe.val_acc[h].item() - float((ih == val.reshape(-1).to(DEV)).double().mean())) < 1e-12
        if h == probe.best:
            assert torch.equal(got, ph) and torch.equal(pred.reshape(-1), ih)
    assert probe.best == int(torch.argmax(probe.val_acc))


def test_linear_probe_scene_separable_classes_score_oa_one():
    """Four 16 x 16 class quadrants, one spectrum each, tiled by 8 x 8 windows: the held-out windows' features are copies of labelled
    ones of their class."""
    m, spec, sd = _model(O.HOUSTON, 2, 81)
    B, H, W = 1, 32, 32
    g = torch.Generator().manual_seed(8)
    truth = torch.zeros(B, H, W, dtype=torch.int64)
    truth[:, :16, 16:] = 1
    truth[:, 16:, :16] = 2
    truth[:, 16:, 16:] = 3
    cube = (3.0 * torch.randn(4, spec.channels, generator=g))[truth].permute(0, 3, 1, 2).contiguous()
    labelled = torch.zeros(B, H, W, dtype=torch.bool)
    for y in (0, 16):
        for x in (0, 16):
            labelled[:, y:y + 8, x:x + 8] = True
            labelled[:, y + 8:y + 16, x + 8:x + 16] = True
    train = torch.where(labelled, truth, torch.full_like(truth, -1))
    held_out = torch.where(labelled, torch.full_like(truth, -1), truth)
    _, pred, probe = linear_probe_scene(m, cube.to(DEV), train.to(DEV), num_classes=4, heads=[(5e-2, 0.0)], epochs=200, batch_size=128,
                                        stride=8)
    metrics = classification_metrics(confusion_matrix(pred, held_out.to(DEV), 4))
    assert metrics["oa"] == 1.0 and metrics["kappa"] == 1.0, metrics
    assert probe.train_loss[-1, 0] < probe.train_loss[0, 0]


def test_c_abi_limits_leave_outputs_untouched():
    L = _lib.lib()
    x = torch.randn(300, 96, device=DEV)
    labels = torch.zeros(300, device=DEV, dtype=torch.int64)
    idx = torch.arange(300, device=DEV)
    params = torch.full((16, 257 * 256), 7.0, device=DEV)
    m, v = params.clone(), params.clone()
    ws = torch.full((3 * 16 * (257 * 256 + 1),), 7.0, device=DEV)
    loss = torch.full((16,), 7.0, device=DEV)
    probs = torch.full((300, 256), 7.0, device=DEV)
    pred = torch.full((300,), 7, device=DEV, dtype=torch.int64)
    st = None

    def dims(**kw):
        d = dict(n=300, dim=96, nc=20, heads=2, batch=300, step=1)
        d.update(kw)
        out = _lib.LinprobeDims(d["n"], d["dim"], d["nc"], d["heads"], d["batch"], d["step"])
        for h in range(16):
            out.lr[h], out.wd[h] = kw.get("lr", 1e-3), kw.get("wd", 0.0)
        return out

    bad = [(dict(dim=80), b"dim=80"), (dict(dim=288), b"dim=288"), (dict(dim=0), b"dim=0"), (dict(nc=0), b"nc=0"), (dict(nc=257), b"nc=257"),
           (dict(heads=0), b"heads=0"), (dict(heads=17), b"heads=17"), (dict(n=0), b"n=0"), (dict(n=2 ** 31), b"n=2147483648"),
           (dict(batch=0), b"batch=0")]
    for kw, what in bad:
        d = dims(**kw)
        assert L.msst_linprobe_grad(ctypes.byref(d), x.data_ptr(), labels.data_ptr(), idx.data_ptr(), params.data_ptr(), ws.data_ptr(), st) == 1
        assert what in L.msst_last_error(), (kw, L.msst_last_error())
        assert L.msst_linprobe_update(ctypes.byref(d), ws.data_ptr(), params.data_ptr(), m.data_ptr(), v.data_ptr(), loss.data_ptr(), st) == 1
        assert what in L.msst_last_error(), (kw, L.msst_last_error())
        assert L.msst_linprobe_workspace(ctypes.byref(d)) == -1
    for kw, what in [(dict(step=0), b"step=0"), (dict(lr=-1.0), b"lr[0]"), (dict(lr=float("nan")), b"lr[0]"), (dict(wd=float("inf")), b"wd[0]")]:
        d = dims(**kw)
        assert L.msst_linprobe_update(ctypes.byref(d), ws.data_ptr(), params.data_ptr(), m.data_ptr(), v.data_ptr(), loss.data_ptr(), st) == 1
        assert what in L.msst_last_error(), (kw, L.msst_last_error())
    d = dims()
    assert L.msst_linprobe_grad(ctypes.byref(d), x.data_ptr(), labels.data_ptr(), None, params.data_ptr(), ws.data_ptr(), st) == 1
    assert b"must be set" in L.msst_last_error()
    assert L.msst_linprobe_update(ctypes.byref(d), ws.data_ptr(), params.data_ptr(), m.data_ptr(), None, loss.data_ptr(), st) == 1
    assert b"must be set" in L.msst_last_error()
    assert L.msst_linprobe_grad(None, x.data_ptr(), labels.data_ptr(), idx.data_ptr(), params.data_ptr(), ws.data_ptr(), st) == 1
    assert b"dims" in L.msst_last_error()
    for args, what in [((300, 80, 20), b"dim=80"), ((300, 96, 0), b"nc=0"), ((300, 96, 257), b"nc=257"), ((0, 96, 20), b"n_query=0"),
                       ((2 ** 31, 96, 20), b"n_query=")]:
        assert L.msst_linprobe_predict(*args, x.data_ptr(), params.data_ptr(), probs.data_ptr(), pred.data_ptr(), st) == 1
        assert what in L.msst_last_error(), (args, L.msst_last_error())
    assert L.msst_linprobe_predict(300, 96, 20, x.data_ptr(), None, probs.data_ptr(), pred.data_ptr(), st) == 1
    torch.cuda.synchronize()
    for t in (params, m, v, ws, loss, probs):
        assert bool((t == 7).all())
    assert bool((pred == 7).all())


def test_labels_outside_the_classes_do_not_reach_memory_or_the_sums():
    """The C layer skips a row whose label is outside [0, nc) or whose index is outside [0, n) (the Python layer rejects both)."""
    x, y = _blobs(600, 32, 3, seed=6)
    bad = y.clone()
    bad[::7] = 1 << 40
    bad[1::7] = -5
    keep = torch.ones(600, dtype=torch.bool, device=DEV)
    keep[::7] = False
    keep[1::7] = False
    heads = [(1e-2, 0.0)]
    run = _Run(x, bad, 3, heads, 600)
    idx = torch.arange(600, device=DEV)
    gk, lk = run.grad(idx)
    want_g, want_l = _grad64(x, y, idx[keep], torch.zeros(1, 3 * 32 + 3, device=DEV), 3)
    assert _rel(gk * 600, want_g * int(keep.sum())) <= 1e-5 and _rel(lk, want_l) <= 1e-5
    idx2 = idx.clone()
    idx2[::7] = 10 ** 9
    idx2[1::7] = -3
    gk2, lk2 = _Run(x, y, 3, heads, 600).grad(idx2)
    assert _rel(gk2, gk) <= 1e-6 and _rel(lk2, lk) <= 1e-6
