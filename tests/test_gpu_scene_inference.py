"""GPU: whole-scene inference (maskedsst_b200/inference.py:predict_scene, csrc/scene.cu): strided / chunked window addressing in the
pixel reader, the deterministic probability blend, and the driver against the CPU oracle."""
import json

import numpy as np
import pytest
import torch

import maskedsst_b200 as M
from maskedsst_b200.inference import blend_windows, predict_scene, predict_tiles, scene_windows
from oracle import maskedsst_oracle as O
from tests.helpers import gold, rel_l2
from tests.test_gpu_parity import make_encoder

pytestmark = pytest.mark.gpu
DEV = "cuda"


def _model(kw, depth, seed, precision="fp32"):
    spec = O.Spec(**kw, depth=depth)
    sd = O.synthetic_state_dict(spec, seed=seed)
    m = make_encoder(spec).eval()
    m.load_state_dict(sd)
    m.precision = precision
    return m.to(DEV), spec, sd


def _stats(tag):
    g = gold("input_pipeline")
    meta = json.loads(str(g[f"{tag}__meta"]))
    return g[f"{tag}__means"], g[f"{tag}__stds"], meta


def _origins(extent, win, step, n):
    return np.minimum(np.arange(n) * step, extent - win)


@pytest.mark.parametrize("tag,shape,stride,rng_", [
    ("houston", (2, 48, 21, 19), 3, (25, 20)),    # crosses the tile boundary at window 30; windows 25-29 are the snapped last row
    ("houston", (2, 48, 21, 19), 3, (0, 60)),
    ("houston", (1, 48, 13, 30), (2, 5), (3, 1)),   # a chunk of one window, unequal strides
    ("enmap", (2, 200, 18, 12), 3, (4, 23)),      # clip of the standardised value; snapped last row and column
])
def test_strided_windows_read_the_same_pixels(tag, shape, stride, rng_):
    means, stds, meta = _stats(tag)
    clip = (-1.0, 1.0) if tag == "enmap" else None
    raw = torch.from_numpy(np.random.default_rng(7).integers(-400, 12000, shape).astype(np.int16)).to(DEV)
    ny, nx = scene_windows(shape[2], shape[3], 8, stride)
    rt = M.RawTiles(raw, means, stds, image_size=8, pad_bands=meta["pad"], clip=clip, windows=(ny, nx), stride=stride,
                    window_range=rng_)
    assert tuple(rt.shape) == (rng_[1], shape[1] + meta["pad"], 8, 8)
    cube = rt.materialize()
    # materialize() itself against the oracle's restatement of the reference pipeline at each window's origin
    sy, sx = (stride, stride) if isinstance(stride, int) else stride
    oy, ox = _origins(shape[2], 8, sy, ny), _origins(shape[3], 8, sx, nx)
    pipe = O.input_pipeline(raw.cpu().numpy(), means, stds, max(shape[2], shape[3]), pad_bands=meta["pad"], clip=clip)  # whole scene
    for k, gw in enumerate(range(rng_[0], rng_[0] + rng_[1])):
        t, w = divmod(gw, ny * nx)
        y0, x0 = oy[w // nx], ox[w % nx]
        assert torch.equal(cube[k].cpu(), pipe[t, :, y0:y0 + 8, x0:x0 + 8])
    m, _, _ = _model(O.HOUSTON if tag == "houston" else O.ENMAP, 1, 13)
    with torch.no_grad():
        assert torch.equal(m(rt), m(cube))


def _oracle_scene(cube, sd, spec, stride, weight):
    """numpy blend of O.encoder_forward over every window (float64 softmax and sums)."""
    B, _, H, W = cube.shape
    ny, nx = scene_windows(H, W, 8, stride)
    oy, ox = _origins(H, 8, stride, ny), _origins(W, 8, stride, nx)
    wins = torch.stack([cube[b, :, y:y + 8, x:x + 8] for b in range(B) for y in oy for x in ox])
    logits = O.encoder_forward(wins, sd, spec).double().numpy().reshape(B, ny, nx, spec.num_classes, 8, 8)
    p = np.exp(logits - logits.max(3, keepdims=True))
    p /= p.sum(3, keepdims=True)
    wt = np.ones((8, 8)) if weight is None else weight.astype(np.float64)
    acc = np.zeros((B, spec.num_classes, H, W))
    ws = np.zeros((B, H, W))
    for b in range(B):
        for i, y in enumerate(oy):
            for j, x in enumerate(ox):
                acc[b, :, y:y + 8, x:x + 8] += wt * p[b, i, j]
                ws[b, y:y + 8, x:x + 8] += wt
    return acc / ws[:, None]


@pytest.mark.parametrize("weighted", [False, True])
def test_predict_scene_vs_oracle(weighted):
    m, spec, sd = _model(O.HOUSTON, 2, 71)
    cube = O.synthetic_cube(O.Spec(**O.HOUSTON, image_size=21), 2, seed=9)[:, :, :, :19].contiguous()   # 2 x 50 x 21 x 19
    yy, xx = np.meshgrid(np.arange(8) - 3.5, np.arange(8) - 3.5, indexing="ij")
    weight = np.exp(-(yy ** 2 + xx ** 2) / (2 * 2.0 ** 2)).astype(np.float32) if weighted else None
    m.train()
    probs, pred = predict_scene(m, cube.to(DEV), stride=3, weight=weight)
    assert m.training                                                          # the training flag is restored
    assert probs.shape == (2, 20, 21, 19) and pred.shape == (2, 21, 19) and pred.dtype == torch.int64
    want = _oracle_scene(cube, sd, spec, 3, weight)
    assert rel_l2(probs, want) < 1e-5
    top2 = np.sort(want, axis=1)[:, -2:]
    sure = (top2[:, 1] - top2[:, 0]) > 1e-4
    assert np.array_equal(pred.cpu().numpy()[sure], want.argmax(1)[sure])
    assert torch.allclose(probs.sum(1), torch.ones_like(probs[:, 0]), atol=1e-5)


def _blend_chunks(logits, acc, wsum, weight, geom, chunk):
    stride, grid = geom
    total = logits.shape[0]
    for first in range(0, total, chunk):
        blend_windows(logits[first:first + chunk], acc, wsum, stride=stride, grid=grid, first=first, weight=weight)


@pytest.mark.parametrize("nc,stride,weighted", [(20, (3, 3), True), (8, (2, 5), False), (64, (1, 1), True)])
def test_blend_is_chunk_invariant_bitwise(nc, stride, weighted):
    B, H, W = 2, 21, 19
    ny, nx = scene_windows(H, W, 8, stride)
    g = torch.Generator(device=DEV).manual_seed(5)
    logits = 4 * torch.randn(B * ny * nx, nc, 8, 8, device=DEV, generator=g)
    weight = torch.rand(8, 8, device=DEV, generator=g) + 0.1 if weighted else None
    res = []
    for chunk in (1, 7, B * ny * nx):
        acc = torch.zeros(B, nc, H, W, device=DEV)
        wsum = torch.zeros(B, H, W, device=DEV)
        _blend_chunks(logits, acc, wsum, weight, (stride, (ny, nx)), chunk)
        res.append((acc, wsum))
    for acc, wsum in res[1:]:
        assert torch.equal(acc, res[0][0]) and torch.equal(wsum, res[0][1])
    # and the sums are the right ones (float64 reference)
    oy, ox = _origins(H, 8, stride[0], ny), _origins(W, 8, stride[1], nx)
    p = torch.softmax(logits.double(), 1).cpu().numpy().reshape(B, ny, nx, nc, 8, 8)
    wt = np.ones((8, 8)) if weight is None else weight.double().cpu().numpy()
    acc = np.zeros((B, nc, H, W))
    ws = np.zeros((B, H, W))
    for b in range(B):
        for i, y in enumerate(oy):
            for j, x in enumerate(ox):
                acc[b, :, y:y + 8, x:x + 8] += wt * p[b, i, j]
                ws[b, y:y + 8, x:x + 8] += wt
    assert rel_l2(res[0][0], acc) < 1e-6 and rel_l2(res[0][1], ws) < 1e-6


def test_predict_scene_chunking():
    """End to end with batch_windows 1, 7 and all: the blend is bitwise chunk-invariant, so any difference comes from the forward
    at a different batch size."""
    m, _, _ = _model(O.HOUSTON, 2, 72)
    cube = torch.randn(1, 50, 21, 19, device=DEV)
    ny, nx = scene_windows(21, 19, 8, 3)
    out = [predict_scene(m, cube, stride=3, batch_windows=bw) for bw in (1, 7, ny * nx)]
    for probs, pred in out[1:]:
        assert (probs - out[0][0]).abs().max().item() <= 1e-6
    exact = all(torch.equal(p, out[0][0]) for p, _ in out[1:])
    print(f"predict_scene over batch_windows 1 / 7 / {ny * nx}: bitwise equal = {exact}")


def test_stride_window_equals_predict_tiles():
    m, _, _ = _model(O.HOUSTON, 2, 73)
    cube = torch.randn(2, 50, 24, 16, device=DEV)
    probs, pred = predict_scene(m, cube)
    want = torch.softmax(predict_tiles(m, cube), 1)
    assert (probs - want).abs().max().item() <= 1e-6
    assert torch.equal(pred, want.argmax(1))
    means, stds, meta = _stats("houston")
    raw = torch.from_numpy(O.synthetic_raw_tiles(1, 48, 64, 23)).to(DEV)
    rt = M.RawTiles(raw, means, stds, image_size=8, pad_bands=meta["pad"])
    probs, pred = predict_scene(m, rt, batch_windows=24)
    want = torch.softmax(predict_tiles(m, rt), 1)
    assert (probs - want).abs().max().item() <= 1e-6
    assert torch.equal(pred, want.argmax(1))


def test_bf16_scene_close_to_fp32():
    means, stds, _ = _stats("enmap")
    raw = torch.from_numpy(np.random.default_rng(11).integers(-400, 12000, (1, 200, 27, 22)).astype(np.int16)).to(DEV)
    rt = M.RawTiles(raw, means, stds, image_size=8, clip=(-2.0, 2.0))
    m32, _, _ = _model(O.ENMAP, 2, 74)
    m16, _, _ = _model(O.ENMAP, 2, 74, precision="bf16")
    p32, _ = predict_scene(m32, rt, stride=4)
    p16, _ = predict_scene(m16, rt, stride=4, batch_windows=10)
    assert p16.shape == (1, 8, 27, 22) and torch.isfinite(p16).all()
    assert rel_l2(p16, p32) < 1e-2


def test_window_level_head_is_rejected():
    """The pixelwise head gives one class vector per window (p1 x p1 pixels, quirk C14 squeezes it further), not a map of the window:
    there is nothing to blend per pixel, and predict_scene says so instead of misreading the output."""
    m = M.ViTSpatialSpectral(image_size=8, spatial_patch_size=1, spectral_patch_size=10, num_classes=20, dim=96, depth=1, heads=8,
                             mlp_dim=64, channels=50, spectral_pos_embed=False, pixelwise=True).to(DEV).eval()
    for bw in (1, 4096):
        with pytest.raises(ValueError, match="every pixel"):
            predict_scene(m, torch.randn(1, 50, 10, 9, device=DEV), stride=2, batch_windows=bw)


def test_predict_scene_argument_checks():
    m, _, _ = _model(O.HOUSTON, 1, 75)
    means, stds, meta = _stats("houston")
    raw = torch.zeros(1, 48, 20, 20, dtype=torch.int16, device=DEV)
    with pytest.raises(ValueError):
        predict_scene(m, M.RawTiles(raw, means, stds, image_size=8, pad_bands=2, crop=(1, 0)))
    with pytest.raises(ValueError):
        predict_scene(m, torch.zeros(1, 50, 7, 20, device=DEV))
    with pytest.raises(ValueError):
        predict_scene(m, torch.zeros(1, 50, 20, 20, device=DEV), stride=9)
    with pytest.raises(ValueError):
        predict_scene(m, torch.zeros(1, 50, 20, 20, device=DEV), weight=torch.ones(4, 4))
