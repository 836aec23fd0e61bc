"""GPU: whole-scene embedding maps (maskedsst_b200.inference.embed_scene / embed_windows, msst_scene_embed in csrc/scene.cu): per-pixel
encoder features blended from overlapping windows, against a float64 numpy blend of the CPU oracle's tokens."""
import numpy as np
import pytest
import torch

import maskedsst_b200 as M
from maskedsst_b200.inference import embed_scene, embed_windows, scene_windows
from oracle import maskedsst_oracle as O
from tests.helpers import rel_l2
from tests.test_gpu_scene_inference import _model, _origins, _stats

pytestmark = pytest.mark.gpu
DEV = "cuda"


def _gauss(w=8, sigma=2.0):
    yy, xx = np.meshgrid(np.arange(w) - (w - 1) / 2, np.arange(w) - (w - 1) / 2, indexing="ij")
    return np.exp(-(yy ** 2 + xx ** 2) / (2 * sigma ** 2)).astype(np.float32)


def _blend_features(f, B, H, W, w, stride, weight):
    """float64 blend of per-window feature maps f [B * ny * nx, D, w, w] into the scene: sum(weight * f) / sum(weight)."""
    sy, sx = (stride, stride) if isinstance(stride, int) else stride
    ny, nx = scene_windows(H, W, w, (sy, sx))
    oy, ox = _origins(H, w, sy, ny), _origins(W, w, sx, nx)
    f = np.asarray(f, dtype=np.float64).reshape(B, ny, nx, -1, w, w)
    wt = np.ones((w, w)) if weight is None else np.asarray(weight, dtype=np.float64)
    acc = np.zeros((B, f.shape[3], H, W))
    ws = np.zeros((B, H, W))
    for b in range(B):
        for i, y in enumerate(oy):
            for j, x in enumerate(ox):
                acc[b, :, y:y + w, x:x + w] += wt * f[b, i, j]
                ws[b, y:y + w, x:x + w] += wt
    return acc, ws


def _window_features(tokens, C, p1):
    """[n, C*S, D] tokens -> [n, D, G*p1, G*p1]: the spectral mean at each spatial patch, repeated over its p1 x p1 pixels."""
    n, T, D = tokens.shape
    G = int(round((T // C) ** 0.5))
    f = tokens.reshape(n, C, G, G, D).mean(1)
    return f.repeat_interleave(p1, 1).repeat_interleave(p1, 2).permute(0, 3, 1, 2)


def _oracle_embed(cube, sd, spec, stride, weight):
    """float64: O.transformer_forward(O.encoder_tokens(window)) for every window, spectral mean, blended in numpy."""
    B, _, H, W = cube.shape
    w = spec.image_size
    sy, sx = (stride, stride) if isinstance(stride, int) else stride
    ny, nx = scene_windows(H, W, w, (sy, sx))
    oy, ox = _origins(H, w, sy, ny), _origins(W, w, sx, nx)
    wins = torch.stack([cube[b, :, y:y + w, x:x + w] for b in range(B) for y in oy for x in ox]).double()
    sd64 = {k: v.double() for k, v in sd.items()}
    tok = O.transformer_forward(O.encoder_tokens(wins, sd64, spec), sd64, spec)
    acc, ws = _blend_features(_window_features(tok, spec.C, spec.spatial_patch_size).numpy(), B, H, W, w, (sy, sx), weight)
    return acc / ws[:, None]


P2X4 = dict(channels=48, num_classes=20, spatial_patch_size=2, spectral_patch_size=4)   # G = 4, C = 12


@pytest.mark.parametrize("case", ["houston", "houston_gauss", "p2x4", "spectral_only", "simmim"])
def test_embed_scene_vs_oracle(case):
    kw = {"p2x4": P2X4, "spectral_only": dict(**O.HOUSTON, spectral_only=True)}.get(case, O.HOUSTON)
    m, spec, sd = _model(kw, 2, 81)
    shape = (2, spec.channels, 21, 19) if case != "p2x4" else (1, spec.channels, 19, 22)
    cube = torch.from_numpy(np.random.default_rng(4).standard_normal(shape).astype(np.float32))
    weight = _gauss() if case == "houston_gauss" else None
    model = M.SimMIMSpatialSpectral(encoder=m, masking_ratio=0.5).to(DEV) if case == "simmim" else m
    model.train()
    feats = embed_scene(model, cube.to(DEV), stride=3, weight=weight)
    assert model.training and m.training                                   # the training flags are restored
    assert feats.shape == (shape[0], spec.dim, shape[2], shape[3]) and feats.dtype == torch.float32
    want = _oracle_embed(cube, sd, spec, 3, weight)
    err = rel_l2(feats, want)
    print(f"{case}: rel-l2 {err:.2e}")
    assert err <= 1e-5


def _embed_chunks(tokens, acc, wsum, C, p1, stride, grid, weight, chunk):
    for first in range(0, tokens.shape[0], chunk):
        embed_windows(tokens[first:first + chunk], acc, wsum, C=C, p1=p1, stride=stride, grid=grid, first=first, weight=weight)


@pytest.mark.parametrize("D,C,p1,weighted", [(32, 3, 2, False), (96, 5, 1, True), (256, 2, 4, True)])
@pytest.mark.parametrize("stride", [(2, 5), (1, 1)])
def test_embed_windows_chunk_invariant_bitwise(D, C, p1, weighted, stride):
    B, H, W, w = 2, 21, 19, 8
    G = w // p1
    ny, nx = scene_windows(H, W, w, stride)
    n = B * ny * nx
    g = torch.Generator(device=DEV).manual_seed(D)
    tokens = torch.randn(n, C * G * G, D, device=DEV, generator=g)
    weight = torch.rand(w, w, device=DEV, generator=g) + 0.1 if weighted else None
    res = []
    for chunk in (1, 7, n):
        acc = torch.zeros(B, D, H, W, device=DEV)
        wsum = torch.zeros(B, H, W, device=DEV)
        _embed_chunks(tokens, acc, wsum, C, p1, stride, (ny, nx), weight, chunk)
        res.append((acc, wsum))
    for acc, wsum in res[1:]:
        assert torch.equal(acc, res[0][0]) and torch.equal(wsum, res[0][1])
    acc, ws = _blend_features(_window_features(tokens.double(), C, p1).cpu().numpy(), B, H, W, w, stride,
                              None if weight is None else weight.cpu().numpy())
    assert rel_l2(res[0][0], acc) <= 1e-6 and rel_l2(res[0][1], ws) <= 1e-6


def _stitched(enc, x, B, gh, gw):
    """per-window forward_features spectral means stitched into the scene in torch (windows do not overlap)."""
    w, C, p1 = enc.image_size, enc.num_spectral_patches, enc.patch_height
    with torch.no_grad():
        f = _window_features(enc.forward_features(x), C, p1)                  # [B*gh*gw, D, w, w]
    D = f.shape[1]
    return f.reshape(B, gh, gw, D, w, w).permute(0, 3, 1, 4, 2, 5).reshape(B, D, gh * w, gw * w)


def test_stride_window_equals_stitched_forward_features():
    m, _, _ = _model(O.HOUSTON, 2, 83)
    cube = torch.randn(2, 50, 24, 16, device=DEV)
    feats = embed_scene(m, cube)
    ident = torch.zeros(50, dtype=torch.float64), torch.ones(50, dtype=torch.float64)
    want = _stitched(m, M.RawTiles(cube, *ident, image_size=8, windows=(3, 2)), 2, 3, 2)
    assert (feats - want).abs().max().item() <= 1e-6
    means, stds, meta = _stats("houston")
    raw = torch.from_numpy(O.synthetic_raw_tiles(1, 48, 64, 23)).to(DEV)
    rt = M.RawTiles(raw, means, stds, image_size=8, pad_bands=meta["pad"])
    feats = embed_scene(m, rt, batch_windows=24)
    want = _stitched(m, M.RawTiles(raw, means, stds, image_size=8, pad_bands=meta["pad"], windows=(8, 8)), 1, 8, 8)
    assert (feats - want).abs().max().item() <= 1e-6


def test_bf16_embedding_close_to_fp32():
    means, stds, _ = _stats("enmap")
    raw = torch.from_numpy(np.random.default_rng(11).integers(-400, 12000, (1, 200, 27, 22)).astype(np.int16)).to(DEV)
    rt = M.RawTiles(raw, means, stds, image_size=8, clip=(-2.0, 2.0))
    m32, _, _ = _model(O.ENMAP, 2, 84)
    m16, _, _ = _model(O.ENMAP, 2, 84, precision="bf16")
    f32 = embed_scene(m32, rt, stride=4)
    f16 = embed_scene(m16, rt, stride=4, batch_windows=10)
    assert f16.shape == (1, 96, 27, 22) and f16.dtype == torch.float32 and torch.isfinite(f16).all()
    err = rel_l2(f16, f32)
    print(f"bf16 vs fp32 rel-l2 {err:.2e}")
    assert err <= 1e-2


@pytest.mark.parametrize("head", ["pixelwise", "spectral_mlp_head"])
def test_heads_predict_scene_refuses_embed_like_the_default_head(head):
    """The head is not run: a model with another head and the same encoder weights gives the same features, bit for bit (the eval
    forward has no float atomics)."""
    m, _, sd = _model(O.HOUSTON, 2, 85)
    other = M.ViTSpatialSpectral(image_size=8, spatial_patch_size=1, spectral_patch_size=10, num_classes=20, dim=96, depth=2, heads=8,
                                 mlp_dim=64, channels=50, spectral_pos_embed=False, **{head: True})
    missing, unexpected = other.load_state_dict({k: v for k, v in sd.items() if not k.startswith("mlp_head")}, strict=False)
    assert all(k.startswith("mlp_head") for k in missing) and not unexpected
    other = other.to(DEV)
    cube = torch.randn(1, 50, 13, 10, device=DEV)
    assert torch.equal(embed_scene(other, cube, stride=2), embed_scene(m, cube, stride=2))


def test_embed_scene_argument_checks():
    m, _, _ = _model(O.HOUSTON, 1, 86)
    means, stds, _ = _stats("houston")
    raw = torch.zeros(1, 48, 20, 20, dtype=torch.int16, device=DEV)
    cube = torch.zeros(1, 50, 20, 20, device=DEV)
    m.train()
    with pytest.raises(ValueError, match="crop"):
        embed_scene(m, M.RawTiles(raw, means, stds, image_size=8, pad_bands=2, crop=(1, 0)))
    with pytest.raises(ValueError, match="smaller"):
        embed_scene(m, torch.zeros(1, 50, 7, 20, device=DEV))
    with pytest.raises(ValueError, match="stride"):
        embed_scene(m, cube, stride=9)
    with pytest.raises(ValueError, match="weight"):
        embed_scene(m, cube, weight=torch.ones(4, 4))
    v1 = M.ViTSpatialSpectral_V1(image_size=8, spatial_patch_size=1, spectral_patch_size=10, num_classes=20, dim=96, depth=1,
                                 heads=8, mlp_dim=64, channels=50).to(DEV)
    for bad in (v1, M.SimMIMSpatialSpectral(encoder=v1, masking_ratio=0.5)):
        with pytest.raises(ValueError, match="ViTSpatialSpectral"):
            embed_scene(bad, cube)
    assert m.training
    embed_scene(m, cube, stride=4)
    assert m.training
    m.eval()
    embed_scene(m, cube, stride=4)
    assert not m.training
    # the one-chunk wrapper checks its tensors before the library does
    tok = torch.zeros(9, 5 * 64, 96, device=DEV)
    acc, wsum = torch.zeros(1, 96, 20, 20, device=DEV), torch.zeros(1, 20, 20, device=DEV)
    for kw in (dict(tokens=tok.double()), dict(tokens=tok[:, :, :48]), dict(acc=acc[:, :48].contiguous()), dict(C=3),
               dict(wsum=wsum[0]), dict(weight=torch.ones(4, 4, device=DEV))):
        a = dict(tokens=tok, acc=acc, wsum=wsum, C=5, weight=None)
        a.update(kw)
        with pytest.raises(ValueError, match="embed_windows"):
            embed_windows(a["tokens"], a["acc"], a["wsum"], C=a["C"], p1=1, stride=(8, 8), grid=(3, 3), first=0, weight=a["weight"])
