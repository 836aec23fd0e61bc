"""GPU parity (fp32 mode): CUDA path through the nn.Module surface / C-ABI vs the CPU oracle and the golden
vectors generated from the unmodified reference.  Tolerances: logits / loss rel-err <= 1e-5 (north star, fp32 mode);
gradients <= 1e-4 on per-tensor summaries (they pass through fp32 atomics in a different summation order)."""
import json
import numpy as np
import pytest
import torch

import maskedsst_b200 as M
from maskedsst_b200 import ops
from oracle import maskedsst_oracle as O
from tests.helpers import gold, rel_l2, grad_rows, check_grad_rows

pytestmark = pytest.mark.gpu
DEV = "cuda"
TOL = 1e-5
GTOL = 1e-4


def make_encoder(spec, dropout=0.0):
    return M.ViTSpatialSpectral(
        image_size=spec.image_size, spatial_patch_size=spec.spatial_patch_size, spectral_patch_size=spec.spectral_patch_size,
        num_classes=spec.num_classes, dim=spec.dim, depth=spec.depth, heads=spec.heads, dim_head=spec.dim_head, mlp_dim=spec.mlp_dim,
        dropout=dropout, emb_dropout=dropout, channels=spec.channels, spectral_pos_embed=spec.spectral_pos_embed,
        blockwise_patch_embed=spec.blockwise_patch_embed, spectral_pos=spec.pos(), spectral_only=spec.spectral_only)


@pytest.mark.parametrize("name,kw,zero_pad,B,seed", [
    ("houston_encoder", dict(**O.HOUSTON), 2, 2, 5),
    ("enmap_encoder", dict(**O.ENMAP), 0, 1, 6),
    ("enmap_encoder_spectralpos", dict(**O.ENMAP, spectral_pos_embed=True), 0, 1, 7),
    ("houston_encoder_spectral_only", dict(**O.HOUSTON, spectral_only=True), 2, 2, 8),
])
def test_encoder_vs_reference_golden(name, kw, zero_pad, B, seed):
    g = gold(name)
    spec = O.Spec(**kw)
    m = make_encoder(spec).eval()
    m.load_state_dict(O.synthetic_state_dict(spec, seed=seed), strict=True)
    m = m.to(DEV)
    x = O.synthetic_cube(spec, B, seed=seed, zero_pad_bands=zero_pad).to(DEV)
    st = int(g["token_stride"])
    with torch.no_grad():
        tok = m.to_patch_embedding(x)
        feats = m.forward_features(x)
        logits = m(x)
    assert rel_l2(tok[:, ::st], g["tokens"]) < TOL
    assert rel_l2(feats[:, ::st], g["features"]) < TOL
    assert rel_l2(logits, g["logits"]) < TOL
    assert logits.shape == g["logits"].shape


@pytest.mark.parametrize("B", [1, 7, 32])
def test_encoder_vs_oracle_batches(B):
    spec = O.Spec(**O.HOUSTON)
    sd = O.synthetic_state_dict(spec, seed=21)
    m = make_encoder(spec).eval()
    m.load_state_dict(sd)
    m.to(DEV)
    x = O.synthetic_cube(spec, B, seed=21, zero_pad_bands=2)
    with torch.no_grad():
        got = m(x.to(DEV))
        want = O.encoder_forward(x, sd, spec)
    assert rel_l2(got, want) < TOL


def test_finetune_ce_step_vs_reference_golden():
    g = gold("houston_finetune_ce")
    spec = O.Spec(**O.HOUSTON)
    m = make_encoder(spec).train()
    m.load_state_dict(O.synthetic_state_dict(spec, seed=9))
    m.to(DEV)
    x = O.synthetic_cube(spec, 3, seed=9).to(DEV)
    labels = torch.from_numpy(g["labels"]).to(DEV)
    logits = m(x)
    loss = M.cross_entropy(logits, labels, ignore_index=-1)
    loss.backward()
    assert rel_l2(logits, g["logits"]) < TOL
    assert abs(loss.item() - float(g["loss"])) < TOL * abs(float(g["loss"]))
    rows = grad_rows([(k, p.grad) for k, p in m.named_parameters() if p.grad is not None])
    check_grad_rows(rows, g["grad_names"], g["grad_rows"], tol=GTOL)
    assert rel_l2(m.mlp_head[1].weight.grad, g["grad_head_w"]) < GTOL
    assert rel_l2(m.to_patch_embedding.pre_norm.weight.grad, g["grad_pre_norm_w"]) < GTOL
    # torch's own CE on our logits gives the same loss (the reference's call, finetune.py:136)
    ref = torch.nn.functional.cross_entropy(logits.detach(), labels, ignore_index=-1)
    assert abs(ref.item() - loss.item()) < 1e-5 * abs(ref.item())


@pytest.mark.parametrize("name,kw", [
    ("houston_simmim_tube", dict(**O.HOUSTON)),
    ("enmap_simmim_block", dict(**O.ENMAP)),
    ("houston_simmim_spectralpos", dict(**O.HOUSTON, spectral_pos_embed=True)),
    ("houston_simmim_patchembed", dict(**O.HOUSTON, blockwise_patch_embed=False)),
])
def test_simmim_step_vs_reference_golden(name, kw):
    g = gold(name)
    meta = json.loads(str(g["meta"]))
    spec = O.Spec(**kw)
    enc = make_encoder(spec)
    m = M.SimMIMSpatialSpectral(encoder=enc, masking_ratio=meta["ratio"], mask_patch_size=meta["mask_patch"],
                                tube_masking=meta["tube"], to_pixels_per_spectral_block=meta["blockwise_decoder"]).train()
    sd = O.synthetic_state_dict(spec, seed=meta["seed"], simmim=True, blockwise_decoder=meta["blockwise_decoder"])
    missing, unexpected = m.load_state_dict(sd, strict=False)
    assert not unexpected and all(k.startswith(("to_patch.", "patch_to_emb.")) for k in missing)
    m.to(DEV)
    x = O.synthetic_cube(spec, meta["B"], seed=meta["seed"], zero_pad_bands=meta["zero_pad"]).to(DEV)
    # the module's own host mask generator reproduces the reference's draw bit for bit
    np.random.seed(meta["seed"])
    mask, idx = m.draw_masks(meta["B"], DEV)
    assert np.array_equal(mask.cpu().numpy(), g["mask"]) and np.array_equal(idx.cpu().numpy(), g["idx"])
    np.random.seed(meta["seed"])
    loss = m(x)
    loss.backward()
    assert abs(loss.item() - float(g["loss"])) < TOL * abs(float(g["loss"]))
    seen, named = set(), []
    for k, p in m.named_parameters():
        if id(p) in seen or p.grad is None:
            continue
        seen.add(id(p)); named.append((k, p.grad))
    rows = grad_rows(named)
    by_name = dict(m.named_parameters(remove_duplicate=False))
    for k in [str(n) for n in g["grad_names"]]:
        if k not in rows and k in by_name and by_name[k].grad is not None:
            rows[k] = grad_rows([(k, by_name[k].grad)])[k]
    check_grad_rows(rows, g["grad_names"], g["grad_rows"], tol=GTOL)
    for k in g.files:
        if k.startswith("grad__"):
            assert rel_l2(by_name[k[6:]].grad, g[k]) < GTOL, k


def test_simmim_external_masks_inconsistent_and_duplicate_indices():
    """C3: the (bool mask, index) pair may disagree and indices may repeat; backward must accumulate."""
    spec = O.Spec(**O.HOUSTON)
    sd = O.synthetic_state_dict(spec, seed=31, simmim=True)
    m = M.SimMIMSpatialSpectral(encoder=make_encoder(spec), masking_ratio=0.7, mask_patch_size=4, tube_masking=True,
                                to_pixels_per_spectral_block=True).train()
    m.load_state_dict(sd)
    m.to(DEV)
    B = 2
    x = O.synthetic_cube(spec, B, seed=31)
    rng = np.random.Generator(np.random.PCG64(3))
    mask = torch.from_numpy(rng.random((B, spec.T)) < 0.6)
    idx = torch.from_numpy(rng.integers(0, spec.T, (B, 100)).astype(np.int64))   # random, with repeats
    idx[:, 1] = idx[:, 0]
    loss = m(x.to(DEV), masks=(mask.to(DEV), idx.to(DEV)))
    loss.backward()
    p = {k: v.clone().requires_grad_(True) for k, v in sd.items()}
    want = O.simmim_forward(x, p, spec, mask, idx)
    want.backward()
    assert abs(loss.item() - want.item()) < TOL * abs(want.item())
    for k, v in m.named_parameters():
        if p[k].grad is None:
            continue
        assert rel_l2(v.grad, p[k].grad) < GTOL or float(p[k].grad.norm()) < 1e-9, k


def _head_variant_oracle(x, sd, spec, kind):
    """pixelwise (vit_spatial_spectral.py:467-479) / spectral_mlp_head (:441-453) heads on top of the oracle features."""
    feats = O.transformer_forward(O.encoder_tokens(x, sd, spec), sd, spec)
    B, g, D, C = x.shape[0], spec.S_sqrt, spec.dim, spec.C
    if kind == "pixelwise":
        z = feats.reshape(B, C, g, g, D).mean(dim=1)
        z = O._ln(z, sd["mlp_head.0.weight"], sd["mlp_head.0.bias"]).reshape(B, g * g * D)
        y = z @ sd["mlp_head.2.weight"].T + sd["mlp_head.2.bias"]
        return y.reshape(B, 1, 1, -1).permute(0, 3, 1, 2).squeeze()
    z = feats.reshape(B, C, g, g, D).permute(0, 2, 3, 1, 4).reshape(B, g, g, C * D)
    z = O._ln(z, sd["mlp_head.0.weight"], sd["mlp_head.0.bias"])
    y = z @ sd["mlp_head.1.weight"].T + sd["mlp_head.1.bias"]
    return y.permute(0, 3, 1, 2)


@pytest.mark.parametrize("kind", ["pixelwise", "spectral_mlp_head"])
def test_head_variants_vs_oracle(kind):
    """second-tier heads (SURVEY a14): LN / Linear through msst_layernorm / msst_linear, forward + gradients."""
    spec = O.Spec(**O.HOUSTON, depth=1)
    torch.manual_seed(0)
    m = M.ViTSpatialSpectral(image_size=8, spatial_patch_size=1, spectral_patch_size=10, num_classes=20, dim=96, depth=1, heads=8,
                             mlp_dim=64, channels=50, spectral_pos_embed=False, pixelwise=kind == "pixelwise",
                             spectral_mlp_head=kind == "spectral_mlp_head")
    sd = {k: v.detach().clone() for k, v in m.state_dict().items()}
    m.to(DEV).train()
    x = O.synthetic_cube(spec, 3, seed=2)
    got = m(x.to(DEV))
    p = {k: v.clone().requires_grad_(True) for k, v in sd.items()}
    want = _head_variant_oracle(x, p, spec, kind)
    assert got.shape == want.shape
    assert rel_l2(got, want) < TOL
    got.square().sum().backward()
    want.square().sum().backward()
    for k, v in m.named_parameters():
        if p[k].grad is not None and float(p[k].grad.norm()) > 1e-9:
            assert rel_l2(v.grad, p[k].grad) < GTOL, k


def test_reference_calling_conventions():
    """to_patch / embed / get_pos_embeddings / forward_features / transformer_forward as the reference's callers use them
    (vit_simmim_original.py:181-182,207-298), and the mask_patch_size == 1 random-mask path (:254-264)."""
    spec = O.Spec(**O.HOUSTON, spectral_pos_embed=True)
    sd = O.synthetic_state_dict(spec, seed=3)
    m = make_encoder(spec).eval()
    m.load_state_dict(sd)
    m.to(DEV)
    x = O.synthetic_cube(spec, 2, seed=3)
    with torch.no_grad():
        patches = m.to_patch_embedding.to_patch(x.to(DEV))
        assert rel_l2(patches, O.to_patch(x, spec)) == 0.0
        tok = m.to_patch_embedding.embed(patches)
        assert rel_l2(tok, O.embed(O.to_patch(x, spec), sd, spec)) < TOL
        assert rel_l2(m.get_pos_embeddings(), O.pos_table(sd, spec)) < 1e-7
        enc = m.transformer_forward(tok + m.get_pos_embeddings())
        assert rel_l2(enc, O.transformer_forward(O.encoder_tokens(x, sd, spec), sd, spec)) < TOL
    sim = M.SimMIMSpatialSpectral(encoder=make_encoder(O.Spec(**O.HOUSTON)), masking_ratio=0.5, mask_patch_size=1).to(DEV).train()
    torch.manual_seed(0)
    mask, idx = sim.draw_masks(4, DEV)
    assert mask.shape == (4, 320) and idx.shape == (4, 160) and int(mask.sum()) == 4 * 160
    assert torch.equal(torch.zeros_like(mask).scatter_(1, idx, True), mask)
    loss = sim(x.to(DEV)[:, :50])
    loss.backward()
    assert torch.isfinite(loss) and sim.mask_token.grad is not None and sim.to_pixels.weight.grad is not None


def test_whole_tile_inference_equals_window_loop():
    from maskedsst_b200.inference import predict_tiles, tile_accuracy
    spec = O.Spec(**O.HOUSTON, depth=1)
    m = make_encoder(spec).eval()
    m.load_state_dict(O.synthetic_state_dict(spec, seed=61))
    m.to(DEV)
    tiles = torch.randn(2, 50, 24, 16, device=DEV)
    full = predict_tiles(m, tiles)
    assert full.shape == (2, 20, 24, 16)
    with torch.no_grad():
        for (i, j) in [(0, 0), (2, 1), (1, 0)]:
            win = m(tiles[:, :, 8 * i:8 * i + 8, 8 * j:8 * j + 8].contiguous())
            assert rel_l2(full[:, :, 8 * i:8 * i + 8, 8 * j:8 * j + 8], win) < 1e-6
    labels = full.argmax(1)
    labels[0, :4] = -1
    acc, n = tile_accuracy(full, labels)
    assert float(acc) == 1.0 and int(n) == 2 * 24 * 16 - 4 * 16


@pytest.mark.parametrize("name,kw", [("houston_v1_intermediate", dict(**O.HOUSTON, v1=True)),
                                     ("houston_v1_linearmerge", dict(**O.HOUSTON, v1=True, v1_merge="linear", depth=2))])
def test_v1_encoder_and_simmim_vs_reference_golden(name, kw):
    """Legacy ViTSpatialSpectral_V1 (reference :600-764): logits, then a SimMIM step with the shared decoder and
    `intermediate_losses` (SURVEY 8(f) rank 4), against vectors from the unmodified reference."""
    g = gold(name)
    meta = json.loads(str(g["meta"]))
    spec = O.Spec(**kw)

    def make():
        return M.ViTSpatialSpectral_V1(image_size=8, spatial_patch_size=1, spectral_patch_size=10, num_classes=spec.num_classes,
                                       dim=spec.dim, depth=spec.depth, heads=spec.heads, mlp_dim=spec.mlp_dim, channels=spec.channels,
                                       merge=meta["merge"])
    enc = make().eval()
    enc.load_state_dict(O.synthetic_state_dict(spec, seed=meta["seed"]), strict=True)
    enc.to(DEV)
    x = O.synthetic_cube(spec, meta["B"], seed=meta["seed"], zero_pad_bands=meta["zero_pad"]).to(DEV)
    with torch.no_grad():
        assert rel_l2(enc(x), g["logits"]) < TOL
    m = M.SimMIMSpatialSpectral(encoder=make(), masking_ratio=0.7, mask_patch_size=4, tube_masking=True,
                                intermediate_losses=meta["intermediate"]).train()
    assert sorted(set(m.state_dict()) - set(dict(O.state_dict_layout(spec, True, False)))) == [str(k) for k in g["extra_keys"]]
    missing, unexpected = m.load_state_dict(O.synthetic_state_dict(spec, seed=meta["seed"] + 100, simmim=True, blockwise_decoder=False),
                                            strict=False)
    assert not unexpected and all(k.startswith("patch_to_emb.") for k in missing)
    m.to(DEV)
    np.random.seed(meta["seed"])
    loss = m(x)
    loss.backward()
    assert abs(loss.item() - float(g["loss"])) < TOL * abs(float(g["loss"]))
    seen, named = set(), []
    for k, p in m.named_parameters():
        if id(p) in seen or p.grad is None:
            continue
        seen.add(id(p)); named.append((k, p.grad))
    check_grad_rows(grad_rows(named), g["grad_names"], g["grad_rows"], tol=GTOL)
    assert rel_l2(m.mask_token.grad, g["grad__mask_token"]) < GTOL
    assert rel_l2(m.to_pixels.weight.grad, g["grad__to_pixels_weight"]) < GTOL
    pg = m.encoder.pos_embedding.grad[0, [0, 1, 2, spec.T]]
    assert float(pg[0].abs().max()) == 0.0 and rel_l2(pg, g["grad__pos_embedding_rows"]) < GTOL
    with pytest.raises(NotImplementedError):
        M.SimMIMSpatialSpectral(encoder=make(), to_pixels_per_spectral_block=True)
    with pytest.raises(NotImplementedError):
        M.SimMIMSpatialSpectral(encoder=make_encoder(O.Spec(**O.HOUSTON)), intermediate_losses=True)
