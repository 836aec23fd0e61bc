"""Checkpoint writer / loader in the reference's pickle layout (SURVEY.md Appendix B, 8(f) rank 4).
CPU only.  The reference itself is not needed: what it must be able to read is checked on the file, against golden
outputs of the unmodified reference (tests/golden/)."""
import pickletools
import zipfile

import torch

import maskedsst_b200 as M
from oracle import maskedsst_oracle as O
from src.utils import Dotdict, load_checkpoint, save_pretrain_checkpoint, save_finetune_checkpoint
from tests.helpers import gold, rel_l2


def _encoder(nc=20):
    return M.ViTSpatialSpectral(image_size=8, spatial_patch_size=1, spectral_patch_size=10, num_classes=nc, dim=96, depth=4, heads=8,
                                mlp_dim=64, channels=50, spectral_pos_embed=False, blockwise_patch_embed=True)


def _write_pretrain(path):
    spec = O.Spec(**O.HOUSTON)
    sim = M.SimMIMSpatialSpectral(encoder=_encoder(), masking_ratio=0.7, mask_patch_size=4, tube_masking=True,
                                  to_pixels_per_spectral_block=True)
    sd = O.synthetic_state_dict(spec, seed=77, simmim=True)
    sim.load_state_dict(sd, strict=True)
    cfg = Dotdict(dict(run_id="t", encoder_name="ViTSpatialSpectral", device=torch.device("cpu"), lr=0.008, image_size=8))
    save_pretrain_checkpoint(path, sim, cfg, [0.5, 0.25], 0.008, O.synthetic_cube(spec, 2, seed=1))
    return sd


def test_pretrain_checkpoint_layout_and_own_loader(tmp_path):
    path = str(tmp_path / "model_ViTSpatialSpectral_ep1.pth")
    sd = _write_pretrain(path)
    ck = torch.load(path, map_location="cpu", weights_only=False)
    assert sorted(ck) == ["config", "input", "losses", "lr_current", "model_state_dict", "transformer_input"]   # pretrain.py:137-144
    assert isinstance(ck["config"], Dotdict) and ck["config"].device == torch.device("cpu")
    assert list(ck["model_state_dict"]) == [k for k, _ in O.state_dict_layout(O.Spec(**O.HOUSTON), True)] or \
        set(ck["model_state_dict"]) == set(sd)
    assert ck["losses"].shape == (2,) and ck["input"].shape == (2, 50, 8, 8)
    enc = _encoder(nc=7)                       # a different class count: the fresh head must survive the load
    head_w = enc.mlp_head[1].weight.detach().clone()
    cfg = Dotdict(dict(checkpoint_path=path, patch_sub=0, image_size=8))
    load_checkpoint(cfg, enc, "mlp_head", "cpu")
    got = enc.state_dict()
    for k, v in sd.items():
        if k.startswith("encoder.") and "mlp_head.1" not in k:
            assert torch.equal(got[k[len("encoder."):]], v), k
    assert torch.equal(enc.mlp_head[1].weight, head_w)


def test_finetune_checkpoint_layout(tmp_path):
    path = str(tmp_path / "best_vit.pth")
    enc = _encoder()
    save_finetune_checkpoint(path, enc, Dotdict(dict(lr=0.0005, method_name="vit")), 0.0005, 3)
    ck = torch.load(path, map_location="cpu", weights_only=True)      # plain dict + tensors only (src/utils.py:589-594)
    assert sorted(ck) == ["config", "epoch", "lr_current", "model_state_dict"] and ck["config"] == {"lr": 0.0005, "method_name": "vit"}
    enc2 = _encoder()
    enc2.load_state_dict(ck["model_state_dict"], strict=True)


def test_reference_loader_reads_our_pretrain_checkpoint(tmp_path):
    """What the unmodified reference needs to read a checkpoint written by save_pretrain_checkpoint (SURVEY C8, Appendix B):
    the pickle names no class outside torch, the standard library and the reference's own src.utils.Dotdict; the stripped
    'encoder.*' keys are exactly the reference encoder's layout, so its strict load_state_dict (src/utils.py:311) succeeds;
    and the weights read back the way load_checkpoint (src/utils.py:276-313) reads them give the logits the unmodified
    reference computed on those weights (tests/golden/houston_encoder.npz, tolerance 1e-5)."""
    spec = O.Spec(**O.HOUSTON)
    enc_sd = O.synthetic_state_dict(spec, seed=5)               # the weights of the golden houston_encoder case
    sd = O.synthetic_state_dict(spec, seed=77, simmim=True)
    sd.update({"encoder." + k: v for k, v in enc_sd.items()})
    sim = M.SimMIMSpatialSpectral(encoder=_encoder(), masking_ratio=0.7, mask_patch_size=4, tube_masking=True,
                                  to_pixels_per_spectral_block=True)
    sim.load_state_dict(sd, strict=True)
    path = str(tmp_path / "ck.pth")
    cfg = Dotdict(dict(run_id="t", encoder_name="ViTSpatialSpectral", device=torch.device("cpu"), lr=0.008, image_size=8))
    save_pretrain_checkpoint(path, sim, cfg, [0.5, 0.25], 0.008, O.synthetic_cube(spec, 2, seed=1))

    with zipfile.ZipFile(path) as z:
        pkl = z.read(next(n for n in z.namelist() if n.endswith("/data.pkl")))
    ops = [(op.name, arg) for op, arg, _ in pickletools.genops(pkl)]
    assert not any(name == "STACK_GLOBAL" for name, _ in ops)   # every class reference is a GLOBAL opcode checked below
    classes = {tuple(arg.split(" ", 1)) for name, arg in ops if name == "GLOBAL"}
    assert ("src.utils", "Dotdict") in classes
    foreign = [c for c in classes if c != ("src.utils", "Dotdict") and c[0].split(".")[0] not in ("torch", "collections", "builtins")]
    assert not foreign, foreign

    ck = torch.load(path, map_location="cpu", weights_only=False)
    stripped = {k[len("encoder."):]: tuple(v.shape) for k, v in ck["model_state_dict"].items() if k.startswith("encoder.")}
    assert stripped == dict(O.state_dict_layout(spec, False))

    enc = _encoder()
    with torch.no_grad():                                       # load_checkpoint keeps the fresh head: make it the golden one
        enc.mlp_head[1].weight.copy_(enc_sd["mlp_head.1.weight"])
        enc.mlp_head[1].bias.copy_(enc_sd["mlp_head.1.bias"])
    load_checkpoint(Dotdict(dict(checkpoint_path=path, patch_sub=0, image_size=8)), enc, "mlp_head", "cpu")
    x = O.synthetic_cube(spec, 2, seed=5, zero_pad_bands=2)
    assert rel_l2(O.encoder_forward(x, enc.state_dict(), spec), gold("houston_encoder")["logits"]) < 1e-5
