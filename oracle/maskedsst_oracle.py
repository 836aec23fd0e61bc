"""CPU oracle for the MaskedSST ViTSpatialSpectral / SimMIM hot path.

TEST INFRASTRUCTURE ONLY.  Nothing in ``maskedsst_b200/`` (the product) may import this
file; only ``tests/``, ``__graft_entry__.smoke()`` and ``bench.py``'s CPU-baseline leg do,
and there only as the checker.

This is a *functional restatement* (plain tensors + a state_dict, no nn.Module) of the
reference algorithm, written from the reference's behaviour, each function citing the
reference file:line it follows (paths relative to the upstream repo root).  It runs on
CPU in fp32 (or fp64 when ``dtype=torch.float64`` is passed) through stock torch ops.

Parity pin: ``tests/golden/make_golden.py`` imports the *unmodified reference modules*
in the build container, feeds them ``synthetic_state_dict``/``synthetic_cube`` and stores
their outputs under ``tests/golden/*.npz``; ``tests/test_oracle_golden.py`` checks this
file against those vectors (the reference has no tests / golden vectors of its own,
SURVEY.md §4, so vectors generated from the reference itself are the pin).
"""
from __future__ import annotations

import math
from dataclasses import dataclass, field
from typing import Dict, List, Optional, Sequence, Tuple

import numpy as np
import torch
import torch.nn.functional as F


# --------------------------------------------------------------------------------------
# configuration
# --------------------------------------------------------------------------------------
@dataclass
class Spec:
    """Constructor arguments of ViTSpatialSpectral (src/vit_spatial_spectral.py:257-301)."""

    image_size: int = 8
    spatial_patch_size: int = 1
    spectral_patch_size: int = 10
    channels: int = 50
    num_classes: int = 20
    dim: int = 96
    depth: int = 4
    heads: int = 8
    dim_head: int = 64
    mlp_dim: int = 64
    spectral_pos_embed: bool = False
    blockwise_patch_embed: bool = True
    spectral_only: bool = False
    spectral_pos: Optional[Sequence[int]] = None
    v1: bool = False           # legacy ViTSpatialSpectral_V1 (vit_spatial_spectral.py:600-764)
    v1_merge: str = "avgpool"  # V1 ctor argument `merge`; "linear" only adds the (unused) merge.fc parameters

    @property
    def C(self) -> int:  # spectral blocks, :326
        return self.channels // self.spectral_patch_size

    @property
    def S_sqrt(self) -> int:  # :324
        return self.image_size // self.spatial_patch_size

    @property
    def S(self) -> int:  # :325
        return self.S_sqrt ** 2

    @property
    def T(self) -> int:  # :328
        return self.C * self.S

    @property
    def P(self) -> int:  # pixels per patch, :307-309
        return self.spectral_patch_size * self.spatial_patch_size ** 2

    def pos(self) -> np.ndarray:
        return np.arange(self.C) if self.spectral_pos is None else np.asarray(self.spectral_pos)


HOUSTON = dict(channels=50, num_classes=20)   # configs/config.yaml:12-16
ENMAP = dict(channels=200, num_classes=8)     # configs/config.yaml:3-6


# --------------------------------------------------------------------------------------
# sin-cos tables (src/pos_embed.py:16-63) -- float64 like the reference (np.float)
# --------------------------------------------------------------------------------------
def sincos_1d(embed_dim: int, pos: np.ndarray) -> np.ndarray:
    """src/pos_embed.py:44-63: [sin(pos*w) | cos(pos*w)], w_k = 10000^(-k/(D/2))."""
    assert embed_dim % 2 == 0
    half = embed_dim // 2
    omega = 1.0 / 10000 ** (np.arange(half, dtype=np.float64) / half)
    ang = np.asarray(pos, dtype=np.float64).reshape(-1)[:, None] * omega[None, :]
    return np.concatenate([np.sin(ang), np.cos(ang)], axis=1)


def sincos_2d(embed_dim: int, grid_size: int) -> np.ndarray:
    """src/pos_embed.py:16-41.  meshgrid(w, h) 'w first': the first half of the features
    encodes the column index, the second half the row index."""
    ys, xs = np.meshgrid(np.arange(grid_size, dtype=np.float32),
                         np.arange(grid_size, dtype=np.float32), indexing="ij")
    first = sincos_1d(embed_dim // 2, xs.reshape(-1))   # grid[0] == column coordinate
    second = sincos_1d(embed_dim // 2, ys.reshape(-1))  # grid[1] == row coordinate
    return np.concatenate([first, second], axis=1)


# --------------------------------------------------------------------------------------
# synthetic weights / inputs (deterministic across torch versions: numpy PCG64)
# --------------------------------------------------------------------------------------
def state_dict_layout(spec: Spec, simmim: bool, blockwise_decoder: bool = True) -> List[Tuple[str, Tuple[int, ...]]]:
    """Key/shape list of the reference state_dict (SURVEY.md Appendix B; verified against the
    reference by tests/golden/make_golden.py)."""
    D, I, M, P, C = spec.dim, spec.heads * spec.dim_head, spec.mlp_dim, spec.P, spec.C
    pre = "encoder." if simmim else ""
    out: List[Tuple[str, Tuple[int, ...]]] = []
    if simmim:
        out.append(("mask_token", (D,)))
    if spec.v1:
        # ViTSpatialSpectral_V1 (:640-650, :652): Sequential(Rearrange, LN(P), Linear(P,D), LN(D)), learned table
        out.append((pre + "pos_embedding", (1, spec.T + 1, D)))
        pe = pre + "to_patch_embedding."
        out += [(pe + "1.weight", (P,)), (pe + "1.bias", (P,)), (pe + "2.weight", (D, P)), (pe + "2.bias", (D,)),
                (pe + "3.weight", (D,)), (pe + "3.bias", (D,))]
    elif spec.spectral_pos_embed:
        out.append((pre + "pos_embed", (1, spec.S, D - D // 3)))
        out.append((pre + "channel_embed", (1, C, D // 3)))
    else:
        out.append((pre + "pos_embedding", (1, spec.T + 1, D)))
    pe = pre + "to_patch_embedding."
    if spec.v1:
        pass
    elif spec.blockwise_patch_embed:
        out += [(pe + "pre_norm.weight", (P,)), (pe + "pre_norm.bias", (P,)),
                (pe + "post_norm.weight", (D,)), (pe + "post_norm.bias", (D,))]
        for i in range(C):
            out += [(pe + f"blockwise_embed.{i}.weight", (D, P)), (pe + f"blockwise_embed.{i}.bias", (D,))]
    else:
        out += [(pe + "to_patch.1.weight", (P,)), (pe + "to_patch.1.bias", (P,)),
                (pe + "embed.0.weight", (D, P)), (pe + "embed.0.bias", (D,)),
                (pe + "embed.1.weight", (D,)), (pe + "embed.1.bias", (D,))]
    for t in ([1] if spec.spectral_only else [1, 3]):
        for l in range(spec.depth):
            b = pre + f"spatial_spectral_transformer.{t}.layers.{l}."
            out += [(b + "0.norm.weight", (D,)), (b + "0.norm.bias", (D,)),
                    (b + "0.fn.to_qkv.weight", (3 * I, D)),
                    (b + "0.fn.to_out.0.weight", (D, I)), (b + "0.fn.to_out.0.bias", (D,)),
                    (b + "1.norm.weight", (D,)), (b + "1.norm.bias", (D,)),
                    (b + "1.fn.net.0.weight", (M, D)), (b + "1.fn.net.0.bias", (M,)),
                    (b + "1.fn.net.3.weight", (D, M)), (b + "1.fn.net.3.bias", (D,))]
    if spec.v1 and spec.v1_merge == "linear":   # LinearMerge.fc (:579-588); never called by V1.forward
        out += [(pre + "merge.fc.weight", (D, 2 * D)), (pre + "merge.fc.bias", (D,))]
    out += [(pre + "mlp_head.0.weight", (D,)), (pre + "mlp_head.0.bias", (D,)),
            (pre + "mlp_head.1.weight", (spec.num_classes * spec.spatial_patch_size ** 2, D)),
            (pre + "mlp_head.1.bias", (spec.num_classes * spec.spatial_patch_size ** 2,))]
    if simmim:
        if blockwise_decoder:
            for i in range(C):
                out += [(f"to_pixels.layers.{i}.weight", (P, D)), (f"to_pixels.layers.{i}.bias", (P,))]
        else:
            out += [("to_pixels.weight", (P, D)), ("to_pixels.bias", (P,))]
    return out


def synthetic_state_dict(spec: Spec, seed: int = 5, simmim: bool = False,
                         blockwise_decoder: bool = True) -> Dict[str, torch.Tensor]:
    """Random checkpoint stand-in (the shipped .pth blobs are absent, SURVEY.md §0.6).
    Linear weights ~ U(-1/sqrt(fan_in), 1/sqrt(fan_in)) like nn.Linear's default, LayerNorm
    weights 1 + 0.1 n, biases 0.1 n, learned tables ~ N(0,1) (vit_spatial_spectral.py:383-389);
    sin-cos tables when spectral_pos_embed (vit_spatial_spectral.py:352-381)."""
    rng = np.random.Generator(np.random.PCG64(seed))
    sd: Dict[str, torch.Tensor] = {}
    for key, shape in state_dict_layout(spec, simmim, blockwise_decoder):
        leaf = key.split(".")[-1]
        if key.endswith("pos_embed") and spec.spectral_pos_embed:
            arr = sincos_2d(shape[-1], spec.S_sqrt)[None] + 0.02 * rng.standard_normal(shape)
        elif key.endswith("channel_embed"):
            arr = sincos_1d(shape[-1], spec.pos())[None] + 0.02 * rng.standard_normal(shape)
        elif ("norm" in key or "mlp_head.0" in key or "to_patch.1" in key or "embed.1" in key
              or key.endswith(("to_patch_embedding.1.weight", "to_patch_embedding.1.bias",
                               "to_patch_embedding.3.weight", "to_patch_embedding.3.bias"))):
            arr = (1.0 if leaf == "weight" else 0.0) + 0.1 * rng.standard_normal(shape)
        elif leaf == "weight" and len(shape) == 2:
            bound = 1.0 / math.sqrt(shape[1])
            arr = rng.uniform(-bound, bound, shape)
        elif leaf == "bias":
            arr = 0.1 * rng.standard_normal(shape)
        else:  # pos_embedding, mask_token
            arr = rng.standard_normal(shape)
        sd[key] = torch.from_numpy(np.ascontiguousarray(arr, dtype=np.float32))
    return sd


def synthetic_cube(spec: Spec, batch: int, seed: int = 5, zero_pad_bands: int = 0) -> torch.Tensor:
    """Band-standardised stand-in cube [B, channels, H, W]; the last ``zero_pad_bands`` bands are
    zero like Houston's 48->50 padding (src/data_houston2018.py:268-269)."""
    rng = np.random.Generator(np.random.PCG64(seed + 1000))
    x = rng.standard_normal((batch, spec.channels, spec.image_size, spec.image_size)).astype(np.float32)
    if zero_pad_bands:
        x[:, spec.channels - zero_pad_bands:] = 0.0
    return torch.from_numpy(x)


def synthetic_raw_tiles(batch: int, bands: int, size: int = 64, seed: int = 21) -> np.ndarray:
    """Stand-in for raw sensor tiles [B, bands, size, size] int16 (reflectance * 10000 range, with some negatives and
    saturated values so a clip has something to do)."""
    rng = np.random.Generator(np.random.PCG64(seed + 2000))
    return rng.integers(-400, 12000, (batch, bands, size, size)).astype(np.int16)


def input_pipeline(raw: np.ndarray, means, stds, image_size: int, crop=(0, 0), pad_bands: int = 0, clip=None) -> torch.Tensor:
    """The reference's path from a raw tile to the model's cube:
      StandardizeEnMAP / StandardizeHouston2018.__call__: (x - means[:,None,None]) / stds[:,None,None] on the numpy array
        -> float64 (src/data_enmap.py:454-457, src/data_houston2018.py:442-445);
      ToTensor: torch.Tensor(x).to(float32) -> one rounding to fp32 (src/data_enmap.py:517-522);
      EnMAP: torch.clip(img, clip[0], clip[1]) on the standardised values (src/data_enmap.py:303-304);
      Houston: F.pad 48 -> 50 zero bands after standardisation (src/data_houston2018.py:268-269);
      one crop window img[:, :, x:x+s, y:y+s] for the whole batch (pretrain.py:99-107)."""
    m = np.asarray(means, dtype=np.float64)[None, :, None, None]
    sd = np.asarray(stds, dtype=np.float64)[None, :, None, None]
    x = torch.from_numpy(((raw - m) / sd)).to(torch.float32)
    if clip is not None:
        x = torch.clip(x, min=clip[0], max=clip[1])
    if pad_bands:
        x = F.pad(x, (0, 0, 0, 0, 0, pad_bands), "constant", 0)
    a, b = crop
    return x[:, :, a: a + image_size, b: b + image_size].contiguous()


# --------------------------------------------------------------------------------------
# forward pieces
# --------------------------------------------------------------------------------------
def to_patch(img: torch.Tensor, spec: Spec) -> torch.Tensor:
    """'b (c p0) (h p1) (w p2) -> b c (h w) (p0 p1 p2)' (vit_spatial_spectral.py:197-202)."""
    B = img.shape[0]
    p0, p1 = spec.spectral_patch_size, spec.spatial_patch_size
    g = spec.S_sqrt
    x = img.reshape(B, spec.C, p0, g, p1, g, p1)
    x = x.permute(0, 1, 3, 5, 2, 4, 6)  # b c h w p0 p1 p2
    return x.reshape(B, spec.C, spec.S, spec.P)


def _ln(x, w, b, eps=1e-5):
    """nn.LayerNorm: biased variance over the last dim, eps inside the sqrt."""
    mu = x.mean(-1, keepdim=True)
    var = ((x - mu) ** 2).mean(-1, keepdim=True)
    return (x - mu) / torch.sqrt(var + eps) * w + b


def embed(patches: torch.Tensor, sd, spec: Spec, pre: str = "") -> torch.Tensor:
    """BlockwisePatchEmbedding.embed (vit_spatial_spectral.py:210-222) / PatchEmbed (:232-253).
    patches [B,C,S,P] raw -> tokens [B,T,D]."""
    pe = pre + "to_patch_embedding."
    B = patches.shape[0]
    if spec.v1:   # ViTSpatialSpectral_V1.to_patch_embedding[1:] (:646-649)
        h = _ln(patches.reshape(B, spec.T, spec.P), sd[pe + "1.weight"], sd[pe + "1.bias"])
        y = h @ sd[pe + "2.weight"].T + sd[pe + "2.bias"]
        return _ln(y, sd[pe + "3.weight"], sd[pe + "3.bias"])
    if spec.blockwise_patch_embed:
        h = _ln(patches, sd[pe + "pre_norm.weight"], sd[pe + "pre_norm.bias"])
        W = torch.stack([sd[pe + f"blockwise_embed.{i}.weight"] for i in range(spec.C)])  # [C,D,P]
        bb = torch.stack([sd[pe + f"blockwise_embed.{i}.bias"] for i in range(spec.C)])   # [C,D]
        y = torch.einsum("bcsp,cdp->bcsd", h, W) + bb[None, :, None, :]
        y = y.reshape(B, spec.T, spec.dim)
        return _ln(y, sd[pe + "post_norm.weight"], sd[pe + "post_norm.bias"])
    h = _ln(patches.reshape(B, spec.T, spec.P), sd[pe + "to_patch.1.weight"], sd[pe + "to_patch.1.bias"])
    y = h @ sd[pe + "embed.0.weight"].T + sd[pe + "embed.0.bias"]
    return _ln(y, sd[pe + "embed.1.weight"], sd[pe + "embed.1.bias"])


def pos_table(sd, spec: Spec, pre: str = "") -> torch.Tensor:
    """[1,T,D] positional table: learned rows [0,T) (vit_spatial_spectral.py:525) or
    cat(spatial[.., :2D/3], spectral[.., D/3]) broadcast (get_pos_embeddings, :501-516)."""
    if not spec.spectral_pos_embed:
        return sd[pre + "pos_embedding"][:, : spec.T]
    pe = sd[pre + "pos_embed"][:, None, :, :].expand(1, spec.C, spec.S, -1)
    ce = sd[pre + "channel_embed"][:, :, None, :].expand(1, spec.C, spec.S, -1)
    return torch.cat([pe, ce], dim=-1).reshape(1, spec.T, spec.dim)


def gelu_erf(x):
    """nn.GELU() default = exact erf form (vit_spatial_spectral.py:37)."""
    return 0.5 * x * (1.0 + torch.erf(x / math.sqrt(2.0)))


SITE_EMB, SITE_LAYER_BASE = 1, 16   # dropout site ids: emb-dropout; layer l of a stack uses base + 8 l + (0 probs, 1 attn out,
                                   # 2 MLP hidden, 3 MLP out); the spectral stack after a spatial one starts at 16 + 8 depth


def _dropout(t, drop, site, layout):
    """drop: a float p = training-mode torch dropout (the CPU-baseline timing leg); or a callable drop(t, site, layout) that
    returns t * mask, so a test can apply the exact masks of a kernel run (layout: "spatial" / "spectral" stack, "emb")."""
    return drop(t, site, layout) if callable(drop) else F.dropout(t, drop)


def attention(x, sd, base: str, heads: int, dim_head: int, drop=0.0, site: int = SITE_LAYER_BASE, layout=None):
    """Attention.forward (vit_spatial_spectral.py:67-78). x [n,N,D].  drop (see _dropout): dropout on the
    probabilities (:74, site) and the output projection (:62, site + 1)."""
    n, N, D = x.shape
    qkv = x @ sd[base + "to_qkv.weight"].T
    q, k, v = qkv.split(heads * dim_head, dim=-1)
    sh = lambda t: t.reshape(n, N, heads, dim_head).permute(0, 2, 1, 3)
    q, k, v = sh(q), sh(k), sh(v)
    dots = (q @ k.transpose(-1, -2)) * dim_head ** -0.5
    p = _dropout(torch.softmax(dots, dim=-1), drop, site, layout)
    o = (p @ v).permute(0, 2, 1, 3).reshape(n, N, heads * dim_head)
    return _dropout(o @ sd[base + "to_out.0.weight"].T + sd[base + "to_out.0.bias"], drop, site + 1, layout)


def transformer(x, sd, base: str, spec: Spec, drop=0.0, layout=None, site_base: int = SITE_LAYER_BASE):
    """Transformer.forward (vit_spatial_spectral.py:100-104): pre-norm attn + pre-norm MLP, no final norm."""
    for l in range(spec.depth):
        b = base + f"layers.{l}."
        site = site_base + 8 * l
        h = _ln(x, sd[b + "0.norm.weight"], sd[b + "0.norm.bias"])
        x = attention(h, sd, b + "0.fn.", spec.heads, spec.dim_head, drop, site, layout) + x
        h = _ln(x, sd[b + "1.norm.weight"], sd[b + "1.norm.bias"])
        u = _dropout(gelu_erf(h @ sd[b + "1.fn.net.0.weight"].T + sd[b + "1.fn.net.0.bias"]), drop, site + 2, layout)
        x = _dropout(u @ sd[b + "1.fn.net.3.weight"].T + sd[b + "1.fn.net.3.bias"], drop, site + 3, layout) + x
    return x


def transformer_forward(tokens, sd, spec: Spec, pre: str = "", drop=0.0):
    """spatial_spectral_transformer (vit_spatial_spectral.py:393-431). tokens [B,T,D], t = c*S + s."""
    B = tokens.shape[0]
    C, S, D = spec.C, spec.S, spec.dim
    base = pre + "spatial_spectral_transformer."
    x = tokens
    if not spec.spectral_only:
        x = transformer(x.reshape(B * C, S, D), sd, base + "1.", spec, drop, "spatial")
        x = x.reshape(B, C, S, D).permute(0, 2, 1, 3).reshape(B * S, C, D)
        x = transformer(x, sd, base + "3.", spec, drop, "spectral", SITE_LAYER_BASE + 8 * spec.depth)
    else:
        x = x.reshape(B, C, S, D).permute(0, 2, 1, 3).reshape(B * S, C, D)
        x = transformer(x, sd, base + "1.", spec, drop, "spectral")
    return x.reshape(B, S, C, D).permute(0, 2, 1, 3).reshape(B, spec.T, D)


def head(x, sd, spec: Spec, pre: str = ""):
    """mean over spectral blocks + default mlp_head (vit_spatial_spectral.py:550-562, 481-493).
    x [B,T,D] -> logits [B, nc, H, W]."""
    B = x.shape[0]
    g, p = spec.S_sqrt, spec.spatial_patch_size
    z = x.reshape(B, spec.C, g, g, spec.dim).mean(dim=1)
    z = _ln(z, sd[pre + "mlp_head.0.weight"], sd[pre + "mlp_head.0.bias"])
    y = z @ sd[pre + "mlp_head.1.weight"].T + sd[pre + "mlp_head.1.bias"]     # [B,g,g,p*p*nc]
    y = y.reshape(B, g, g, p, p, spec.num_classes).permute(0, 1, 3, 2, 4, 5)
    y = y.reshape(B, g * p, g * p, spec.num_classes)
    return y.permute(0, 3, 1, 2)


def encoder_tokens(img, sd, spec: Spec, pre: str = ""):
    """to_patch_embedding + pos-embed add (forward_features :518-528), emb-dropout off."""
    return embed(to_patch(img, spec), sd, spec, pre) + pos_table(sd, spec, pre)


def encoder_forward(img, sd, spec: Spec, pre: str = ""):
    """ViTSpatialSpectral.forward in eval mode (vit_spatial_spectral.py:536-564)."""
    return head(transformer_forward(encoder_tokens(img, sd, spec, pre), sd, spec, pre), sd, spec, pre)


def simmim_forward(img, sd, spec: Spec, bool_mask: torch.Tensor, idx: torch.Tensor,
                   blockwise_decoder: bool = True, return_parts: bool = False, drop=0.0,
                   intermediate_losses: bool = False):
    """SimMIMSpatialSpectral.forward (vit_simmim_original.py:203-340) with the mask pair supplied
    from outside (the pair may be mutually inconsistent, SURVEY.md C3).  Dropout off; the SimMIM
    path never applies emb-dropout (C5).  loss = mean|pred-target| / num_masked (C4)."""
    pre = "encoder."
    B = img.shape[0]
    patches = to_patch(img, spec)
    tokens = embed(patches, sd, spec, pre)
    if spec.blockwise_patch_embed or spec.v1:
        target = patches.reshape(B, spec.T, spec.P)                 # raw pixels (C6); V1: to_patch = Rearrange only (:174-178)
    else:
        pe = pre + "to_patch_embedding."
        target = _ln(patches.reshape(B, spec.T, spec.P), sd[pe + "to_patch.1.weight"], sd[pe + "to_patch.1.bias"])
    if spec.v1:
        pos = sd[pre + "pos_embedding"][:, 1: spec.T + 1]            # V1 + SimMIM reads rows [1, T] (:233, C11)
    else:
        pos = pos_table(sd, spec, pre)
    tokens = tokens + pos
    mask_tokens = sd["mask_token"][None, None, :] + pos
    tokens = torch.where(bool_mask[..., None], mask_tokens, tokens)
    enc = transformer_forward(tokens, sd, spec, pre, drop)
    nm = idx.shape[1]
    br = torch.arange(B, device=idx.device)[:, None]
    sel = enc[br, idx]                                              # [B,nm,D]
    if blockwise_decoder:
        blk = idx // spec.S                                         # arange(C).repeat_interleave(S)[idx]
        W = torch.stack([sd[f"to_pixels.layers.{i}.weight"] for i in range(spec.C)])
        bb = torch.stack([sd[f"to_pixels.layers.{i}.bias"] for i in range(spec.C)])
        pred = torch.einsum("bnd,bnpd->bnp", sel, W[blk]) + bb[blk]
    else:
        pred = sel @ sd["to_pixels.weight"].T + sd["to_pixels.bias"]
    tgt = target[br, idx]
    loss = (pred - tgt).abs().mean() / nm
    if intermediate_losses:
        # :311-338 with a V1 encoder: the "spatial" and "spectral" representations V1.transformer_forward returns are the
        # final one (:735-744 `return x, x, x`), so the same term is accumulated three times: 0.0 + a + a + a
        loss = (loss + loss) + loss
    if return_parts:
        return loss, tokens, enc, pred
    return loss


def cross_entropy(logits, labels, ignore_index: int = -1):
    """nn.CrossEntropyLoss(ignore_index=-1) (finetune.py:136): mean NLL over valid pixels."""
    lp = torch.log_softmax(logits, dim=1)
    valid = labels != ignore_index
    safe = labels.clamp(min=0)
    nll = -lp.gather(1, safe[:, None]).squeeze(1)
    return (nll * valid).sum() / valid.sum()


# --------------------------------------------------------------------------------------
# mask generation (host, numpy global RNG -- bit-compatible with the reference)
# --------------------------------------------------------------------------------------
class MaskGen:
    """MaskGenerator (vit_simmim_original.py:343-416).  Draws from numpy's *global* RNG exactly
    like the reference (np.random.permutation), so np.random.seed(s) reproduces its masks."""

    def __init__(self, input_size, mask_patch_size, model_patch_size, mask_ratio):
        self.rand = input_size // mask_patch_size
        self.scale = mask_patch_size // model_patch_size
        self.cells = self.rand ** 2
        self.count = int(np.ceil(self.cells * mask_ratio))

    def one(self) -> np.ndarray:
        m = np.zeros(self.cells, dtype=bool)
        m[np.random.permutation(self.cells)[: self.count]] = True
        m = m.reshape(self.rand, self.rand)
        return m.repeat(self.scale, axis=0).repeat(self.scale, axis=1)

    @staticmethod
    def indices(flat: np.ndarray, num_masked: int) -> np.ndarray:
        """bool_mask_to_indices (:372-382): column ids of nonzero(), sliced in strides of
        num_masked regardless of how many are set per row (the C3 quirk)."""
        cols = np.nonzero(flat)[1]
        B = flat.shape[0]
        return np.stack([cols[num_masked * b: num_masked * (b + 1)] for b in range(B)]).astype(np.int64)

    def batch(self, B: int, C: int, num_masked: int, tube: bool):
        if tube:   # get_batch_tube_masked :402-416
            m = np.stack([self.one() for _ in range(B)])[:, None].repeat(C, axis=1)
        else:      # get_batch :384-400
            m = np.stack([self.one() for _ in range(B * C)]).reshape(B, C, *([self.rand * self.scale] * 2))
        flat = m.reshape(B, -1)
        return torch.from_numpy(flat), torch.from_numpy(self.indices(flat, num_masked))


# --------------------------------------------------------------------------------------
# optimiser update rules (torch.optim.AdamW / Adam as used by src/utils.py:36-44, finetune.py:133)
# --------------------------------------------------------------------------------------
def adam_step(p, g, m, v, step: int, lr: float, beta1=0.9, beta2=0.999, eps=1e-8,
              weight_decay=0.0, decoupled=True, clamp: Optional[float] = None, grad_scale: float = 1.0):
    """One update, returns (p, m, v).  clamp = elementwise grad clamp of pretrain.py:71-73."""
    g = g * grad_scale
    if clamp is not None:
        g = g.clamp(-clamp, clamp)
    if decoupled:
        p = p * (1.0 - lr * weight_decay)
    else:
        g = g + weight_decay * p
    m = beta1 * m + (1 - beta1) * g
    v = beta2 * v + (1 - beta2) * g * g
    bc1 = 1 - beta1 ** step
    bc2 = 1 - beta2 ** step
    denom = v.sqrt() / math.sqrt(bc2) + eps
    p = p - (lr / bc1) * m / denom
    return p, m, v
