"""Whole-tile sliding-window inference (SURVEY.md §8(f) rank 3).

The reference classifies a 64x64 tile by looping over its 8x8 windows and calling the model once per window with a
host synchronisation each time (inference_example.ipynb cell 13, src/utils.py:477-605: 64 forwards of batch B).  Here all
windows of all tiles go through ONE forward: the patch-embedding kernel reads every window straight out of the tile through
per-sample window offsets (csrc/pixel_source.cuh, `win_y` / `win_x` of msst_raw_input) -- no permute / copy of the input cube,
raw int16 tiles with on-the-fly standardisation included -- and the argmax / accuracy stay on the device.

Whole-scene inference (`predict_scene`) lifts the three limits of that path: any scene size (the last window row / column is
snapped to the border), overlapping windows whose class probabilities are blended per pixel on the device (csrc/scene.cu, no seams
every window), and chunks of windows so that a scene of any size fits.  `confusion_matrix` / `classification_metrics` score the
resulting map as hyperspectral classification results are reported: overall accuracy, average (macro) accuracy and Cohen's kappa.

`embed_scene` returns per-pixel encoder features of whole scenes.  `knn_neighbors` / `knn_classify` / `knn_scene` probe them with
k-nearest neighbours by cosine similarity (csrc/knn.cu).  The references stream through the tensor cores past each query tile, and
every query keeps its running top k on chip, so the [queries, references] score matrix is never stored.

`linear_probe_fit` / `LinearProbe` / `linear_probe_scene` are the other standard probe: softmax regression on LayerNorm'ed frozen
features, trained with AdamW for several (lr, weight_decay) heads at once (csrc/linprobe.cu: per minibatch one gradient launch, which
writes fixed 128-row slice partials for every head, and one launch that sums them in order and applies AdamW to every head).  Fits are
bitwise reproducible and each head is bitwise the head fitted alone.  `LinearProbe.load_into` writes a probe into the default head of
a ViTSpatialSpectral, whose LayerNorm and per-patch Linear then compute exactly the probe's function of the embed_scene features.

`kmeans_fit` / `KMeans` / `cluster_scene` cluster the features without labels (csrc/kmeans.cu: Lloyd's algorithm, per iteration one
assignment launch that writes fixed 4096-row slice partials for every restart and one launch that sums them in order; k-means++ seeding
in at most two launches per centroid).  `clustering_metrics` scores a clustering against ground truth: NMI, ARI and the accuracy of the
best one-to-one (Hungarian) and of the majority cluster -> class maps.

`reconstruct_scene` runs the SimMIM objective itself on whole scenes: a scene mask [B, C, H, W] hides spectral blocks at pixels (a
`scene_mask` drawn with the model's masking settings, or a map of dead stripes / saturated pixels), every window masks the tokens whose
patch touches a hidden entry, and csrc/scene.cu decodes the masked tokens with the trained to_pixels and blends each hidden entry's
predictions over the covering windows with the same ownership contract as the blends above.  The result is the inpainted scene in
the model's units; `reconstruction_metrics` gives the held-out masked L1 / RMSE per band and overall, and |recon - scene| is a
per-pixel reconstruction-error map.

`pca_fit` / `PCA` / `pca_scene` give the principal components of features (or of any rows of up to 256 values): csrc/moments.cu computes
the mean and the two-pass covariance in FP64 over fixed 16384-row slices, the host takes the float64 eigendecomposition, and the
projection kernel projects every row in FP64.  `false_colour` turns the first three components into the usual RGB picture of an
encoder's features.  `rx_scene` is the global RX anomaly detector, the squared Mahalanobis distance of each pixel from the scene's
Gaussian, on the encoder's features or (model=None) on the raw spectra; `anomaly_metrics` scores any anomaly map, RX or a
reconstruction-error map, against ground truth: ROC AUC, the ROC and the TPR at fixed false-positive rates.
"""
import ctypes
import math

import numpy as np
import torch

from . import _lib
from .input import RawTiles
from .vit_simmim_original import SimMIMSpatialSpectral
from .vit_spatial_spectral import ViTSpatialSpectral


@torch.no_grad()
def predict_tiles(model, tiles, window=None):
    """tiles: fp32 cube [B, C, H, W] (already standardised) or RawTiles over [B, raw_bands, H, W] sensor tiles
    -> logits [B, num_classes, H', W'] over the non-overlapping windows of the model's image_size that fit the tile."""
    w = window or model.image_size
    if isinstance(tiles, RawTiles):
        raw = tiles
        H, W = raw.tiles.shape[2:]
        gh, gw = (H - raw.crop[0]) // w, (W - raw.crop[1]) // w
        x = RawTiles(raw.tiles, raw.means, raw.stds, image_size=w, crop=raw.crop, pad_bands=raw.pad_bands, clip=raw.clip, windows=(gh, gw))
        B = raw.tiles.shape[0]
    else:
        B, C, H, W = tiles.shape
        assert H % w == 0 and W % w == 0, "tile size must be a multiple of the window"
        gh, gw = H // w, W // w
        if tiles.dtype != torch.float32:
            tiles = tiles.float()
        # identity statistics: (v - 0) / 1 in float64 rounds back to the same fp32 value
        x = RawTiles(tiles, torch.zeros(C, dtype=torch.float64), torch.ones(C, dtype=torch.float64), image_size=w, windows=(gh, gw))
    was_training = model.training
    model.eval()
    y = model(x)                                                     # [B*gh*gw, nc, w, w]
    model.train(was_training)
    nc = y.shape[1]
    return y.reshape(B, gh, gw, nc, w, w).permute(0, 3, 1, 4, 2, 5).reshape(B, nc, gh * w, gw * w)


@torch.no_grad()
def tile_accuracy(logits, labels, ignore_index=-1):
    """(overall accuracy, valid-pixel count) on the device; labels [B, H, W] int64."""
    pred = logits.argmax(dim=1)
    valid = labels != ignore_index
    n = valid.sum()
    return ((pred == labels) & valid).sum().float() / n.clamp_min(1), n


def scene_windows(H, W, window, stride):
    """(ny, nx): windows per scene column / row for a step of stride = (sy, sx) (or one int): ceil((H - window) / sy) + 1, so every
    pixel is covered and the last window row / column, snapped to the border, ends flush with it."""
    sy, sx = (stride, stride) if isinstance(stride, int) else stride
    if not (1 <= sy <= window and 1 <= sx <= window):
        raise ValueError(f"stride {(sy, sx)} must be in [1, window={window}]")
    if H < window or W < window:
        raise ValueError(f"scene {H}x{W} is smaller than the window {window}")
    return -(-(H - window) // sy) + 1, -(-(W - window) // sx) + 1


def _scene_input(who, scene, w, stride, weight):
    """The window view of a scene shared by predict_scene / embed_scene -> (RawTiles over all windows, (sy, sx), (ny, nx), weight on
    the scene's device or None)."""
    stride = stride if stride is not None else w
    if isinstance(scene, RawTiles):
        if scene.crop != (0, 0):
            raise ValueError(f"{who}: RawTiles must cover whole scenes (crop (0, 0)), got crop {scene.crop}")
        tiles, means, stds, pad, clip = scene.tiles, scene.means, scene.stds, scene.pad_bands, scene.clip
    else:
        if scene.dim() != 4:
            raise ValueError(f"{who}: scene must be [B, C, H, W], got {tuple(scene.shape)}")
        tiles = scene if scene.dtype == torch.float32 else scene.float()
        C_ = tiles.shape[1]
        # identity statistics: (v - 0) / 1 in float64 rounds back to the same fp32 value
        means, stds, pad, clip = torch.zeros(C_, dtype=torch.float64), torch.ones(C_, dtype=torch.float64), 0, None
    _, _, H, W = tiles.shape
    ny, nx = scene_windows(H, W, w, stride)
    sy, sx = (stride, stride) if isinstance(stride, int) else stride
    x = RawTiles(tiles, means, stds, image_size=w, pad_bands=pad, clip=clip, windows=(ny, nx), stride=(sy, sx))
    if weight is not None:
        weight = torch.as_tensor(weight, dtype=torch.float32, device=tiles.device).contiguous()
        if weight.shape != (w, w):
            raise ValueError(f"{who}: weight must be [{w}, {w}], got {tuple(weight.shape)}")
    return x, (sy, sx), (ny, nx), weight


@torch.no_grad()
def predict_scene(model, scene, *, stride=None, weight=None, batch_windows=4096):
    """Classifies whole scenes with overlapping windows.

    scene: standardised fp32 cube [B, C, H, W] (CUDA) or RawTiles over whole sensor scenes (crop (0, 0)); any H, W >= image_size.
    stride: window step (int or (sy, sx)), 1 <= stride <= image_size, default image_size (no overlap).
    weight: optional [image_size, image_size] per-window-pixel weight of a window's probabilities (e.g. a Gaussian that trusts window
    centres more than borders); default uniform.
    The windows run through the model in chunks of batch_windows (eval mode, no activations kept); each chunk's class probabilities
    are accumulated into the scene on the device, deterministically and independently of batch_windows.
    -> (probs [B, nc, H, W] fp32 = weighted mean of the covering windows' softmax, pred [B, H, W] int64 = probs.argmax(1))."""
    w = model.image_size
    x, (sy, sx), (ny, nx), weight = _scene_input("predict_scene", scene, w, stride, weight)
    B, _, H, W = x.tiles.shape
    dev = x.tiles.device
    nc = model.num_classes
    acc = torch.zeros(B, nc, H, W, device=dev, dtype=torch.float32)
    wsum = torch.zeros(B, H, W, device=dev, dtype=torch.float32)
    total, step = x.num_windows, max(1, int(batch_windows))
    was_training = model.training
    model.eval()
    try:
        for first in range(0, total, step):
            n = min(step, total - first)
            y = model(x.set_window_range(first, n))
            if y.numel() != n * nc * w * w:   # e.g. the pixelwise head: one class vector per window, not a map of the window
                raise ValueError(f"predict_scene: the model must classify every pixel of a window ([{n}, {nc}, {w}, {w}]), "
                                 f"got {tuple(y.shape)}")
            y = y.reshape(n, nc, w, w).float().contiguous()   # also restores a batch dim squeezed away for n == 1 (quirk C14)
            blend_windows(y, acc, wsum, stride=(sy, sx), grid=(ny, nx), first=first, weight=weight)
    finally:
        model.train(was_training)
    probs = acc / wsum[:, None]
    return probs, probs.argmax(1)


def blend_windows(logits, acc, wsum, *, stride, grid, first, weight=None):
    """One chunk of msst_scene_blend: acc [B, nc, H, W] += weight * softmax(logits), wsum [B, H, W] += weight over the pixels of
    global windows [first, first + n) (logits [n, nc, w, w] fp32, windows laid out as scene_windows / RawTiles(stride=...) lay them
    out: grid = (ny, nx) per scene).  Chunks must be blended in ascending order; the sums are then bitwise independent of the
    chunking."""
    n, nc, w = logits.shape[0], logits.shape[1], logits.shape[-1]
    B, _, H, W = acc.shape
    for t, name in ((logits, "logits"), (acc, "acc"), (wsum, "wsum"), (weight, "weight")):
        if t is not None and not (t.is_cuda and t.dtype == torch.float32 and t.is_contiguous()):
            raise ValueError(f"blend_windows: {name} must be a contiguous fp32 CUDA tensor")
    if logits.shape != (n, nc, w, w) or acc.shape[1] != nc or wsum.shape != (B, H, W) or (weight is not None and weight.shape != (w, w)):
        raise ValueError(f"blend_windows: shapes logits {tuple(logits.shape)}, acc {tuple(acc.shape)}, wsum {tuple(wsum.shape)} disagree")
    dims = _lib.SceneDims(B, nc, H, W, w, stride[0], stride[1], grid[0], grid[1], first, n)
    _lib.check(_lib.lib().msst_scene_blend(ctypes.byref(dims), logits.data_ptr(), weight.data_ptr() if weight is not None else None,
                                           acc.data_ptr(), wsum.data_ptr(), torch.cuda.current_stream(acc.device).cuda_stream))


@torch.no_grad()
def embed_scene(model, scene, *, stride=None, weight=None, batch_windows=4096):
    """Per-pixel encoder features of whole scenes from overlapping windows: the map a k-NN / linear probe, a clustering or another
    model starts from after pretraining.

    model: ViTSpatialSpectral with any head (the head is not run; spectral_only too), or SimMIMSpatialSpectral, whose encoder is used
    (so a pretraining checkpoint embeds directly).  fp32 or bf16 precision; the features are fp32 either way.
    scene, stride, weight, batch_windows: as in predict_scene (weight weighs a window's features instead of its probabilities).
    A window's feature at a pixel is the spectral mean of its tokens at the pixel's spatial patch, the input of the default head's
    LayerNorm; the covering windows' features are blended on the device, deterministically and independently of batch_windows.
    -> features [B, dim, H, W] fp32 = weighted mean of the covering windows' features."""
    enc = model.encoder if isinstance(model, SimMIMSpatialSpectral) else model
    if not isinstance(enc, ViTSpatialSpectral):   # ViTSpatialSpectral_V1.forward_features returns a tuple of token sets
        raise ValueError(f"embed_scene: needs a ViTSpatialSpectral encoder, got {type(enc).__name__}")
    w = enc.image_size
    x, (sy, sx), (ny, nx), weight = _scene_input("embed_scene", scene, w, stride, weight)
    B, _, H, W = x.tiles.shape
    D, nblk, p1 = enc.dim, enc.num_spectral_patches, enc.patch_height
    acc = torch.zeros(B, D, H, W, device=x.tiles.device, dtype=torch.float32)
    wsum = torch.zeros(B, H, W, device=x.tiles.device, dtype=torch.float32)
    total, step = x.num_windows, max(1, int(batch_windows))
    was_training = enc.training
    enc.eval()
    try:
        for first in range(0, total, step):
            n = min(step, total - first)
            tokens = enc.forward_features(x.set_window_range(first, n))   # [n, C*S, D] fp32 (the residual stream)
            embed_windows(tokens, acc, wsum, C=nblk, p1=p1, stride=(sy, sx), grid=(ny, nx), first=first, weight=weight)
    finally:
        enc.train(was_training)
    return acc / wsum[:, None]


def embed_windows(tokens, acc, wsum, *, C, p1, stride, grid, first, weight=None):
    """One chunk of msst_scene_embed: acc [B, D, H, W] += weight * f, wsum [B, H, W] += weight over the pixels of global windows
    [first, first + n), where f is the window's spectral-mean feature at the pixel's spatial patch, (1/C) sum_c tokens[c*S + s]
    (tokens [n, C*S, D] fp32 = forward_features of the chunk, S = G*G, window side G*p1; windows laid out as in blend_windows).
    Chunks must be embedded in ascending order; the sums are then bitwise independent of the chunking."""
    for t, name in ((tokens, "tokens"), (acc, "acc"), (wsum, "wsum"), (weight, "weight")):
        if t is not None and not (t.is_cuda and t.dtype == torch.float32 and t.is_contiguous()):
            raise ValueError(f"embed_windows: {name} must be a contiguous fp32 CUDA tensor")
    if tokens.dim() != 3 or acc.dim() != 4 or C < 1 or p1 < 1:
        raise ValueError(f"embed_windows: tokens must be [n, C*S, D] and acc [B, D, H, W], got {tuple(tokens.shape)}, {tuple(acc.shape)}")
    n, T, D = tokens.shape
    B, _, H, W = acc.shape
    S = T // C
    G = math.isqrt(S)
    w = G * p1
    if (T != C * S or G * G != S or acc.shape[1] != D or wsum.shape != (B, H, W)
            or (weight is not None and weight.shape != (w, w))):
        raise ValueError(f"embed_windows: shapes tokens {tuple(tokens.shape)} (C={C}, p1={p1}), acc {tuple(acc.shape)}, "
                         f"wsum {tuple(wsum.shape)} disagree")
    dims = _lib.SceneEmbedDims(B, D, H, W, w, stride[0], stride[1], grid[0], grid[1], first, n, C, p1)
    _lib.check(_lib.lib().msst_scene_embed(ctypes.byref(dims), tokens.data_ptr(), weight.data_ptr() if weight is not None else None,
                                           acc.data_ptr(), wsum.data_ptr(), torch.cuda.current_stream(acc.device).cuda_stream))


def _recon_encoder(who, model):
    """The encoder of a SimMIM model whose decoder output maps back to scene pixels, else ValueError."""
    if not isinstance(model, SimMIMSpatialSpectral):
        raise ValueError(f"{who}: needs a SimMIMSpatialSpectral model (its decoder reconstructs the masked values), got "
                         f"{type(model).__name__}")
    enc = model.encoder
    if model.v1 or not isinstance(enc, ViTSpatialSpectral):
        raise ValueError(f"{who}: needs a ViTSpatialSpectral encoder, got {type(enc).__name__}")
    if not enc.blockwise_patch_embed:
        raise ValueError(f"{who}: needs the blockwise patch embedding (blockwise_patch_embed=True): with PatchEmbed the decoder predicts "
                         f"LayerNorm'ed patches, which do not map back to pixel values")
    return enc


def _model_units(scene, pad):
    """The scene as the model sees it, fp32 [B, bands, H, W]: the cube itself, or RawTiles standardised (pad: with the pad bands)."""
    if isinstance(scene, RawTiles):
        return scene.standardize(scene.tiles, pad=pad)
    return scene if scene.dtype == torch.float32 else scene.float()


def _patch_any(mask, p1):
    """[B, C, H, W] bool -> [B, C, H - p1 + 1, W - p1 + 1]: whether any pixel of the p1 x p1 square with top-left corner (y, x) is set."""
    if p1 == 1:
        return mask
    h, w = mask.shape[2] - p1 + 1, mask.shape[3] - p1 + 1
    out = mask[:, :, :h, :w].clone()
    for i in range(p1):
        for j in range(p1):
            out |= mask[:, :, i:i + h, j:j + w]
    return out


def _window_mask(pany, p1, window, stride, grid, first, n):
    """Token mask [n, C*S] (t = c*S + s) of global windows [first, first + n), laid out as in blend_windows, from _patch_any(scene mask,
    p1): token (c, s) of a window is masked when any pixel of its spatial patch s has block c set."""
    B, C, h, w = pany.shape
    H, W = h + p1 - 1, w + p1 - 1
    (sy, sx), (ny, nx) = stride, grid
    dev = pany.device
    g = torch.arange(first, first + n, device=dev)
    b, k = g // (ny * nx), g % (ny * nx)
    oy = torch.clamp_max((k // nx) * sy, H - window)                    # the origin rule of window_origin (csrc/pixel_source.cuh)
    ox = torch.clamp_max((k % nx) * sx, W - window)
    r = torch.arange(window // p1, device=dev) * p1
    c = torch.arange(C, device=dev)
    m = pany[b[:, None, None, None], c[None, :, None, None], (oy[:, None] + r)[:, None, :, None], (ox[:, None] + r)[:, None, None, :]]
    return m.reshape(n, -1)


def _check_scene_mask(who, mask, B, C, H, W, device):
    if (not isinstance(mask, torch.Tensor) or mask.dtype != torch.bool or tuple(mask.shape) != (B, C, H, W)
            or mask.device != device):
        got = (f"{mask.dtype} {tuple(mask.shape)} on {mask.device}" if isinstance(mask, torch.Tensor) else type(mask).__name__)
        raise ValueError(f"{who}: mask must be a bool tensor [{B}, {C}, {H}, {W}] (one entry per spectral block) on {device}, got {got}")


@torch.no_grad()
def reconstruct_scene(model, scene, mask, *, stride=None, weight=None, batch_windows=4096):
    """Masked reconstruction of whole scenes by a SimMIM checkpoint: inpainting of hidden values, held-out reconstruction error
    (reconstruction_metrics) and per-pixel error maps.

    model: SimMIMSpatialSpectral over a ViTSpatialSpectral with the blockwise patch embedding, either decoder (to_pixels or
    BlockwiseToPixels), spectral_only too; fp32 or bf16 precision.
    scene, stride, weight, batch_windows: as in predict_scene (weight weighs a window's predictions).
    mask [B, C, H, W] bool on the scene's device, C = encoder.num_spectral_patches: entry (b, c, y, x) hides the p0 bands
    c*p0 ... c*p0 + p0 - 1 at pixel (y, x) (scene_mask draws one; a map of dead stripes or saturated pixels works the same way).
    In every window, token (c, s) is masked when any pixel of spatial patch s has block c hidden, so a hidden entry is masked in every
    window that covers it and its own value never reaches the encoder.  The windows run in chunks through the patch embedding (with
    the mask token) and the encoder in eval mode; msst_scene_reconstruct decodes the masked tokens and blends each hidden entry's
    predictions over the covering windows on the device, deterministically and independently of batch_windows.
    -> recon [B, C*p0, H, W] fp32 in the model's units: hidden entries hold the weighted mean prediction, visible entries the input
    (the standardised cube, pad bands included for RawTiles)."""
    who = "reconstruct_scene"
    enc = _recon_encoder(who, model)
    tiles = scene.tiles if isinstance(scene, RawTiles) else scene
    if not isinstance(tiles, torch.Tensor) or tiles.dim() != 4:
        raise ValueError(f"{who}: scene must be a [B, C, H, W] tensor or RawTiles")
    if not tiles.is_cuda:
        raise ValueError(f"{who}: the scene must be on a CUDA device")
    C, p0, p1 = enc.num_spectral_patches, enc.patch_depth, enc.patch_height
    B, nb, H, W = tiles.shape
    nb += scene.pad_bands if isinstance(scene, RawTiles) else 0
    if nb != C * p0:
        raise ValueError(f"{who}: the scene has {nb} bands, the model {C * p0}")
    _check_scene_mask(who, mask, B, C, H, W, tiles.device)
    w = enc.image_size
    x, (sy, sx), (ny, nx), weight = _scene_input(who, scene, w, stride, weight)
    if model.to_pixels_per_spectral_block:
        Wd, bd = model.to_pixels.kernel_params()
    else:
        Wd, bd = model.to_pixels.weight[None], model.to_pixels.bias[None]
    Wd, bd = Wd.detach().float().contiguous(), bd.detach().float().contiguous()
    mask = mask.contiguous()
    pany = _patch_any(mask, p1)
    acc = torch.zeros(B, C * p0, H, W, device=tiles.device, dtype=torch.float32)
    wsum = torch.zeros(B, H, W, device=tiles.device, dtype=torch.float32)
    total, step = x.num_windows, max(1, int(batch_windows))
    was_training = model.training
    model.eval()
    try:
        pos = enc._pos_rows()
        for first in range(0, total, step):
            n = min(step, total - first)
            wmask = _window_mask(pany, p1, w, (sy, sx), (ny, nx), first, n)
            tokens = enc.to_patch_embedding._embed_img(x.set_window_range(first, n), pos=pos, mask_token=model.mask_token, mask=wmask)
            tokens = enc.transformer_forward(tokens)                        # [n, C*S, D] fp32
            reconstruct_windows(tokens, mask.view(torch.uint8), Wd, bd, acc, wsum, C=C, p0=p0, p1=p1, stride=(sy, sx), grid=(ny, nx),
                                first=first, weight=weight)
    finally:
        model.train(was_training)
    acc.div_(wsum[:, None])
    return torch.where(mask.repeat_interleave(p0, 1), acc, _model_units(scene, pad=True))


def reconstruct_windows(tokens, mask, W, bias, acc, wsum, *, C, p0, p1, stride, grid, first, weight=None):
    """One chunk of msst_scene_reconstruct: for every entry (b, c*p0 + j, y, x) that the scene mask [B, C, H, W] (uint8 or bool) hides,
    acc [B, C*p0, H, W] += weight * (W[blk] . token + bias[blk])[j*p1^2 + (py % p1)*p1 + px % p1] over the global windows
    [first, first + n) that cover (y, x), token = tokens[window, c*S + (py // p1)*G + px // p1] ((py, px): the pixel in the window;
    blk = c for a per-block decoder W [C, P, D], bias [C, P], else 0 for W [1, P, D], bias [1, P]; P = p0*p1^2), and wsum [B, H, W]
    += weight once per covering window.  tokens [n, C*S, D] fp32 is the encoder output of the chunk's masked windows; windows laid out
    as in blend_windows.  Chunks must be added in ascending order; the sums are then bitwise independent of the chunking."""
    who = "reconstruct_windows"
    for t, name in ((tokens, "tokens"), (W, "W"), (bias, "bias"), (acc, "acc"), (wsum, "wsum"), (weight, "weight")):
        if (t is not None or name != "weight") and not (isinstance(t, torch.Tensor) and t.is_cuda and t.dtype == torch.float32
                                                         and t.is_contiguous()):
            raise ValueError(f"{who}: {name} must be a contiguous fp32 CUDA tensor")
    if not (isinstance(mask, torch.Tensor) and mask.is_cuda and mask.dtype in (torch.uint8, torch.bool) and mask.is_contiguous()):
        raise ValueError(f"{who}: mask must be a contiguous uint8 or bool CUDA tensor")
    if any(t is not None and t.device != acc.device for t in (tokens, mask, W, bias, wsum, weight)):
        raise ValueError(f"{who}: all tensors must be on {acc.device}")
    if tokens.dim() != 3 or acc.dim() != 4 or W.dim() != 3 or bias.dim() != 2 or min(C, p0, p1) < 1:
        raise ValueError(f"{who}: tokens must be [n, C*S, D], acc [B, C*p0, H, W], W [n_wb, P, D] and bias [n_wb, P], got "
                         f"{tuple(tokens.shape)}, {tuple(acc.shape)}, {tuple(W.shape)}, {tuple(bias.shape)}")
    n, T, D = tokens.shape
    B, nb, H, Wd = acc.shape
    S = T // C
    G = math.isqrt(S)
    w, P = G * p1, p0 * p1 * p1
    if (T != C * S or G * G != S or nb != C * p0 or tuple(mask.shape) != (B, C, H, Wd) or tuple(wsum.shape) != (B, H, Wd)
            or W.shape[0] not in (1, C) or tuple(W.shape[1:]) != (P, D) or tuple(bias.shape) != (W.shape[0], P)
            or (weight is not None and tuple(weight.shape) != (w, w))):
        raise ValueError(f"{who}: shapes tokens {tuple(tokens.shape)} (C={C}, p0={p0}, p1={p1}), mask {tuple(mask.shape)}, "
                         f"W {tuple(W.shape)}, bias {tuple(bias.shape)}, acc {tuple(acc.shape)}, wsum {tuple(wsum.shape)} disagree")
    dims = _lib.SceneReconstructDims(B, D, H, Wd, w, stride[0], stride[1], grid[0], grid[1], first, n, C, p0, p1, W.shape[0])
    _lib.check(_lib.lib().msst_scene_reconstruct(ctypes.byref(dims), tokens.data_ptr(), mask.data_ptr(), W.data_ptr(), bias.data_ptr(),
                                                 weight.data_ptr() if weight is not None else None, acc.data_ptr(), wsum.data_ptr(),
                                                 torch.cuda.current_stream(acc.device).cuda_stream))


def scene_mask(model, B, H, W, *, seed=0, device):
    """A random scene mask [B, C, H, W] bool (C = spectral blocks) drawn with a SimMIM model's own settings, for held-out evaluation
    with reconstruct_scene / reconstruction_metrics.  The scene is cut into mask_patch_size x mask_patch_size cells aligned to its
    origin (partial cells at the bottom / right border count as cells), and exactly ceil(masking_ratio * cells) cells are hidden per
    scene with tube_masking (every block alike), else per (scene, block) -- MaskGenerator's count, over the scene instead of a window.
    (Per-window masks would disagree where windows overlap.)  Drawn from a CPU torch.Generator seeded with seed: rows in (scene, block)
    order, one randperm each, so the mask is reproducible on any machine."""
    if not isinstance(model, SimMIMSpatialSpectral):
        raise ValueError(f"scene_mask: needs a SimMIMSpatialSpectral model, got {type(model).__name__}")
    for name, v in (("B", B), ("H", H), ("W", W)):
        if isinstance(v, bool) or not isinstance(v, int) or v < 1:
            raise ValueError(f"scene_mask: {name}={v!r} must be a positive int")
    if isinstance(seed, bool) or not isinstance(seed, int) or seed < 0:
        raise ValueError(f"scene_mask: seed={seed!r} must be an int >= 0")
    C, m = model.encoder.num_spectral_patches, model.mask_patch_size
    ncy, ncx = -(-H // m), -(-W // m)
    ncells = ncy * ncx
    count = int(np.ceil(ncells * model.masking_ratio))
    rows = B if model.tube_masking else B * C
    g = torch.Generator().manual_seed(seed)
    cells = torch.zeros(rows, ncells, dtype=torch.bool)
    for r in range(rows):
        cells[r, torch.randperm(ncells, generator=g)[:count]] = True
    cells = cells.view(rows, ncy, ncx).repeat_interleave(m, 1).repeat_interleave(m, 2)[:, :H, :W]
    out = cells[:, None].expand(B, C, H, W) if model.tube_masking else cells.view(B, C, H, W)
    return out.contiguous().to(device)


def reconstruction_metrics(recon, scene, mask):
    """Reconstruction error of recon [B, C*p0, H, W] (reconstruct_scene) against the scene in the model's units, in float64 over the
    hidden entries of mask [B, C, H, W] (pad bands of RawTiles left out):
      count                                 hidden entries
      l1   = mean |recon - target|,  rmse = sqrt(mean (recon - target)^2)
      baseline_l1 = mean |target|           the error of predicting each band's mean of standardised data (0), so l1 / baseline_l1
                                            is a scale-free figure
      per_band_l1 / per_band_rmse / per_band_count   the same per band ([bands] float64 / int64 tensors on the CPU)
    An empty mask gives count 0 and NaN errors.  For a one-window scene, l1 / num_masked is SimMIM's training loss on that mask.
    -> dict."""
    who = "reconstruction_metrics"
    tiles = scene.tiles if isinstance(scene, RawTiles) else scene
    if not isinstance(tiles, torch.Tensor) or tiles.dim() != 4:
        raise ValueError(f"{who}: scene must be a [B, C, H, W] tensor or RawTiles")
    B, nb, H, W = tiles.shape
    if not isinstance(recon, torch.Tensor) or recon.dim() != 4 or recon.shape[0] != B or tuple(recon.shape[2:]) != (H, W):
        raise ValueError(f"{who}: recon must be a [{B}, bands, {H}, {W}] tensor, got "
                         f"{tuple(recon.shape) if isinstance(recon, torch.Tensor) else type(recon).__name__}")
    if not isinstance(mask, torch.Tensor) or mask.dim() != 4 or mask.shape[1] < 1 or recon.shape[1] % mask.shape[1]:
        raise ValueError(f"{who}: mask must be [B, C, H, W] with C dividing the {recon.shape[1]} bands of recon")
    C = mask.shape[1]
    _check_scene_mask(who, mask, B, C, H, W, recon.device)
    p0 = recon.shape[1] // C
    if not isinstance(scene, RawTiles) and nb != recon.shape[1] or isinstance(scene, RawTiles) and nb + scene.pad_bands != recon.shape[1]:
        raise ValueError(f"{who}: recon has {recon.shape[1]} bands, the scene {nb}"
                         f"{f' + {scene.pad_bands} pad' if isinstance(scene, RawTiles) else ''}")
    target = _model_units(scene, pad=False).to(device=recon.device, dtype=torch.float64)
    hidden = mask.repeat_interleave(p0, 1)[:, :nb]
    d = torch.where(hidden, recon[:, :nb].double() - target, 0.0)
    t = torch.where(hidden, target, 0.0)
    cnt = hidden.sum((0, 2, 3)).cpu()
    s1, s2, st = d.abs().sum((0, 2, 3)).cpu(), (d * d).sum((0, 2, 3)).cpu(), t.abs().sum((0, 2, 3)).cpu()
    n = cnt.sum().double()
    return dict(count=int(n), l1=float(s1.sum() / n), rmse=float((s2.sum() / n).sqrt()), baseline_l1=float(st.sum() / n),
                per_band_l1=s1 / cnt, per_band_rmse=(s2 / cnt).sqrt(), per_band_count=cnt)


def confusion_matrix(pred, labels, num_classes, ignore_index=-1):
    """[nc, nc] int64 counts, rows = true class, columns = predicted class.  A pixel counts when its label is not ignore_index and lies
    in [0, num_classes) -- the validity rule of the fine-tuning loss (ce_kernel, csrc/head.cu).  Runs wherever the tensors are."""
    labels = labels.reshape(-1).to(torch.int64)
    pred = pred.reshape(-1).to(device=labels.device, dtype=torch.int64)
    if pred.numel() != labels.numel():
        raise ValueError(f"confusion_matrix: {pred.numel()} predictions for {labels.numel()} labels")
    valid = (labels != ignore_index) & (labels >= 0) & (labels < num_classes)
    lab, prd = labels[valid], pred[valid]
    if bool(((prd < 0) | (prd >= num_classes)).any()):
        raise ValueError(f"confusion_matrix: predictions outside [0, {num_classes})")
    return torch.bincount(lab * num_classes + prd, minlength=num_classes * num_classes).reshape(num_classes, num_classes)


def classification_metrics(conf):
    """OA / AA / kappa of a confusion matrix (rows = true class), in float64:
      oa    = trace / total                                      (overall accuracy)
      per_class_acc[k] = conf[k, k] / conf[k, :].sum()           (recall; nan for a class absent from the labels)
      aa    = mean of per_class_acc over the classes that occur in the labels (average accuracy; absent classes are left out
              rather than counted as 0 or 1, so a scene that lacks a class is not penalised for it)
      kappa = (oa - pe) / (1 - pe),  pe = sum_k rows_k * cols_k / total^2   (Cohen's kappa; nan when pe == 1)
    -> dict(oa=float, aa=float, kappa=float, per_class_acc=[nc] float64 tensor on the CPU)."""
    conf = torch.as_tensor(conf).detach().to("cpu", torch.float64)
    total = conf.sum()
    rows, cols, diag = conf.sum(1), conf.sum(0), conf.diagonal()
    per_class = diag / rows                                   # 0 / 0 = nan for absent classes
    present = rows > 0
    oa = float(diag.sum() / total)
    aa = float(per_class[present].mean()) if bool(present.any()) else float("nan")
    pe = float((rows * cols).sum() / (total * total))
    kappa = (oa - pe) / (1.0 - pe) if pe != 1.0 else float("nan")
    return dict(oa=oa, aa=aa, kappa=kappa, per_class_acc=per_class)


KNN_MAX_K, KNN_MAX_DIM, KNN_MAX_CLASSES = 64, 256, 256


def _knn_features(who, name, x):
    if not isinstance(x, torch.Tensor) or x.dim() != 2 or x.dtype != torch.float32 or not x.is_cuda:
        raise ValueError(f"{who}: {name} must be a 2-D fp32 CUDA tensor [rows, dim], got "
                         f"{tuple(x.shape) if isinstance(x, torch.Tensor) else type(x).__name__}"
                         f"{f' {x.dtype} on {x.device}' if isinstance(x, torch.Tensor) else ''}")
    D = x.shape[1]
    if D % 32 or not 32 <= D <= KNN_MAX_DIM:
        raise ValueError(f"{who}: feature width {D} must be a multiple of 32 in [32, {KNN_MAX_DIM}]")
    return x.contiguous()


def _knn_check(who, ref, query, k, batch_queries):
    ref, query = _knn_features(who, "ref", ref), _knn_features(who, "query", query)
    if ref.shape[1] != query.shape[1] or ref.device != query.device:
        raise ValueError(f"{who}: ref {tuple(ref.shape)} on {ref.device} and query {tuple(query.shape)} on {query.device} disagree")
    if isinstance(k, bool) or not isinstance(k, int) or not 1 <= k <= KNN_MAX_K:
        raise ValueError(f"{who}: k={k!r} must be an int in [1, {KNN_MAX_K}]")
    if not k <= ref.shape[0] < 2 ** 31:
        raise ValueError(f"{who}: {ref.shape[0]} reference rows; need k={k} <= rows < 2^31")
    if isinstance(batch_queries, bool) or not isinstance(batch_queries, int) or batch_queries < 1:
        raise ValueError(f"{who}: batch_queries={batch_queries!r} must be a positive int")
    return ref, query


def _knn_prepare(x):
    """msst_knn_prepare: rows [n, D] fp32 -> normalised, split operand rows [n, 3 * D] bf16."""
    out = torch.empty(x.shape[0], 3 * x.shape[1], device=x.device, dtype=torch.bfloat16)
    _lib.check(_lib.lib().msst_knn_prepare(x.data_ptr(), x.shape[0], x.shape[1], out.data_ptr(),
                                           torch.cuda.current_stream(x.device).cuda_stream))
    return out


def _knn_chunks(ref, query, k, batch_queries):
    """Yields (first, last, scores [n, k], index [n, k]) for the query chunks [first, last) in order."""
    N, D = ref.shape
    rp = _knn_prepare(ref)
    stream = torch.cuda.current_stream(ref.device).cuda_stream
    for first in range(0, query.shape[0], batch_queries):
        last = min(first + batch_queries, query.shape[0])
        qp = _knn_prepare(query[first:last])
        scores = torch.empty(last - first, k, device=ref.device, dtype=torch.float32)
        index = torch.empty(last - first, k, device=ref.device, dtype=torch.int64)
        dims = _lib.KnnDims(N, last - first, D, k)
        _lib.check(_lib.lib().msst_knn_topk(ctypes.byref(dims), rp.data_ptr(), qp.data_ptr(), scores.data_ptr(), index.data_ptr(), stream))
        yield first, last, scores, index


@torch.no_grad()
def knn_neighbors(ref, query, k, *, batch_queries=262144):
    """The k nearest references of every query by cosine similarity, found on the device without the [Q, N] score matrix.

    ref [N, D], query [Q, D]: fp32 CUDA tensors, D a multiple of 32 in [32, 256], 1 <= k <= 64, k <= N < 2^31.  Rows are normalised as
    F.normalize does (eps 1e-12), so a zero row scores 0 against everything.  Scores are fp32-accurate (three-part bf16 split on the
    tensor cores, DESIGN.md §3).  Queries run in chunks of batch_queries; the result is bitwise the same for any chunk size.
    -> (scores [Q, k] fp32, descending; index [Q, k] int64), ordered by (score descending, reference index ascending)."""
    ref, query = _knn_check("knn_neighbors", ref, query, k, batch_queries)
    scores = torch.empty(query.shape[0], k, device=ref.device, dtype=torch.float32)
    index = torch.empty(query.shape[0], k, device=ref.device, dtype=torch.int64)
    for first, last, s, i in _knn_chunks(ref, query, k, batch_queries):
        scores[first:last], index[first:last] = s, i
    return scores, index


def _knn_vote_args(who, ref, ref_labels, num_classes, temperature):
    if isinstance(num_classes, bool) or not isinstance(num_classes, int) or not 1 <= num_classes <= KNN_MAX_CLASSES:
        raise ValueError(f"{who}: num_classes={num_classes!r} must be an int in [1, {KNN_MAX_CLASSES}]")
    t = float(temperature)
    if not t > 0:   # NaN fails too
        raise ValueError(f"{who}: temperature={temperature!r} must be > 0 (float('inf') for a uniform vote)")
    if (not isinstance(ref_labels, torch.Tensor) or ref_labels.shape != (ref.shape[0],) or ref_labels.device != ref.device
            or ref_labels.dtype.is_floating_point or ref_labels.dtype.is_complex or ref_labels.dtype == torch.bool):
        raise ValueError(f"{who}: ref_labels must be an integer tensor [{ref.shape[0]}] on {ref.device}, got "
                         f"{tuple(ref_labels.shape) if isinstance(ref_labels, torch.Tensor) else type(ref_labels).__name__}")
    ref_labels = ref_labels.to(torch.int64).contiguous()
    if bool(((ref_labels < 0) | (ref_labels >= num_classes)).any()):
        raise ValueError(f"{who}: reference labels outside [0, {num_classes})")
    return ref_labels, t


@torch.no_grad()
def knn_classify(ref, ref_labels, query, *, num_classes, k=20, temperature=0.07, batch_queries=262144):
    """k-NN classification of queries by labelled references (the usual probe of a self-supervised encoder).

    ref, query, k, batch_queries: as in knn_neighbors.  ref_labels [N] integers in [0, num_classes), num_classes <= 256.
    Each query's k nearest references vote with weight w_j = exp((s_j - s_0) / temperature) (s: cosine similarities, s_0 the largest;
    the DINO k-NN protocol), normalised to sum 1; temperature=float('inf') gives the uniform vote.
    -> (probs [Q, num_classes] fp32, pred [Q] int64 = argmax, lowest class on ties)."""
    ref, query = _knn_check("knn_classify", ref, query, k, batch_queries)
    ref_labels, t = _knn_vote_args("knn_classify", ref, ref_labels, num_classes, temperature)
    probs = torch.empty(query.shape[0], num_classes, device=ref.device, dtype=torch.float32)
    pred = torch.empty(query.shape[0], device=ref.device, dtype=torch.int64)
    stream = torch.cuda.current_stream(ref.device).cuda_stream
    for first, last, s, i in _knn_chunks(ref, query, k, batch_queries):
        _lib.check(_lib.lib().msst_knn_vote(last - first, k, ref.shape[0], s.data_ptr(), i.data_ptr(), ref_labels.data_ptr(), num_classes,
                                            t, probs[first:last].data_ptr(), pred[first:last].data_ptr(), stream))
    return probs, pred


@torch.no_grad()
def knn_scene(model, scene, train_labels, *, num_classes, k=20, temperature=0.07, stride=None, weight=None, batch_windows=4096,
              ignore_index=-1, batch_queries=262144):
    """k-NN probe of an encoder on whole scenes: embed_scene features, the labelled pixels as references, every pixel as a query.

    model, scene, stride, weight, batch_windows: as in embed_scene (a SimMIMSpatialSpectral checkpoint works directly).
    train_labels [B, H, W] integers on the scene's device: a pixel is a reference when its label is != ignore_index and in
    [0, num_classes) (the rule of confusion_matrix).  k, temperature, batch_queries: as in knn_classify.
    Score the result against held-out labels with confusion_matrix / classification_metrics.
    -> (probs [B, num_classes, H, W] fp32, pred [B, H, W] int64)."""
    labels, valid = _scene_labels("knn_scene", scene, train_labels, num_classes, ignore_index)
    feats = embed_scene(model, scene, stride=stride, weight=weight, batch_windows=batch_windows)   # [B, D, H, W]
    flat = _pixel_rows(feats)
    probs, pred = knn_classify(flat[valid], labels[valid], flat, num_classes=num_classes, k=k, temperature=temperature,
                               batch_queries=batch_queries)
    return _pixel_map(probs, feats), pred.reshape(feats.shape[0], *feats.shape[2:])


def _scene_labels(who, scene, train_labels, num_classes, ignore_index, name="train_labels"):
    """Checks a whole-scene probe's scene and per-pixel labels -> (labels [B*H*W] int64, valid [B*H*W] bool).  A pixel is valid when
    its label is != ignore_index and in [0, num_classes): the rule of confusion_matrix."""
    tiles = scene.tiles if isinstance(scene, RawTiles) else scene
    if not isinstance(tiles, torch.Tensor) or tiles.dim() != 4:
        raise ValueError(f"{who}: scene must be a [B, C, H, W] tensor or RawTiles")
    B, _, H, W = tiles.shape
    if (not isinstance(train_labels, torch.Tensor) or train_labels.shape != (B, H, W) or train_labels.dtype.is_floating_point
            or train_labels.dtype == torch.bool or train_labels.device != tiles.device):
        raise ValueError(f"{who}: {name} must be an integer tensor [{B}, {H}, {W}] on {tiles.device}")
    if not tiles.is_cuda:
        raise ValueError(f"{who}: the scene must be on a CUDA device")
    if isinstance(num_classes, bool) or not isinstance(num_classes, int) or not 1 <= num_classes <= KNN_MAX_CLASSES:
        raise ValueError(f"{who}: num_classes={num_classes!r} must be an int in [1, {KNN_MAX_CLASSES}]")
    labels = train_labels.reshape(-1).to(torch.int64)
    return labels, (labels != ignore_index) & (labels >= 0) & (labels < num_classes)


def _pixel_rows(feats):
    """[B, D, H, W] -> [B*H*W, D]: the one copy that makes pixels rows."""
    return feats.permute(0, 2, 3, 1).reshape(-1, feats.shape[1])


def _pixel_map(rows, feats):
    """[B*H*W, nc] per-pixel rows -> [B, nc, H, W] over the scenes of feats [B, D, H, W]."""
    B, _, H, W = feats.shape
    return rows.reshape(B, H, W, rows.shape[1]).permute(0, 3, 1, 2).contiguous()


LINPROBE_MAX_HEADS = 16


def _linprobe_heads(who, heads):
    try:
        pairs = [(float(lr), float(wd)) for lr, wd in heads]
    except (TypeError, ValueError):
        raise ValueError(f"{who}: heads must be a sequence of (lr, weight_decay) pairs, got {heads!r}") from None
    if not 1 <= len(pairs) <= LINPROBE_MAX_HEADS:
        raise ValueError(f"{who}: {len(pairs)} heads; need 1 to {LINPROBE_MAX_HEADS}")
    for lr, wd in pairs:
        if not (0 <= lr < math.inf and 0 <= wd < math.inf):   # NaN fails too
            raise ValueError(f"{who}: lr={lr!r} and weight_decay={wd!r} must be finite and >= 0")
    return pairs


def _int_arg(who, name, v, lo):
    if isinstance(v, bool) or not isinstance(v, int) or v < lo:
        raise ValueError(f"{who}: {name}={v!r} must be an int >= {lo}")


def _labelled_rows(who, x, y, num_classes, name):
    x = _knn_features(who, name, x)
    if not x.shape[0] < 2 ** 31 or x.shape[0] < 1:
        raise ValueError(f"{who}: {name} has {x.shape[0]} rows; need 1 <= rows < 2^31")
    if (not isinstance(y, torch.Tensor) or y.shape != (x.shape[0],) or y.device != x.device or y.dtype.is_floating_point
            or y.dtype.is_complex or y.dtype == torch.bool):
        raise ValueError(f"{who}: labels of {name} must be an integer tensor [{x.shape[0]}] on {x.device}, got "
                         f"{tuple(y.shape) if isinstance(y, torch.Tensor) else type(y).__name__}")
    y = y.to(torch.int64).contiguous()
    if bool(((y < 0) | (y >= num_classes)).any()):
        raise ValueError(f"{who}: labels of {name} outside [0, {num_classes})")
    return x, y


def _linprobe_dims(n, dim, nc, heads, batch=1, step=1):
    d = _lib.LinprobeDims(n, dim, nc, len(heads), batch, step)
    for h, (lr, wd) in enumerate(heads):
        d.lr[h], d.wd[h] = lr, wd
    return d


def _linprobe_grad(dims, x, labels, index, params, workspace):
    """One msst_linprobe_grad launch: the minibatch x[index] -> per-slice partials in workspace (dims.batch = index.numel())."""
    _lib.check(_lib.lib().msst_linprobe_grad(ctypes.byref(dims), x.data_ptr(), labels.data_ptr(), index.data_ptr(), params.data_ptr(),
                                             workspace.data_ptr(), torch.cuda.current_stream(x.device).cuda_stream))


def _linprobe_update(dims, workspace, params, m, v, loss_sum):
    """One msst_linprobe_update launch: AdamW step dims.step of every head; loss_sum [H] = the step's CE sums."""
    _lib.check(_lib.lib().msst_linprobe_update(ctypes.byref(dims), workspace.data_ptr(), params.data_ptr(), m.data_ptr(), v.data_ptr(),
                                               loss_sum.data_ptr(), torch.cuda.current_stream(params.device).cuda_stream))


class LinearProbe:
    """A fitted linear probe: per head h, W[h] [nc, dim] and b[h] [nc] on LN(x) (F.layer_norm(x, (dim,)), no affine).

    params [H, nc*dim + nc] fp32 (CUDA): head h is W_h row-major followed by b_h (the msst_linprobe layout); W / b are views.
    heads: the (lr, weight_decay) pairs; train_loss [epochs, H] float64: mean training CE per epoch; val_acc [H] float64 or None: OA of
    each head on the validation rows; best: the head predict / load_into use by default (argmax of val_acc, lowest index on ties)."""

    def __init__(self, params, num_classes, dim, heads, train_loss=None, val_acc=None, best=0):
        self.params, self.num_classes, self.dim, self.heads = params, num_classes, dim, list(heads)
        self.train_loss, self.val_acc, self.best = train_loss, val_acc, best

    @property
    def W(self):
        return self.params[:, :self.num_classes * self.dim].view(-1, self.num_classes, self.dim)

    @property
    def b(self):
        return self.params[:, self.num_classes * self.dim:]

    def _head(self, who, head):
        head = self.best if head is None else head
        if isinstance(head, bool) or not isinstance(head, int) or not 0 <= head < self.params.shape[0]:
            raise ValueError(f"{who}: head={head!r} must be an int in [0, {self.params.shape[0]})")
        return head

    @torch.no_grad()
    def predict(self, x, *, head=None, batch_queries=262144):
        """x [Q, dim] fp32 CUDA -> (probs [Q, nc] fp32 = softmax(W z + b), pred [Q] int64 = argmax, lowest class on ties) of one head
        (default: best).  Queries run in chunks of batch_queries; the result is bitwise the same for any chunk size."""
        head = self._head("LinearProbe.predict", head)
        x = _knn_features("LinearProbe.predict", "x", x)
        if x.shape[1] != self.dim or x.device != self.params.device:
            raise ValueError(f"LinearProbe.predict: x {tuple(x.shape)} on {x.device} does not match dim {self.dim} on {self.params.device}")
        if isinstance(batch_queries, bool) or not isinstance(batch_queries, int) or batch_queries < 1:
            raise ValueError(f"LinearProbe.predict: batch_queries={batch_queries!r} must be a positive int")
        nc, Q = self.num_classes, x.shape[0]
        probs = torch.empty(Q, nc, device=x.device, dtype=torch.float32)
        pred = torch.empty(Q, device=x.device, dtype=torch.int64)
        p = self.params[head].contiguous()
        stream = torch.cuda.current_stream(x.device).cuda_stream
        for first in range(0, Q, batch_queries):
            last = min(first + batch_queries, Q)
            _lib.check(_lib.lib().msst_linprobe_predict(last - first, self.dim, nc, x[first:last].data_ptr(), p.data_ptr(),
                                                        probs[first:last].data_ptr(), pred[first:last].data_ptr(), stream))
        return probs, pred

    @torch.no_grad()
    def load_into(self, model, head=None):
        """Writes head `head` (default: best) into the default head of a ViTSpatialSpectral: LayerNorm weight 1 and bias 0 (so the
        head normalises as the probe does), the Linear's rows (pi*p1 + pj)*nc + c = W[c] and bias b[c] for every sub-pixel (pi, pj)
        of a spatial patch (HeadRearrange order).  The model then classifies windows as the probe classifies their embed_scene
        features.  Writes in place (copy_), so optimiser state built over the model's parameters stays valid."""
        head = self._head("LinearProbe.load_into", head)
        if not isinstance(model, ViTSpatialSpectral):
            raise ValueError(f"LinearProbe.load_into: needs a ViTSpatialSpectral, got {type(model).__name__}")
        if model.pixelwise or model.spectral_mlp_head:
            raise ValueError("LinearProbe.load_into: only the default head (LayerNorm + Linear per spatial patch) can take a probe; "
                             "this model has a pixelwise or spectral-MLP head")
        if model.dim != self.dim or model.num_classes != self.num_classes:
            raise ValueError(f"LinearProbe.load_into: model dim {model.dim} / num_classes {model.num_classes} do not match the probe's "
                             f"{self.dim} / {self.num_classes}")
        ln, lin = model.mlp_head[0], model.mlp_head[1]
        reps = model.patch_height * model.patch_width
        ln.weight.fill_(1.0)
        ln.bias.zero_()
        lin.weight.copy_(self.W[head].repeat(reps, 1))
        lin.bias.copy_(self.b[head].repeat(reps))


@torch.no_grad()
def linear_probe_fit(ref, ref_labels, *, num_classes, heads=((1e-3, 0.0),), epochs=100, batch_size=4096, seed=0, val=None):
    """Fits linear probes (softmax regression) on frozen features: the usual second probe of a self-supervised encoder next to k-NN,
    and the first step of linear-probe-then-fine-tune (LinearProbe.load_into).

    ref [N, dim] fp32 CUDA (dim a multiple of 32 in [32, 256], N < 2^31), ref_labels [N] integers in [0, num_classes), num_classes <= 256.
    Rows are normalised as F.layer_norm(x, (dim,)) does (no affine).  heads: 1 to 16 (lr, weight_decay) pairs, trained together in
    the same launches; W and b start at 0.  Per epoch: perm = torch.randperm(N, generator=g, device=ref.device) with one
    g = torch.Generator(ref.device).manual_seed(seed) for the whole fit, minibatches = consecutive slices of batch_size rows of perm
    (the last may be shorter), the minibatch mean of cross-entropy, torch.optim.AdamW (betas (0.9, 0.999), eps 1e-8, decoupled decay on
    W and b, one 1-based step counter over the fit).  Bitwise reproducible, and each head is bitwise the head fitted alone.
    val: optional (x_val [M, dim], y_val [M]): val_acc[h] = OA of head h on it, best = argmax (lowest index on ties).  Without val
    only one head is allowed (there is nothing to choose with).
    -> LinearProbe with train_loss [epochs, H] float64: per epoch the sum of its steps' CE sums, added in step order, over N."""
    who = "linear_probe_fit"
    if isinstance(num_classes, bool) or not isinstance(num_classes, int) or not 1 <= num_classes <= KNN_MAX_CLASSES:
        raise ValueError(f"{who}: num_classes={num_classes!r} must be an int in [1, {KNN_MAX_CLASSES}]")
    ref, ref_labels = _labelled_rows(who, ref, ref_labels, num_classes, "ref")
    heads = _linprobe_heads(who, heads)
    _int_arg(who, "epochs", epochs, 1)
    _int_arg(who, "batch_size", batch_size, 1)
    _int_arg(who, "seed", seed, 0)
    if val is not None:
        if not isinstance(val, (tuple, list)) or len(val) != 2:
            raise ValueError(f"{who}: val must be a pair (x_val, y_val)")
        xv, yv = _labelled_rows(who, val[0], val[1], num_classes, "val")
        if xv.shape[1] != ref.shape[1] or xv.device != ref.device:
            raise ValueError(f"{who}: val rows {tuple(xv.shape)} on {xv.device} do not match ref {tuple(ref.shape)} on {ref.device}")
    elif len(heads) > 1:
        raise ValueError(f"{who}: {len(heads)} heads need val=(x_val, y_val) to choose the best one")
    N, D = ref.shape
    H, nc, dev = len(heads), num_classes, ref.device
    batch = min(batch_size, N)
    params = torch.zeros(H, nc * D + nc, device=dev, dtype=torch.float32)
    m, v = torch.zeros_like(params), torch.zeros_like(params)
    dims = _linprobe_dims(N, D, nc, heads, batch=batch)
    workspace = torch.empty(_lib.lib().msst_linprobe_workspace(ctypes.byref(dims)) // 4, device=dev, dtype=torch.float32)
    steps_per_epoch = -(-N // batch)
    loss = torch.empty(epochs * steps_per_epoch, H, device=dev, dtype=torch.float32)
    g = torch.Generator(device=dev).manual_seed(seed)
    step = 0
    for _ in range(epochs):
        perm = torch.randperm(N, generator=g, device=dev)
        for first in range(0, N, batch):
            idx = perm[first:first + batch]
            step += 1
            dims.batch, dims.step = idx.numel(), step
            _linprobe_grad(dims, ref, ref_labels, idx, params, workspace)
            _linprobe_update(dims, workspace, params, m, v, loss[step - 1])
    sums = loss.cpu().double().numpy().reshape(epochs, steps_per_epoch, H).cumsum(axis=1)[:, -1]   # cumsum: in step order
    probe = LinearProbe(params, nc, D, heads, train_loss=torch.from_numpy(sums / N))
    if val is not None:
        acc = [float((probe.predict(xv, head=h)[1] == yv).double().mean()) for h in range(H)]
        probe.val_acc = torch.tensor(acc, dtype=torch.float64)
        probe.best = int(torch.argmax(probe.val_acc))
    return probe


@torch.no_grad()
def linear_probe_scene(model, scene, train_labels, *, num_classes, val_labels=None, heads=((1e-3, 0.0),), epochs=100, batch_size=4096,
                       seed=0, stride=None, weight=None, batch_windows=4096, ignore_index=-1, batch_queries=262144):
    """Linear probe of an encoder on whole scenes: embed_scene features, fitted on the labelled pixels of train_labels (validated on
    those of val_labels), then every pixel predicted.

    model, scene, stride, weight, batch_windows: as in embed_scene (a SimMIMSpatialSpectral checkpoint works directly).
    train_labels / val_labels [B, H, W] integers on the scene's device: a pixel is used when its label is != ignore_index and in
    [0, num_classes) (the rule of confusion_matrix).  heads, epochs, batch_size, seed: as in linear_probe_fit (several heads need
    val_labels).  Score the result against held-out labels with confusion_matrix / classification_metrics.
    -> (probs [B, num_classes, H, W] fp32, pred [B, H, W] int64 of the best head, the LinearProbe)."""
    who = "linear_probe_scene"
    labels, valid = _scene_labels(who, scene, train_labels, num_classes, ignore_index)
    if val_labels is not None:
        vlabels, vvalid = _scene_labels(who, scene, val_labels, num_classes, ignore_index, name="val_labels")
    _linprobe_heads(who, heads)
    if val_labels is None and len(heads) > 1:
        raise ValueError(f"{who}: {len(heads)} heads need val_labels to choose the best one")
    if not bool(valid.any()) or (val_labels is not None and not bool(vvalid.any())):
        raise ValueError(f"{who}: train_labels and val_labels need at least one labelled pixel each")
    feats = embed_scene(model, scene, stride=stride, weight=weight, batch_windows=batch_windows)   # [B, D, H, W]
    flat = _pixel_rows(feats)
    val = (flat[vvalid], vlabels[vvalid]) if val_labels is not None else None
    probe = linear_probe_fit(flat[valid], labels[valid], num_classes=num_classes, heads=heads, epochs=epochs, batch_size=batch_size,
                             seed=seed, val=val)
    probs, pred = probe.predict(flat, batch_queries=batch_queries)
    return _pixel_map(probs, feats), pred.reshape(feats.shape[0], *feats.shape[2:]), probe


KMEANS_MAX_K, KMEANS_MAX_RESTARTS, KMEANS_MAX_KD = 256, 16, 16384


def _kmeans_args(who, num_clusters, dim, n, restarts, iters, seed, normalize):
    """The checks of kmeans_fit that need no tensor: the feature width dim, K, R, iterations, seed, normalize and the row count n."""
    if isinstance(num_clusters, bool) or not isinstance(num_clusters, int) or not 1 <= num_clusters <= KMEANS_MAX_K:
        raise ValueError(f"{who}: num_clusters={num_clusters!r} must be an int in [1, {KMEANS_MAX_K}]")
    if dim % 32 or not 32 <= dim <= KNN_MAX_DIM:
        raise ValueError(f"{who}: feature width {dim} must be a multiple of 32 in [32, {KNN_MAX_DIM}]")
    if num_clusters * dim > KMEANS_MAX_KD:
        raise ValueError(f"{who}: num_clusters * dim = {num_clusters} * {dim} exceeds {KMEANS_MAX_KD} (the per-cluster sums live in "
                         f"shared memory)")
    if isinstance(restarts, bool) or not isinstance(restarts, int) or not 1 <= restarts <= KMEANS_MAX_RESTARTS:
        raise ValueError(f"{who}: restarts={restarts!r} must be an int in [1, {KMEANS_MAX_RESTARTS}]")
    _int_arg(who, "iters", iters, 1)
    _int_arg(who, "seed", seed, 0)
    if not isinstance(normalize, bool):
        raise ValueError(f"{who}: normalize={normalize!r} must be a bool")
    if not num_clusters <= n < 2 ** 31:
        raise ValueError(f"{who}: {n} rows; need num_clusters={num_clusters} <= rows < 2^31")


def _kmeans_dims(n, dim, k, restarts, normalize):
    return _lib.KmeansDims(n, dim, k, restarts, 1 if normalize else 0)


def _stream(t):
    return torch.cuda.current_stream(t.device).cuda_stream


def _kmeans_seed(dims, rnd, x, u, centroids, index, mindist, workspace):
    """One msst_kmeans_seed round (k-means++ choice `rnd` of every restart, then the mindist refresh unless it is the last)."""
    _lib.check(_lib.lib().msst_kmeans_seed(ctypes.byref(dims), rnd, x.data_ptr(), u.data_ptr(), centroids.data_ptr(), index.data_ptr(),
                                           mindist.data_ptr(), workspace.data_ptr(), _stream(x)))


def _kmeans_assign(dims, x, centroids, labels, dist=None, workspace=None):
    """One msst_kmeans_assign launch: labels [R, n] (and dist [R, n]); with a workspace also the slice partials of the update."""
    _lib.check(_lib.lib().msst_kmeans_assign(ctypes.byref(dims), x.data_ptr(), centroids.data_ptr(), labels.data_ptr(),
                                             dist.data_ptr() if dist is not None else None,
                                             workspace.data_ptr() if workspace is not None else None, _stream(x)))


def _kmeans_update(dims, workspace, centroids, inertia, changed, empty):
    """One msst_kmeans_update launch: new centroids in place, inertia [R] fp64, changed [R] / empty [R] int32."""
    _lib.check(_lib.lib().msst_kmeans_update(ctypes.byref(dims), workspace.data_ptr(), centroids.data_ptr(), inertia.data_ptr(),
                                             changed.data_ptr(), empty.data_ptr(), _stream(centroids)))


def _kmeans_uniforms(seed, restarts, k, device):
    """u [R, K] float64: restart r draws torch.rand(K) from torch.Generator(device).manual_seed(seed + r)."""
    return torch.stack([torch.rand(k, generator=torch.Generator(device=device).manual_seed(seed + r), device=device, dtype=torch.float64)
                        for r in range(restarts)])


class KMeans:
    """A k-means fit of R restarts.

    centroids [R, K, dim] fp32 (CUDA), in the space the rows were clustered in (normalised rows when normalize);
    inertia [R] float64: sum over the rows of the squared distance to their centroid, for the last assignment of the restart (the
    one that produced its centroids; for a converged restart that is its final centroids' own inertia);
    iterations [R] int64: assign + update passes run until the restart's labels stopped changing (iters when they never did);
    converged [R] bool; best: the restart of lowest inertia, lowest index on ties; seed_index [R, K] int64: the rows k-means++ chose
    (None for a fit from init)."""

    def __init__(self, centroids, inertia, iterations, converged, normalize, seed_index=None):
        self.centroids, self.inertia, self.iterations, self.converged = centroids, inertia, iterations, converged
        self.normalize, self.seed_index = normalize, seed_index
        self.best = int(torch.argmin(inertia))   # the first of equal minima

    @property
    def num_clusters(self):
        return self.centroids.shape[1]

    @torch.no_grad()
    def predict(self, x, *, restart=None, batch_queries=262144):
        """x [Q, dim] fp32 CUDA -> (labels [Q] int64 = the nearest centroid of restart `restart` (default: best), lowest index on ties;
        dist [Q] fp32 = the squared distance to it), rows normalised as in the fit.  Queries run in chunks of batch_queries; the result is
        bitwise the same for any chunk size."""
        who = "KMeans.predict"
        restart = self.best if restart is None else restart
        R, K, D = self.centroids.shape
        if isinstance(restart, bool) or not isinstance(restart, int) or not 0 <= restart < R:
            raise ValueError(f"{who}: restart={restart!r} must be an int in [0, {R})")
        x = _knn_features(who, "x", x)
        if x.shape[1] != D or x.device != self.centroids.device:
            raise ValueError(f"{who}: x {tuple(x.shape)} on {x.device} does not match dim {D} on {self.centroids.device}")
        if isinstance(batch_queries, bool) or not isinstance(batch_queries, int) or batch_queries < 1:
            raise ValueError(f"{who}: batch_queries={batch_queries!r} must be a positive int")
        Q = x.shape[0]
        if not Q < 2 ** 31:
            raise ValueError(f"{who}: {Q} rows; need rows < 2^31")
        labels = torch.empty(Q, device=x.device, dtype=torch.int64)
        dist = torch.empty(Q, device=x.device, dtype=torch.float32)
        c = self.centroids[restart].contiguous()
        for first in range(0, Q, batch_queries):
            last = min(first + batch_queries, Q)
            dims = _kmeans_dims(last - first, D, K, 1, self.normalize)
            _kmeans_assign(dims, x[first:last], c, labels[first:last], dist[first:last])
        return labels, dist


@torch.no_grad()
def kmeans_fit(x, num_clusters, *, restarts=1, iters=100, seed=0, normalize=True, init=None):
    """k-means (Lloyd's algorithm) on the device: the unsupervised probe of an encoder and the usual clustering of a scene.

    x [n, dim] fp32 CUDA, dim a multiple of 32 in [32, 256], num_clusters <= n < 2^31; 1 <= num_clusters <= 256 with
    num_clusters * dim <= 16384; 1 <= restarts <= 16.  normalize: cluster F.normalize(x, dim=1) (cosine geometry, the usual choice for
    self-supervised features); the rows are normalised on the fly and never stored.  Distances are squared Euclidean in fp32 in the
    direct difference form, a centroid is the mean of its rows (fp64 sums, not renormalised), an empty cluster keeps its centroid.
    Seeding: k-means++, restart r drawing its K uniforms from torch.Generator(x.device).manual_seed(seed + r), so restart r of a fit
    equals a one-restart fit with seed + r.  init: optional [restarts, num_clusters, dim] fp32 CUDA starting centroids (no seeding).
    Each iteration is one assignment and one update launch for all restarts; the fit stops when no restart changed a label, or after
    iters.  Bitwise reproducible; a restart does not depend on the others.
    -> KMeans."""
    who = "kmeans_fit"
    x = _knn_features(who, "x", x)
    n, D = x.shape
    _kmeans_args(who, num_clusters, D, n, restarts, iters, seed, normalize)
    R, K, dev = restarts, num_clusters, x.device
    if init is not None:
        if (not isinstance(init, torch.Tensor) or init.shape != (R, K, D) or init.dtype != torch.float32 or not init.is_cuda
                or init.device != dev):
            raise ValueError(f"{who}: init must be an fp32 tensor [{R}, {K}, {D}] on {dev}, got "
                             f"{tuple(init.shape) if isinstance(init, torch.Tensor) else type(init).__name__}"
                             f"{f' {init.dtype} on {init.device}' if isinstance(init, torch.Tensor) else ''}")
    dims = _kmeans_dims(n, D, K, R, normalize)
    workspace = torch.empty(_lib.lib().msst_kmeans_workspace(ctypes.byref(dims)), device=dev, dtype=torch.uint8)
    seed_index = None
    if init is not None:
        centroids = init.clone().contiguous()
    else:
        centroids = torch.empty(R, K, D, device=dev, dtype=torch.float32)
        seed_index = torch.empty(R, K, device=dev, dtype=torch.int64)
        u = _kmeans_uniforms(seed, R, K, dev)
        mindist = torch.empty(R, n, device=dev, dtype=torch.float32)
        for j in range(K):
            _kmeans_seed(dims, j, x, u, centroids, seed_index, mindist, workspace)
        del mindist
    labels = torch.full((R, n), -1, device=dev, dtype=torch.int64)
    inertia = torch.empty(R, device=dev, dtype=torch.float64)
    changed = torch.empty(R, device=dev, dtype=torch.int32)
    empty = torch.empty(R, device=dev, dtype=torch.int32)
    iterations = torch.full((R,), iters, dtype=torch.int64)
    converged = torch.zeros(R, dtype=torch.bool)
    for it in range(1, iters + 1):
        _kmeans_assign(dims, x, centroids, labels, workspace=workspace)
        _kmeans_update(dims, workspace, centroids, inertia, changed, empty)
        done = changed.cpu() == 0                      # the one read-back per iteration
        iterations[done & ~converged] = it
        converged |= done
        if bool(converged.all()):
            break
    return KMeans(centroids, inertia.cpu(), iterations, converged, normalize,
                  seed_index=seed_index.cpu() if seed_index is not None else None)


@torch.no_grad()
def cluster_scene(model, scene, *, num_clusters, restarts=1, iters=100, seed=0, normalize=True, stride=None, weight=None,
                  batch_windows=4096, batch_queries=262144):
    """k-means of an encoder's features on whole scenes: embed_scene, every pixel a row, kmeans_fit on all pixels, every pixel assigned
    to the nearest centroid of the best restart (the unsupervised segmentation of the scene).

    model, scene, stride, weight, batch_windows: as in embed_scene (a SimMIMSpatialSpectral checkpoint works directly).
    num_clusters, restarts, iters, seed, normalize: as in kmeans_fit; batch_queries: as in KMeans.predict.
    Score the result against ground truth with clustering_metrics.
    -> (clusters [B, H, W] int64, the KMeans)."""
    who = "cluster_scene"
    tiles = scene.tiles if isinstance(scene, RawTiles) else scene
    if not isinstance(tiles, torch.Tensor) or tiles.dim() != 4:
        raise ValueError(f"{who}: scene must be a [B, C, H, W] tensor or RawTiles")
    if not tiles.is_cuda:
        raise ValueError(f"{who}: the scene must be on a CUDA device")
    enc = model.encoder if isinstance(model, SimMIMSpatialSpectral) else model
    if not isinstance(enc, ViTSpatialSpectral):
        raise ValueError(f"{who}: needs a ViTSpatialSpectral encoder, got {type(enc).__name__}")
    B, _, H, W = tiles.shape
    _kmeans_args(who, num_clusters, enc.dim, B * H * W, restarts, iters, seed, normalize)
    if isinstance(batch_queries, bool) or not isinstance(batch_queries, int) or batch_queries < 1:
        raise ValueError(f"{who}: batch_queries={batch_queries!r} must be a positive int")
    feats = embed_scene(model, scene, stride=stride, weight=weight, batch_windows=batch_windows)   # [B, D, H, W]
    flat = _pixel_rows(feats)
    km = kmeans_fit(flat, num_clusters, restarts=restarts, iters=iters, seed=seed, normalize=normalize)
    clusters, _ = km.predict(flat, batch_queries=batch_queries)
    return clusters.reshape(B, H, W), km


def _min_cost_assignment(cost):
    """Rows of cost [n, m] (int64, n <= m) to distinct columns at the least total cost (the Hungarian method with potentials,
    O(n^2 m), one vectorised pass over the columns per step) -> col [n] int64."""
    n, m = cost.shape
    big = np.iinfo(np.int64).max // 4
    u, v = np.zeros(n + 1, np.int64), np.zeros(m + 1, np.int64)
    p, way = np.zeros(m + 1, np.int64), np.zeros(m + 1, np.int64)   # p[j]: 1-based row on column j (0: none); column 0 is the root
    for i in range(1, n + 1):
        p[0], j0 = i, 0
        minv = np.full(m + 1, big, np.int64)
        used = np.zeros(m + 1, bool)
        while True:
            used[j0] = True
            i0 = p[j0]
            free = ~used[1:]
            cur = cost[i0 - 1] - u[i0] - v[1:]
            better = free & (cur < minv[1:])
            minv[1:][better] = cur[better]
            way[1:][better] = j0
            cand = np.where(free, minv[1:], big)
            j1 = int(np.argmin(cand)) + 1
            delta = cand[j1 - 1]
            u[p[used]] += delta
            v[used] -= delta
            minv[~used] -= delta
            j0 = j1
            if p[j0] == 0:
                break
        while j0:
            j1 = way[j0]
            p[j0] = p[j1]
            j0 = j1
    col = np.full(n, -1, np.int64)
    rows = p[1:] > 0
    col[p[1:][rows] - 1] = np.nonzero(rows)[0]
    return col


def clustering_metrics(clusters, labels, *, num_clusters, num_classes, ignore_index=-1):
    """Scores a clustering against ground-truth classes on the host, in float64.  A pixel counts when its label is != ignore_index and in
    [0, num_classes) (the rule of confusion_matrix); its cluster must then lie in [0, num_clusters).  num_clusters, num_classes <= 256.
      contingency [nc, K] int64        pixels of class c in cluster k
      nmi            mutual information / ((H(classes) + H(clusters)) / 2), natural log; 1.0 when both sides have one occupied label
      ari            adjusted Rand index (Hubert and Arabie); 1.0 in the degenerate cases (both sides one label, or all singletons)
      hungarian_map [K] int64, oa_hungarian   the one-to-one cluster -> class matching with the most matched pixels (-1 for the
                     clusters left unmatched when K > nc) and the share of pixels it gets right
      majority_map [K] int64, oa_majority     each cluster to its most frequent class (lowest class on ties; class 0 for an empty
                     cluster) and the share of pixels that gets right
    With a map, map[clusters] is a class prediction for confusion_matrix / classification_metrics (AA, kappa); pixels of a cluster
    that hungarian_map leaves at -1 are outside the classes there, so score K > nc with majority_map.
    -> dict of the above (maps and contingency as CPU tensors, the scores as floats)."""
    who = "clustering_metrics"
    for name, v in (("num_clusters", num_clusters), ("num_classes", num_classes)):
        if isinstance(v, bool) or not isinstance(v, int) or not 1 <= v <= KMEANS_MAX_K:
            raise ValueError(f"{who}: {name}={v!r} must be an int in [1, {KMEANS_MAX_K}]")
    K, nc = num_clusters, num_classes
    cl, lab = torch.as_tensor(clusters), torch.as_tensor(labels)
    for name, t in (("clusters", cl), ("labels", lab)):
        if t.dtype.is_floating_point or t.dtype.is_complex or t.dtype == torch.bool:
            raise ValueError(f"{who}: {name} must be an integer tensor, got {t.dtype}")
    if cl.numel() != lab.numel():
        raise ValueError(f"{who}: {cl.numel()} clusters for {lab.numel()} labels")
    cl = cl.reshape(-1).to("cpu", torch.int64).numpy()
    lab = lab.reshape(-1).to("cpu", torch.int64).numpy()
    valid = (lab != ignore_index) & (lab >= 0) & (lab < nc)
    cl, lab = cl[valid], lab[valid]
    if cl.size == 0:
        raise ValueError(f"{who}: no labelled pixel")
    if bool(((cl < 0) | (cl >= K)).any()):
        raise ValueError(f"{who}: clusters outside [0, {K})")
    cont = np.bincount(lab * K + cl, minlength=nc * K).reshape(nc, K)
    N = float(cl.size)
    a, b = cont.sum(1).astype(np.float64), cont.sum(0).astype(np.float64)
    if np.count_nonzero(a) == 1 and np.count_nonzero(b) == 1:
        nmi = 1.0
    else:
        nz = cont > 0
        nij = cont[nz].astype(np.float64)
        outer = np.outer(a, b)[nz]
        mi = float(np.sum(nij / N * (np.log(nij) + math.log(N) - np.log(outer))))
        ent = lambda s: float(-np.sum(s[s > 0] / N * np.log(s[s > 0] / N)))
        nmi = mi / ((ent(a) + ent(b)) / 2)
    comb = lambda v: v * (v - 1) / 2
    index, sa, sb, pairs = float(comb(cont.astype(np.float64)).sum()), float(comb(a).sum()), float(comb(b).sum()), comb(N)
    expected = sa * sb / pairs if pairs > 0 else 0.0
    top = (sa + sb) / 2
    ari = 1.0 if top == expected else (index - expected) / (top - expected)
    hmap = np.full(K, -1, np.int64)
    if K <= nc:
        hmap[:] = _min_cost_assignment(-cont.T.astype(np.int64))
    else:
        hmap[_min_cost_assignment(-cont.astype(np.int64))] = np.arange(nc)
    matched = int(sum(cont[hmap[k], k] for k in range(K) if hmap[k] >= 0))
    mmap = cont.argmax(0).astype(np.int64)
    return dict(contingency=torch.from_numpy(cont.astype(np.int64)), nmi=nmi, ari=ari, oa_hungarian=matched / N,
                hungarian_map=torch.from_numpy(hmap), oa_majority=float(cont.max(0).sum()) / N, majority_map=torch.from_numpy(mmap))


MOMENTS_MAX_DIM = 256


def _moment_rows(who, x, dim=None):
    """x [n, dim] fp32 CUDA with 1 <= dim <= 256 (and == dim when given) -> contiguous x, else ValueError."""
    if not isinstance(x, torch.Tensor) or x.dim() != 2 or x.dtype != torch.float32 or not x.is_cuda:
        raise ValueError(f"{who}: x must be a 2-D fp32 CUDA tensor [rows, dim], got "
                         f"{tuple(x.shape) if isinstance(x, torch.Tensor) else type(x).__name__}"
                         f"{f' {x.dtype} on {x.device}' if isinstance(x, torch.Tensor) else ''}")
    D = x.shape[1]
    if not 1 <= D <= MOMENTS_MAX_DIM:
        raise ValueError(f"{who}: feature width {D} outside [1, {MOMENTS_MAX_DIM}]")
    if dim is not None and D != dim:
        raise ValueError(f"{who}: x has {D} features, the fit {dim}")
    if not x.shape[0] < 2 ** 31:
        raise ValueError(f"{who}: {x.shape[0]} rows; need rows < 2^31")
    return x.contiguous()


def _ridge_arg(who, ridge):
    if isinstance(ridge, bool) or not isinstance(ridge, (int, float)) or not 0 <= ridge < math.inf:
        raise ValueError(f"{who}: ridge={ridge!r} must be a finite number >= 0")
    return float(ridge)


def _moments_mean(x, workspace, mean):
    """msst_moments_mean: mean [dim] fp64 of x [n, dim] (the slice partials go to the workspace)."""
    _lib.check(_lib.lib().msst_moments_mean(x.shape[0], x.shape[1], x.data_ptr(), workspace.data_ptr(), mean.data_ptr(), _stream(x)))


def _moments_cov(x, mean, workspace, cov):
    """msst_moments_cov: cov [dim, dim] fp64 of x [n, dim] centred on mean (two passes)."""
    _lib.check(_lib.lib().msst_moments_cov(x.shape[0], x.shape[1], x.data_ptr(), mean.data_ptr(), workspace.data_ptr(), cov.data_ptr(),
                                           _stream(x)))


def _moments_project(x, mean, W, y=None, score=None):
    """msst_moments_project: y [n, k] = (x - mean) W^T and / or score [n] = sum_j y_j^2, for W [k, dim] fp64."""
    _lib.check(_lib.lib().msst_moments_project(x.shape[0], x.shape[1], W.shape[0], x.data_ptr(), mean.data_ptr(), W.data_ptr(),
                                               y.data_ptr() if y is not None else None,
                                               score.data_ptr() if score is not None else None, _stream(x)))


def _sign_rule(vecs):
    """Flips each row of vecs [k, dim] (numpy float64) so that its entry of largest |value| is positive, the lowest index on ties."""
    idx = np.argmax(np.abs(vecs), axis=1)
    flip = vecs[np.arange(vecs.shape[0]), idx] < 0
    vecs[flip] *= -1.0
    return vecs


class PCA:
    """Principal components of n rows of dim features, fitted by pca_fit.

    n; mean [dim] and covariance [dim, dim] float64 on the rows' device (covariance with the 1 / (n - 1) normalisation);
    eigenvalues [dim] float64, descending (as numpy.linalg.eigh returns them, so a zero-variance direction may show as -1e-17);
    components [dim, dim] float64, one unit eigenvector per row, in the order of the eigenvalues, each signed so that its entry of
    largest |value| is positive (the lowest index on ties), which keeps false-colour maps stable from run to run."""

    def __init__(self, n, mean, covariance, eigenvalues, components):
        self.n, self.mean, self.covariance, self.eigenvalues, self.components = n, mean, covariance, eigenvalues, components

    @property
    def dim(self):
        return self.mean.shape[0]

    @property
    def explained_variance_ratio(self):
        """[dim] float64: each eigenvalue (clipped at 0) over their sum."""
        lam = self.eigenvalues.clamp_min(0)
        return lam / lam.sum()

    def _whitening(self, who, k, ridge):
        """W [k, dim] float64 = components[:k] / sqrt(max(lambda, 0) + eps), eps = ridge * trace / dim."""
        eps = ridge * float(torch.diagonal(self.covariance).sum()) / self.dim
        den = self.eigenvalues[:k].clamp_min(0) + eps
        if not bool((den > 0).all()):
            raise ValueError(f"{who}: a zero-variance direction with ridge * trace / dim = {eps!r}; raise the ridge")
        return (self.components[:k] / torch.sqrt(den)[:, None]).contiguous()

    def _project(self, who, x, W, batch_queries, want_y):
        x = _moment_rows(who, x, self.dim)
        if x.device != self.mean.device:
            raise ValueError(f"{who}: x on {x.device}, the fit on {self.mean.device}")
        if isinstance(batch_queries, bool) or not isinstance(batch_queries, int) or batch_queries < 1:
            raise ValueError(f"{who}: batch_queries={batch_queries!r} must be a positive int")
        Q = x.shape[0]
        out = (torch.empty(Q, W.shape[0], device=x.device, dtype=torch.float32) if want_y
               else torch.empty(Q, device=x.device, dtype=torch.float32))
        for first in range(0, Q, batch_queries):
            last = min(first + batch_queries, Q)
            if want_y:
                _moments_project(x[first:last], self.mean, W, y=out[first:last])
            else:
                _moments_project(x[first:last], self.mean, W, score=out[first:last])
        return out

    @torch.no_grad()
    def transform(self, x, n_components=None, *, whiten=False, ridge=1e-6, batch_queries=262144):
        """x [Q, dim] fp32 CUDA -> y [Q, k] fp32, y_j = components[j] . (x - mean) in float64, rounded once (k = n_components, default
        dim).  whiten: y_j / sqrt(max(lambda_j, 0) + eps), eps = ridge * trace(covariance) / dim.  Queries run in chunks of batch_queries;
        the result is bitwise the same for any chunk size."""
        who = "PCA.transform"
        k = self.dim if n_components is None else n_components
        if isinstance(k, bool) or not isinstance(k, int) or not 1 <= k <= self.dim:
            raise ValueError(f"{who}: n_components={n_components!r} must be an int in [1, dim={self.dim}]")
        if not isinstance(whiten, bool):
            raise ValueError(f"{who}: whiten={whiten!r} must be a bool")
        ridge = _ridge_arg(who, ridge)
        W = self._whitening(who, k, ridge) if whiten else self.components[:k].contiguous()
        return self._project(who, x, W, batch_queries, True)

    @torch.no_grad()
    def mahalanobis(self, x, *, ridge=1e-6, batch_queries=262144):
        """x [Q, dim] fp32 CUDA -> [Q] fp32: the squared Mahalanobis distance (x - mean)^T (covariance + eps I)^-1 (x - mean),
        eps = ridge * trace(covariance) / dim, as the sum over all components of the whitened projections squared (eigenvalues clipped
        at 0), added in float64 and rounded once: the global RX anomaly score.  Bitwise the same for any batch_queries."""
        who = "PCA.mahalanobis"
        ridge = _ridge_arg(who, ridge)
        W = self._whitening(who, self.dim, ridge)
        return self._project(who, x, W, batch_queries, False)


@torch.no_grad()
def pca_fit(x):
    """Principal component analysis of rows on the device: csrc/moments.cu computes the fp64 mean and the two-pass fp64 covariance in a
    fixed order (bitwise reproducible), then the host takes numpy's float64 eigh of the (at most 256 x 256) covariance.

    x [n, dim] fp32 CUDA, 1 <= dim <= 256, 2 <= n < 2^31.  -> PCA."""
    who = "pca_fit"
    x = _moment_rows(who, x)
    n, D = x.shape
    if n < 2:
        raise ValueError(f"{who}: {n} rows; need at least 2")
    dev = x.device
    workspace = torch.empty(_lib.lib().msst_moments_workspace(n, D), device=dev, dtype=torch.uint8)
    mean = torch.empty(D, device=dev, dtype=torch.float64)
    cov = torch.empty(D, D, device=dev, dtype=torch.float64)
    _moments_mean(x, workspace, mean)
    _moments_cov(x, mean, workspace, cov)
    lam, vec = np.linalg.eigh(cov.cpu().numpy())
    lam, vec = lam[::-1].copy(), _sign_rule(vec[:, ::-1].T.copy())
    return PCA(n, mean, cov, torch.from_numpy(lam).to(dev), torch.from_numpy(vec).to(dev))


def _valid_rows(who, valid, B, H, W, device):
    """valid [B, H, W] bool on device (None: every pixel) -> flat [B*H*W] bool or None, else ValueError."""
    if valid is None:
        return None
    if not isinstance(valid, torch.Tensor) or valid.dtype != torch.bool or valid.shape != (B, H, W) or valid.device != device:
        raise ValueError(f"{who}: valid must be a bool tensor [{B}, {H}, {W}] on {device}")
    return valid.reshape(-1)


def _feature_width(who, model):
    """The feature width of embed_scene(model, ...), else ValueError."""
    enc = model.encoder if isinstance(model, SimMIMSpatialSpectral) else model
    if not isinstance(enc, ViTSpatialSpectral):
        raise ValueError(f"{who}: needs a ViTSpatialSpectral encoder, got {type(enc).__name__}")
    return enc.dim


def _scene_rows(who, model, scene, valid, stride, weight, batch_windows):
    """Checks a scene and its valid mask, then -> (feats [B, D, H, W] fp32, the pixel rows [B*H*W, D], the rows to fit on): the
    embed_scene features of model, or with model=None the scene's own spectra in model units (RawTiles: standardised and clipped,
    no pad bands)."""
    tiles = scene.tiles if isinstance(scene, RawTiles) else scene
    if not isinstance(tiles, torch.Tensor) or tiles.dim() != 4:
        raise ValueError(f"{who}: scene must be a [B, C, H, W] tensor or RawTiles")
    if not tiles.is_cuda:
        raise ValueError(f"{who}: the scene must be on a CUDA device")
    B, _, H, W = tiles.shape
    D = tiles.shape[1] if model is None else _feature_width(who, model)
    if not 1 <= D <= MOMENTS_MAX_DIM:
        raise ValueError(f"{who}: feature width {D} outside [1, {MOMENTS_MAX_DIM}]")
    keep = _valid_rows(who, valid, B, H, W, tiles.device)
    fit_n = B * H * W if keep is None else int(keep.sum())
    if not 2 <= fit_n < 2 ** 31:
        raise ValueError(f"{who}: {fit_n} pixels to fit on; need 2 <= pixels < 2^31")
    if model is None:
        feats = _model_units(scene, pad=False)
    else:
        feats = embed_scene(model, scene, stride=stride, weight=weight, batch_windows=batch_windows)
    flat = _pixel_rows(feats).contiguous()
    return feats, flat, (flat if keep is None else flat[keep])


@torch.no_grad()
def pca_scene(model, scene, *, n_components=3, valid=None, stride=None, weight=None, batch_windows=4096, batch_queries=262144):
    """PCA of an encoder's features on whole scenes: embed_scene, a fit on the pixels where valid [B, H, W] (bool, default every pixel)
    is set, every pixel projected on the first n_components components.  With n_components=3, false_colour(maps) is the usual picture
    of a self-supervised encoder's features.

    model, scene, stride, weight, batch_windows: as in embed_scene (a SimMIMSpatialSpectral checkpoint works directly);
    batch_queries: as in PCA.transform.  -> (maps [B, n_components, H, W] fp32, the PCA)."""
    who = "pca_scene"
    D = _feature_width(who, model)
    if isinstance(n_components, bool) or not isinstance(n_components, int) or not 1 <= n_components <= D:
        raise ValueError(f"{who}: n_components={n_components!r} must be an int in [1, dim={D}]")
    feats, flat, fit = _scene_rows(who, model, scene, valid, stride, weight, batch_windows)
    pca = pca_fit(fit)
    return _pixel_map(pca.transform(flat, n_components, batch_queries=batch_queries), feats), pca


@torch.no_grad()
def rx_scene(model, scene, *, ridge=1e-6, valid=None, stride=None, weight=None, batch_windows=4096, batch_queries=262144):
    """Global RX (Reed-Xiaoli) anomaly detection on whole scenes: every pixel scored by its squared Mahalanobis distance from the
    Gaussian (mean, covariance + eps I, eps = ridge * trace / dim) fitted on the pixels where valid [B, H, W] is set (default all).

    model: RX on its embed_scene features (model, scene, stride, weight, batch_windows as in embed_scene); None: RX on the scene's own
    spectra in model units, the classical baseline (a RawTiles scene standardised and clipped as the model sees it, without the pad
    bands, whose zero variance would make the covariance singular; stride / weight / batch_windows are not used).
    Score the map against ground truth with anomaly_metrics.  -> (scores [B, H, W] fp32, the PCA of the fit)."""
    who = "rx_scene"
    ridge = _ridge_arg(who, ridge)
    feats, flat, fit = _scene_rows(who, model, scene, valid, stride, weight, batch_windows)
    pca = pca_fit(fit)
    B, _, H, W = feats.shape
    return pca.mahalanobis(flat, ridge=ridge, batch_queries=batch_queries).reshape(B, H, W), pca


def _quantile_sorted(s, q):
    """Linear-interpolation quantile q of the sorted float64 vector s (numpy's default method)."""
    pos = q * (s.numel() - 1)
    i = min(int(math.floor(pos)), s.numel() - 1)
    j = min(i + 1, s.numel() - 1)
    t = pos - i
    a, b = float(s[i]), float(s[j])
    return a + t * (b - a) if t < 0.5 else b - (b - a) * (1 - t)


@torch.no_grad()
def false_colour(maps, *, lo=0.01, hi=0.99):
    """maps [B, 3, H, W] (e.g. pca_scene's first three components) -> an RGB image [B, 3, H, W] fp32 in [0, 1]: each channel clipped at
    its lo / hi quantiles over all pixels of all scenes (linear interpolation, numpy's default) and rescaled to [0, 1]; a channel whose
    two quantiles are equal maps to 0.  The quantiles come from one sort per channel (torch.quantile refuses more than 2^24 values)."""
    who = "false_colour"
    if not isinstance(maps, torch.Tensor) or maps.dim() != 4 or maps.shape[1] != 3 or not maps.dtype.is_floating_point:
        raise ValueError(f"{who}: maps must be a floating-point tensor [B, 3, H, W], got "
                         f"{tuple(maps.shape) if isinstance(maps, torch.Tensor) else type(maps).__name__}")
    if maps.numel() == 0:
        raise ValueError(f"{who}: maps is empty")
    for name, v in (("lo", lo), ("hi", hi)):
        if isinstance(v, bool) or not isinstance(v, (int, float)) or not 0 <= v <= 1:
            raise ValueError(f"{who}: {name}={v!r} must be a number in [0, 1]")
    if not lo < hi:
        raise ValueError(f"{who}: lo={lo!r} must be below hi={hi!r}")
    out = torch.empty(maps.shape, device=maps.device, dtype=torch.float32)
    for c in range(3):
        v = maps[:, c].double()
        s = torch.sort(v.reshape(-1)).values
        a, b = _quantile_sorted(s, lo), _quantile_sorted(s, hi)
        out[:, c] = ((v.clamp(a, b) - a) / (b - a)).float() if b > a else 0.0
    return out


ANOMALY_FPRS = (1e-3, 1e-2, 1e-1)


def anomaly_metrics(score, anomalies, valid=None):
    """Scores an anomaly map against ground truth on the host, in float64: any per-pixel score (rx_scene, |recon - scene| reduced over
    bands, ...) where larger means more anomalous.  score: a real tensor / array; anomalies: bool of the same shape; valid: optional
    bool of the same shape, the pixels that count (default all).  NaN scores among them are refused.
      auc                     the Mann-Whitney statistic: the share of (anomaly, background) pairs whose anomaly scores higher, tied
                              pairs counting 1/2 (= the area under the ROC below)
      n_anomalies, n_background
      thresholds, fpr, tpr    the ROC over the distinct scores t in descending order, a pixel counted anomalous when score >= t
                              (float64 CPU tensors)
      tpr_at_fpr              {f: the best TPR among the thresholds with FPR <= f} for f in 1e-3, 1e-2, 1e-1 (0.0 when none, the
                              threshold above every score)
    ValueError when either class is empty."""
    who = "anomaly_metrics"
    s = torch.as_tensor(score)
    a = torch.as_tensor(anomalies)
    if s.dtype == torch.bool or s.dtype.is_complex:
        raise ValueError(f"{who}: score must be a real tensor, got {s.dtype}")
    if a.dtype != torch.bool or a.shape != s.shape:
        raise ValueError(f"{who}: anomalies must be a bool tensor of the score's shape {tuple(s.shape)}, got {a.dtype} {tuple(a.shape)}")
    s = s.detach().reshape(-1).to("cpu", torch.float64).numpy()
    a = a.reshape(-1).cpu().numpy()
    if valid is not None:
        v = torch.as_tensor(valid)
        if v.dtype != torch.bool or v.numel() != s.size:
            raise ValueError(f"{who}: valid must be a bool tensor of the score's shape")
        v = v.reshape(-1).cpu().numpy()
        s, a = s[v], a[v]
    if np.isnan(s).any():
        raise ValueError(f"{who}: NaN scores")
    na, nb = int(a.sum()), int((~a).sum())
    if na == 0 or nb == 0:
        raise ValueError(f"{who}: {na} anomalous and {nb} background pixels; need both")
    u, inv = np.unique(s, return_inverse=True)
    tp_g = np.bincount(inv, weights=a.astype(np.float64), minlength=u.size)[::-1]   # per distinct score, descending
    fp_g = np.bincount(inv, weights=(~a).astype(np.float64), minlength=u.size)[::-1]
    tp, fp = np.cumsum(tp_g), np.cumsum(fp_g)
    auc = float(np.sum(fp_g * (tp - 0.5 * tp_g))) / (float(na) * float(nb))
    tpr, fpr = tp / na, fp / nb
    at = {f: float(tpr[fpr <= f].max()) if bool((fpr <= f).any()) else 0.0 for f in ANOMALY_FPRS}
    return dict(auc=auc, n_anomalies=na, n_background=nb, thresholds=torch.from_numpy(u[::-1].copy()),
                fpr=torch.from_numpy(fpr), tpr=torch.from_numpy(tpr), tpr_at_fpr=at)
