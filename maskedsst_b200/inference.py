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
"""
import ctypes
import math

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
    tiles = scene.tiles if isinstance(scene, RawTiles) else scene
    if not isinstance(tiles, torch.Tensor) or tiles.dim() != 4:
        raise ValueError("knn_scene: scene must be a [B, C, H, W] tensor or RawTiles")
    B, _, H, W = tiles.shape
    if (not isinstance(train_labels, torch.Tensor) or train_labels.shape != (B, H, W) or train_labels.dtype.is_floating_point
            or train_labels.dtype == torch.bool or train_labels.device != tiles.device):
        raise ValueError(f"knn_scene: train_labels must be an integer tensor [{B}, {H}, {W}] on {tiles.device}")
    if not tiles.is_cuda:
        raise ValueError("knn_scene: the scene must be on a CUDA device")
    if isinstance(num_classes, bool) or not isinstance(num_classes, int) or not 1 <= num_classes <= KNN_MAX_CLASSES:
        raise ValueError(f"knn_scene: num_classes={num_classes!r} must be an int in [1, {KNN_MAX_CLASSES}]")
    labels = train_labels.reshape(-1).to(torch.int64)
    valid = (labels != ignore_index) & (labels >= 0) & (labels < num_classes)
    feats = embed_scene(model, scene, stride=stride, weight=weight, batch_windows=batch_windows)   # [B, D, H, W]
    D = feats.shape[1]
    flat = feats.permute(0, 2, 3, 1).reshape(B * H * W, D)   # the one copy: pixels as rows
    probs, pred = knn_classify(flat[valid], labels[valid], flat, num_classes=num_classes, k=k, temperature=temperature,
                               batch_queries=batch_queries)
    return probs.reshape(B, H, W, num_classes).permute(0, 3, 1, 2).contiguous(), pred.reshape(B, H, W)
