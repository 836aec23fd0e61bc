"""Whole-scene embedding-map throughput (maskedsst_b200.inference.embed_scene), bf16 model, synthetic int16 scenes from a fixed seed.

    python profiles/bench_scene_embed.py [--out FILE] [--batch-windows 4096] [--reps 3]

Cases: Houston-shaped [1, 48, 601, 2384] (zero-padded to 50 bands) and EnMAP-shaped [1, 200, 1024, 1024] (with clip), each at
strides 8 / 4; the model, scenes and statistics are bench_scene.py's.  Per case:
  - seconds per scene: host clock around embed_scene ending in a device synchronise (median of --reps), and windows/s from it;
  - the split between the forward chunks and the embedding blend, from CUDA events around every chunk's forward_features and
    embed_windows (a separate pass that runs the driver's loop with events; its features are checked equal to embed_scene's);
  - the embedding kernel's algorithmic bytes (each chunk's tokens read once + the acc / wsum rows it visits read and written) over its
    event time, against the 7.7 TB/s HBM3e data-sheet figure;
  - peak device memory during embed_scene (torch.cuda.max_memory_allocated), in all and above the model + int16 scene;
  - predict_scene's windows/s on the same scene in the same run (median of --reps), for comparison.
The GPU name and power limit are read in the same run.  Needs a CUDA device (no CPU fallback).
"""
import argparse
import json
import os
import statistics
import sys
import time

import torch

sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))
from bench_scene import HBM_PEAK, gpu_info, make_model, make_scene, visited_pixels   # noqa: E402  (also puts the repo on sys.path)

import maskedsst_b200 as M                                                      # noqa: E402
from maskedsst_b200.inference import embed_scene, embed_windows, predict_scene, scene_windows   # noqa: E402
from oracle import maskedsst_oracle as O                                        # noqa: E402

CASES = [("houston", (1, 48, 601, 2384), 8), ("houston", (1, 48, 601, 2384), 4),
         ("enmap", (1, 200, 1024, 1024), 8), ("enmap", (1, 200, 1024, 1024), 4)]


def instrumented(model, rt, stride, batch_windows):
    """embed_scene's chunk loop with CUDA events around each forward and each embedding blend."""
    B, _, H, W = rt.tiles.shape
    w, D, C, p1 = model.image_size, model.dim, model.num_spectral_patches, model.patch_height
    ny, nx = scene_windows(H, W, w, stride)
    x = M.RawTiles(rt.tiles, rt.means, rt.stds, image_size=w, pad_bands=rt.pad_bands, clip=rt.clip, windows=(ny, nx),
                   stride=(stride, stride))
    acc = torch.zeros(B, D, H, W, device="cuda")
    wsum = torch.zeros(B, H, W, device="cuda")
    ev = []
    embed_bytes = 0
    with torch.no_grad():
        for first in range(0, x.num_windows, batch_windows):
            n = min(batch_windows, x.num_windows - first)
            e = [torch.cuda.Event(enable_timing=True) for _ in range(3)]
            e[0].record()
            tokens = model.forward_features(x.set_window_range(first, n))
            e[1].record()
            embed_windows(tokens, acc, wsum, C=C, p1=p1, stride=(stride, stride), grid=(ny, nx), first=first)
            e[2].record()
            ev.append(e)
            embed_bytes += tokens.numel() * 4 + visited_pixels(H, W, w, stride, (ny, nx), first, n) * (D + 1) * 4 * 2
    torch.cuda.synchronize()
    fwd = sum(e[0].elapsed_time(e[1]) for e in ev) / 1e3
    emb = sum(e[1].elapsed_time(e[2]) for e in ev) / 1e3
    return acc / wsum[:, None], fwd, emb, embed_bytes, len(ev)


def timed(fn, reps):
    fn()                                                                 # warm-up (module loads, allocator)
    torch.cuda.synchronize()
    times = []
    for _ in range(reps):
        t0 = time.perf_counter()
        out = fn()
        torch.cuda.synchronize()
        times.append(time.perf_counter() - t0)
    return out, times


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=None)
    ap.add_argument("--batch-windows", type=int, default=4096)
    ap.add_argument("--reps", type=int, default=3)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("bench_scene_embed: needs a CUDA device")
    res = dict(gpu=gpu_info(), precision="bf16", batch_windows=args.batch_windows, reps=args.reps, cases=[])
    models = {}
    for tag, shape, stride in CASES:
        if tag not in models:
            models[tag] = make_model(O.HOUSTON if tag == "houston" else O.ENMAP)
        model, spec = models[tag]
        rt = make_scene(tag, shape)
        H, W = shape[2:]
        ny, nx = scene_windows(H, W, 8, stride)
        nwin = ny * nx * shape[0]
        embed_scene(model, rt, stride=stride, batch_windows=args.batch_windows)   # warm-up, then the peak-memory pass
        torch.cuda.synchronize()
        torch.cuda.reset_peak_memory_stats()
        base = torch.cuda.memory_allocated()
        embed_scene(model, rt, stride=stride, batch_windows=args.batch_windows)
        torch.cuda.synchronize()
        peak = torch.cuda.max_memory_allocated()
        feats, times = timed(lambda: embed_scene(model, rt, stride=stride, batch_windows=args.batch_windows), args.reps)
        _, ptimes = timed(lambda: predict_scene(model, rt, stride=stride, batch_windows=args.batch_windows), args.reps)
        f2, fwd, emb, ebytes, chunks = instrumented(model, rt, stride, args.batch_windows)
        sec, psec = statistics.median(times), statistics.median(ptimes)
        row = dict(scene=tag, shape=list(shape), model_bands=spec.channels, dim=spec.dim, spectral_blocks=spec.C, stride=stride,
                   windows=nwin, chunks=chunks, seconds_per_scene=round(sec, 4), seconds_all_reps=[round(t, 4) for t in times],
                   windows_per_s=round(nwin / sec), forward_s=round(fwd, 4), embed_s=round(emb, 5),
                   embed_share=round(emb / (fwd + emb), 4), embed_bytes=ebytes, embed_TBps=round(ebytes / emb / 1e12, 3),
                   embed_frac_of_7p7TBps=round(ebytes / emb / HBM_PEAK, 3), peak_mem_GB=round(peak / 1e9, 3),
                   peak_mem_above_model_and_scene_GB=round((peak - base) / 1e9, 3),
                   instrumented_equals_embed_scene=bool(torch.equal(f2, feats)), features_finite=bool(torch.isfinite(feats).all()),
                   predict_scene_seconds_per_scene=round(psec, 4), predict_scene_windows_per_s=round(nwin / psec))
        print(json.dumps(row), flush=True)
        res["cases"].append(row)
        del feats, f2, rt
        torch.cuda.empty_cache()
    res["gpu_after"] = gpu_info()
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            json.dump(res, f, indent=1)
    print(json.dumps(dict(gpu=res["gpu"])))


if __name__ == "__main__":
    main()
