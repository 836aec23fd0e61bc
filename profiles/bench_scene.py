"""Whole-scene inference throughput (maskedsst_b200.inference.predict_scene), bf16 model, synthetic int16 scenes from a fixed seed.

    python profiles/bench_scene.py [--out FILE] [--batch-windows 4096] [--reps 3]

Cases: Houston-shaped [1, 48, 601, 2384] (zero-padded to 50 bands) at strides 8 / 4 / 2 and EnMAP-shaped [1, 200, 1024, 1024]
(with clip) at strides 8 / 4.  Per case:
  - seconds per scene: host clock around predict_scene ending in a device synchronise (median of --reps), and windows/s from it;
  - the split between the forward chunks and the blend, from CUDA events around every chunk's forward and blend (a separate pass
    that runs the driver's loop with events; its probabilities are checked equal to predict_scene's);
  - the blend kernel's algorithmic bytes (each chunk's logits read once + the acc / wsum rows it visits read and written) over its
    event time, against the 7.7 TB/s HBM3e data-sheet figure;
  - peak device memory during predict_scene (torch.cuda.max_memory_allocated), in all and above the model + int16 scene.
The GPU name and power limit are read in the same run.  Needs a CUDA device (no CPU fallback).
"""
import argparse
import json
import os
import statistics
import subprocess
import sys
import time

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

import maskedsst_b200 as M                                            # noqa: E402
from maskedsst_b200.inference import blend_windows, predict_scene, scene_windows   # noqa: E402
from oracle import maskedsst_oracle as O                              # noqa: E402

HBM_PEAK = 7.7e12   # B/s, HGX B200 data sheet, one GPU

CASES = [("houston", (1, 48, 601, 2384), 8), ("houston", (1, 48, 601, 2384), 4), ("houston", (1, 48, 601, 2384), 2),
         ("enmap", (1, 200, 1024, 1024), 8), ("enmap", (1, 200, 1024, 1024), 4)]


def gpu_info():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True)
    return dict(torch_name=torch.cuda.get_device_name(0), nvidia_smi=q.stdout.strip().splitlines()[:1])


def make_model(kw):
    spec = O.Spec(**kw)                                                  # depth 4, dim 96 (configs/config.yaml)
    m = M.ViTSpatialSpectral(image_size=spec.image_size, spatial_patch_size=spec.spatial_patch_size,
                             spectral_patch_size=spec.spectral_patch_size, num_classes=spec.num_classes, dim=spec.dim, depth=spec.depth,
                             heads=spec.heads, mlp_dim=spec.mlp_dim, channels=spec.channels, spectral_pos_embed=False,
                             precision="bf16")
    m.load_state_dict(O.synthetic_state_dict(spec, seed=3))
    return m.cuda().eval(), spec


def make_scene(tag, shape):
    rng = np.random.default_rng(1234)
    raw = torch.from_numpy(rng.integers(-400, 12000, shape).astype(np.int16)).cuda()
    nb = shape[1]
    means, stds = rng.uniform(1000, 3000, nb), rng.uniform(500, 1500, nb)
    if tag == "houston":
        return M.RawTiles(raw, means, stds, image_size=8, pad_bands=2)
    return M.RawTiles(raw, means, stds, image_size=8, clip=(-5.0, 5.0))


def visited_pixels(H, W, win, stride, grid, first, n):
    """Pixels the blend kernel visits for chunk [first, first + n) (msst_scene_blend: first window's top row .. last window's bottom)."""
    nwin = grid[0] * grid[1]

    def row(g):
        return (g // nwin) * H + min((g % nwin) // grid[1] * stride, H - win)
    return (row(first + n - 1) + win - row(first)) * W


def instrumented(model, rt, stride, batch_windows):
    """predict_scene's chunk loop with CUDA events around each forward and each blend."""
    B, _, H, W = rt.tiles.shape
    w, nc = model.image_size, model.num_classes
    ny, nx = scene_windows(H, W, w, stride)
    x = M.RawTiles(rt.tiles, rt.means, rt.stds, image_size=w, pad_bands=rt.pad_bands, clip=rt.clip, windows=(ny, nx),
                   stride=(stride, stride))
    acc = torch.zeros(B, nc, H, W, device="cuda")
    wsum = torch.zeros(B, H, W, device="cuda")
    ev = []
    blend_bytes = 0
    with torch.no_grad():
        for first in range(0, x.num_windows, batch_windows):
            n = min(batch_windows, x.num_windows - first)
            e = [torch.cuda.Event(enable_timing=True) for _ in range(3)]
            e[0].record()
            y = model(x.set_window_range(first, n)).reshape(n, nc, w, w).float().contiguous()
            e[1].record()
            blend_windows(y, acc, wsum, stride=(stride, stride), grid=(ny, nx), first=first)
            e[2].record()
            ev.append(e)
            blend_bytes += n * nc * w * w * 4 + visited_pixels(H, W, w, stride, (ny, nx), first, n) * (nc + 1) * 4 * 2
    torch.cuda.synchronize()
    fwd = sum(e[0].elapsed_time(e[1]) for e in ev) / 1e3
    blend = sum(e[1].elapsed_time(e[2]) for e in ev) / 1e3
    return acc / wsum[:, None], fwd, blend, blend_bytes, len(ev)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=None)
    ap.add_argument("--batch-windows", type=int, default=4096)
    ap.add_argument("--reps", type=int, default=3)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("bench_scene: needs a CUDA device")
    res = dict(gpu=gpu_info(), precision="bf16", batch_windows=args.batch_windows, reps=args.reps, cases=[])
    models = {}
    for tag, shape, stride in CASES:
        if tag not in models:
            models[tag] = make_model(O.HOUSTON if tag == "houston" else O.ENMAP)
        model, spec = models[tag]
        rt = make_scene(tag, shape)
        H, W = shape[2:]
        ny, nx = scene_windows(H, W, 8, stride)
        predict_scene(model, rt, stride=stride, batch_windows=args.batch_windows)   # warm-up (module loads, allocator)
        torch.cuda.synchronize()
        times = []
        for _ in range(args.reps):
            torch.cuda.reset_peak_memory_stats()
            base = torch.cuda.memory_allocated()
            t0 = time.perf_counter()
            probs, pred = predict_scene(model, rt, stride=stride, batch_windows=args.batch_windows)
            torch.cuda.synchronize()
            times.append(time.perf_counter() - t0)
        peak = torch.cuda.max_memory_allocated()
        p2, fwd, blend, bbytes, chunks = instrumented(model, rt, stride, args.batch_windows)
        nwin = ny * nx * shape[0]
        sec = statistics.median(times)
        row = dict(scene=tag, shape=list(shape), model_bands=spec.channels, num_classes=spec.num_classes, stride=stride,
                   windows=nwin, chunks=chunks, seconds_per_scene=round(sec, 4), seconds_all_reps=[round(t, 4) for t in times],
                   windows_per_s=round(nwin / sec), forward_s=round(fwd, 4), blend_s=round(blend, 5),
                   blend_share=round(blend / (fwd + blend), 4), blend_bytes=bbytes, blend_TBps=round(bbytes / blend / 1e12, 3),
                   blend_frac_of_7p7TBps=round(bbytes / blend / HBM_PEAK, 3), peak_mem_GB=round(peak / 1e9, 3),
                   peak_mem_above_model_and_scene_GB=round((peak - base) / 1e9, 3),
                   instrumented_equals_predict_scene=bool(torch.equal(p2, probs)),
                   pred_class_histogram=torch.bincount(pred.flatten(), minlength=spec.num_classes).tolist())
        print(json.dumps(row), flush=True)
        res["cases"].append(row)
        del probs, pred, p2, rt
        torch.cuda.empty_cache()
    res["gpu_after"] = gpu_info()
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            json.dump(res, f, indent=1)
    print(json.dumps(dict(gpu=res["gpu"])))


if __name__ == "__main__":
    main()
