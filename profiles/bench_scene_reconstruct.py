"""Whole-scene masked-reconstruction throughput (maskedsst_b200.inference.reconstruct_scene), bf16 SimMIM model, synthetic int16 scenes
from a fixed seed.

    python profiles/bench_scene_reconstruct.py [--out FILE] [--batch-windows 4096] [--reps 3]

Cases: Houston-shaped [1, 48, 601, 2384] (zero-padded to 50 bands) and EnMAP-shaped [1, 200, 1024, 1024] (with clip), each at
strides 8 / 4; the encoder, scenes and statistics are bench_scene.py's, wrapped in SimMIMSpatialSpectral with the benchmark's masking
(ratio 0.7, 4-pixel cells, tube masking) and the per-block decoder; the mask is scene_mask(seed=0).  Per case:
  - seconds per scene: host clock around reconstruct_scene ending in a device synchronise (median of --reps), and windows/s from it;
  - the split between the forward chunks (window mask, patch embedding with the mask token, encoder) and the reconstruct kernel, from
    CUDA events around each (a separate pass that runs the driver's loop with events; its recon is checked bitwise equal to
    reconstruct_scene's);
  - the reconstruct kernel's algorithmic bytes (each chunk's tokens read once + the acc / wsum rows it visits read and written + the
    mask bytes of those rows) over its event time, against the 7.7 TB/s HBM3e data-sheet figure;
  - its FMAs: D per decoded value, p0 values per (hidden block, covering window) at each pixel, i.e. D * p0 * sum over pixels of
    (covering windows x hidden blocks); over its event time, against 148 SMs x 128 FP32 lanes x the SM clock nvidia-smi reports in
    this run (the current clock right after the case, and the maximum);
  - peak device memory during reconstruct_scene (torch.cuda.max_memory_allocated), in all and above the model + int16 scene + mask.
The GPU name and power limit are read in the same run.  Needs a CUDA device (no CPU fallback).
"""
import argparse
import json
import os
import statistics
import subprocess
import sys
import time

import torch

sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))
from bench_scene import HBM_PEAK, gpu_info, make_model, make_scene, visited_pixels   # noqa: E402  (also puts the repo on sys.path)

import maskedsst_b200 as M                                                      # noqa: E402
from maskedsst_b200.inference import (_patch_any, _window_mask, reconstruct_scene, reconstruct_windows, scene_mask,   # noqa: E402
                                      scene_windows)
from oracle import maskedsst_oracle as O                                        # noqa: E402

CASES = [("houston", (1, 48, 601, 2384), 8), ("houston", (1, 48, 601, 2384), 4),
         ("enmap", (1, 200, 1024, 1024), 8), ("enmap", (1, 200, 1024, 1024), 4)]


def sm_clocks():
    q = subprocess.run(["nvidia-smi", "--query-gpu=clocks.sm,clocks.max.sm", "--format=csv,noheader,nounits"], capture_output=True,
                       text=True)
    cur, mx = (int(v) for v in q.stdout.strip().splitlines()[0].split(","))
    return cur, mx


def make_simmim(kw):
    enc, spec = make_model(kw)
    torch.manual_seed(0)
    m = M.SimMIMSpatialSpectral(encoder=enc, masking_ratio=0.7, mask_patch_size=4, tube_masking=True, to_pixels_per_spectral_block=True)
    return m.cuda().eval(), spec


def instrumented(model, rt, mask, stride, batch_windows):
    """reconstruct_scene's chunk loop with CUDA events around each forward and each reconstruct launch."""
    enc = model.encoder
    B, _, H, W = rt.tiles.shape
    w, C, p0, p1 = enc.image_size, enc.num_spectral_patches, enc.patch_depth, enc.patch_height
    ny, nx = scene_windows(H, W, w, stride)
    x = M.RawTiles(rt.tiles, rt.means, rt.stds, image_size=w, pad_bands=rt.pad_bands, clip=rt.clip, windows=(ny, nx),
                   stride=(stride, stride))
    Wd, bd = (t.detach().float().contiguous() for t in model.to_pixels.kernel_params())
    acc = torch.zeros(B, C * p0, H, W, device="cuda")
    wsum = torch.zeros(B, H, W, device="cuda")
    pany = _patch_any(mask, p1)
    ev = []
    nbytes = 0
    with torch.no_grad():
        pos = enc._pos_rows()
        for first in range(0, x.num_windows, batch_windows):
            n = min(batch_windows, x.num_windows - first)
            e = [torch.cuda.Event(enable_timing=True) for _ in range(3)]
            e[0].record()
            wm = _window_mask(pany, p1, w, (stride, stride), (ny, nx), first, n)
            tokens = enc.to_patch_embedding._embed_img(x.set_window_range(first, n), pos=pos, mask_token=model.mask_token, mask=wm)
            tokens = enc.transformer_forward(tokens)
            e[1].record()
            reconstruct_windows(tokens, mask.view(torch.uint8), Wd, bd, acc, wsum, C=C, p0=p0, p1=p1, stride=(stride, stride),
                                grid=(ny, nx), first=first)
            e[2].record()
            ev.append(e)
            nbytes += tokens.numel() * 4 + visited_pixels(H, W, w, stride, (ny, nx), first, n) * ((C * p0 + 1) * 4 * 2 + C)
    torch.cuda.synchronize()
    fwd = sum(e[0].elapsed_time(e[1]) for e in ev) / 1e3
    rec = sum(e[1].elapsed_time(e[2]) for e in ev) / 1e3
    fmas = enc.dim * p0 * int((wsum.double() * mask.sum(1).double()).sum().item())   # wsum = covering windows (uniform weight)
    acc.div_(wsum[:, None])
    recon = torch.where(mask.repeat_interleave(p0, 1), acc, rt.standardize(rt.tiles, pad=True))
    return recon, fwd, rec, nbytes, fmas, len(ev)


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
        raise SystemExit("bench_scene_reconstruct: needs a CUDA device")
    res = dict(gpu=gpu_info(), precision="bf16", batch_windows=args.batch_windows, reps=args.reps, masking_ratio=0.7, mask_patch_size=4,
               tube_masking=True, decoder="BlockwiseToPixels", cases=[])
    models = {}
    for tag, shape, stride in CASES:
        if tag not in models:
            models[tag] = make_simmim(O.HOUSTON if tag == "houston" else O.ENMAP)
        model, spec = models[tag]
        rt = make_scene(tag, shape)
        B, _, H, W = shape
        mask = scene_mask(model, B, H, W, seed=0, device="cuda")
        ny, nx = scene_windows(H, W, 8, stride)
        nwin = ny * nx * B
        run = lambda: reconstruct_scene(model, rt, mask, stride=stride, batch_windows=args.batch_windows)   # noqa: E731
        run()                                                            # warm-up, then the peak-memory pass
        torch.cuda.synchronize()
        torch.cuda.reset_peak_memory_stats()
        base = torch.cuda.memory_allocated()
        run()
        torch.cuda.synchronize()
        peak = torch.cuda.max_memory_allocated()
        recon, times = timed(run, args.reps)
        r2, fwd, rec, nbytes, fmas, chunks = instrumented(model, rt, mask, stride, args.batch_windows)
        cur, mx = sm_clocks()
        sec = statistics.median(times)
        lanes = 148 * 128
        row = dict(scene=tag, shape=list(shape), model_bands=spec.channels, dim=spec.dim, spectral_blocks=spec.C, stride=stride,
                   windows=nwin, chunks=chunks, hidden_fraction=round(float(mask.float().mean()), 4),
                   seconds_per_scene=round(sec, 4), seconds_all_reps=[round(t, 4) for t in times], windows_per_s=round(nwin / sec),
                   forward_s=round(fwd, 4), reconstruct_s=round(rec, 5), reconstruct_share=round(rec / (fwd + rec), 4),
                   reconstruct_bytes=nbytes, reconstruct_TBps=round(nbytes / rec / 1e12, 3),
                   reconstruct_frac_of_7p7TBps=round(nbytes / rec / HBM_PEAK, 3), reconstruct_fmas=fmas,
                   reconstruct_TFMAps=round(fmas / rec / 1e12, 3), sm_clock_mhz=cur, sm_clock_max_mhz=mx,
                   fma_frac_of_fp32_at_current_clock=round(fmas / rec / (lanes * cur * 1e6), 4),
                   fma_frac_of_fp32_at_max_clock=round(fmas / rec / (lanes * mx * 1e6), 4),
                   peak_mem_GB=round(peak / 1e9, 3), peak_mem_above_model_scene_and_mask_GB=round((peak - base) / 1e9, 3),
                   instrumented_equals_reconstruct_scene=bool(torch.equal(r2, recon)), recon_finite=bool(torch.isfinite(recon).all()))
        print(json.dumps(row), flush=True)
        res["cases"].append(row)
        del recon, r2, rt, mask
        torch.cuda.empty_cache()
    res["gpu_after"] = gpu_info()
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            json.dump(res, f, indent=1)
    print(json.dumps(dict(gpu=res["gpu"])))


if __name__ == "__main__":
    main()
