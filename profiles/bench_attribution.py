"""Input-gradient and integrated-gradients attribution throughput (msst_patch_embed_bwd_data, maskedsst_b200.inference.attribute_scene),
synthetic data from fixed seeds.

    python profiles/bench_attribution.py [--out FILE] [--reps 3]

  - msst_patch_embed_bwd_data at the Houston training shape (B = 1024, 50 bands, C = 5, P = 10, D = 96, blockwise) and the EnMAP shape
    (B = 1024, 200 bands, C = 20): CUDA-event time over 50 launches after a warm-up, with its algorithmic bytes (img read + d_tokens
    read + d_img written) over that time against the 7.7 TB/s HBM3e data-sheet figure; msst_patch_embed_bwd (the parameter gradients
    of the same shape) beside it for scale.  The inputs (~60 / 250 MB) exceed the 126 MB L2 at EnMAP only.
  - attribute_scene on bench_scene.py's Houston scene [1, 48, 601, 2384] (int16, 2 pad bands) with the bf16 encoder, stride 8, steps
    16 / 32, batch_samples 4096: seconds per scene (host clock around the call, ending in a synchronise; median of --reps) and
    interpolated samples per second; the split into gather + interpolation, forward, backward and msst_scene_attribute from CUDA events
    around each in a copy of the chunk loop (its result checked bitwise equal to attribute_scene's); peak device memory.
  - one chunk's backward under torch.profiler: time per kernel name, the share of weight-gradient GEMMs (gemm_wgrad) and of the fused
    MLP-block backward (data and weight gradients in one kernel), and the data-gradient kernel's time.
  - the same IG for one chunk (4096 samples) through the oracle's torch modules, fp32 eager on the same GPU, as a baseline.
The GPU name and power limit are read in the same run.  Needs a CUDA device.
"""
import argparse
import ctypes as C
import json
import os
import statistics
import sys
import time

import numpy as np
import torch

sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))
from bench_scene import HBM_PEAK, gpu_info, make_model, make_scene   # noqa: E402  (also puts the repo on sys.path)

from maskedsst_b200 import _lib                                     # noqa: E402
from maskedsst_b200.inference import (_AttributionMode, _gather_windows, _input_grads, _interpolate, _model_units,   # noqa: E402
                                      _objective_weights, attribute_scene, attribute_sum, scene_windows)
from oracle import maskedsst_oracle as O                            # noqa: E402


def ev_time(fn, reps=50):
    fn()
    torch.cuda.synchronize()
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record()
    for _ in range(reps):
        fn()
    b.record()
    torch.cuda.synchronize()
    return a.elapsed_time(b) / 1e3 / reps


def kernel_bench(tag, bands, B=1024):
    C_, G, p0, D = bands // 10, 8, 10, 96
    P, T = p0, C_ * G * G
    g = torch.Generator(device="cuda").manual_seed(0)
    r = lambda *s: torch.randn(*s, device="cuda", generator=g)
    img, dt = r(B, bands, 8, 8), r(B, T, D)
    pre_w, pre_b, W, bias, post_w, post_b = r(P), r(P), r(C_, D, P) / P ** 0.5, r(C_, D), r(D), r(D)
    out = torch.empty_like(img)
    grads = [torch.zeros_like(t) for t in (pre_w, pre_b, W, bias, post_w, post_b)] + [torch.zeros(T, D, device="cuda")]
    dims = _lib.EmbedDims(B, C_, G, p0, 1, D, C_, 0.0, 0, None, None)
    L, st = _lib.lib(), torch.cuda.current_stream().cuda_stream
    args = [img.data_ptr(), pre_w.data_ptr(), pre_b.data_ptr(), W.data_ptr(), bias.data_ptr(), post_w.data_ptr(), post_b.data_ptr(), None,
            dt.data_ptr(), None]
    t_data = ev_time(lambda: _lib.check(L.msst_patch_embed_bwd_data(C.byref(dims), *args, out.data_ptr(), st)))
    t_param = ev_time(lambda: _lib.check(L.msst_patch_embed_bwd(C.byref(dims), *args, *[x.data_ptr() for x in grads], None, st)))
    nbytes = 4 * (2 * img.numel() + dt.numel())
    return dict(shape=dict(B=B, bands=bands, C=C_, P=P, D=D), bwd_data_s=t_data, bwd_data_bytes=nbytes,
                bwd_data_TBps=nbytes / t_data / 1e12, bwd_data_share_of_hbm_peak=nbytes / t_data / HBM_PEAK, param_bwd_s=t_param)


def instrumented(model, rt, steps, stride, batch_samples):
    """attribute_scene's chunk loop with CUDA events around the gather, the forward, the backward and the step-sum blend."""
    bands, w, nc = model.num_spectral_patches * model.patch_depth, model.image_size, model.num_classes
    B, _, H, W = rt.tiles.shape
    ny, nx = scene_windows(H, W, w, stride)
    x = _model_units(rt, pad=True).contiguous()
    target = torch.zeros(B, H, W, dtype=torch.int64, device="cuda")
    base = torch.zeros(bands, device="cuda")
    acc = torch.zeros(B, bands, H, W, device="cuda")
    wsum = torch.zeros(B, H, W, device="cuda")
    total, step = B * ny * nx, max(1, batch_samples // steps)
    split = dict(gather_s=0.0, forward_s=0.0, backward_s=0.0, blend_s=0.0)
    pending = []
    with _AttributionMode(model):
        for first in range(0, total, step):
            n = min(step, total - first)
            e = [torch.cuda.Event(enable_timing=True) for _ in range(5)]
            e[0].record()
            xi = _interpolate(_gather_windows(x, w, (stride, stride), (ny, nx), first, n), base, steps).requires_grad_(True)
            dF = _objective_weights(_gather_windows(target, w, (stride, stride), (ny, nx), first, n), nc).repeat_interleave(steps, 0)
            e[1].record()
            with torch.enable_grad():
                y = model(xi)
                e[2].record()
                (gr,) = torch.autograd.grad(y, xi, dF)
            e[3].record()
            attribute_sum(gr.contiguous(), acc, wsum, steps=steps, stride=(stride, stride), grid=(ny, nx), first=first)
            e[4].record()
            pending.append(e)
    torch.cuda.synchronize()
    for e in pending:
        for k, (i, j) in zip(split, ((0, 1), (1, 2), (2, 3), (3, 4))):
            split[k] += e[i].elapsed_time(e[j]) / 1e3
    return (x - base[:, None, None]) * (acc / (steps * wsum[:, None])), split


def profile_chunk(model, rt, steps, n):
    x = _model_units(rt, pad=True)
    w = model.image_size
    xw = _gather_windows(x, w, (8, 8), scene_windows(*x.shape[2:], w, 8), 0, n)
    dF = _objective_weights(torch.zeros(n, w, w, dtype=torch.int64, device="cuda"), model.num_classes).repeat_interleave(steps, 0)
    xi = _interpolate(xw, torch.zeros(x.shape[1], device="cuda"), steps)
    with _AttributionMode(model):
        _input_grads(model, xi, dF)
        torch.cuda.synchronize()
        with torch.enable_grad():
            xr = xi.detach().requires_grad_(True)
            y = model(xr)
            torch.cuda.synchronize()
            with torch.profiler.profile(activities=[torch.profiler.ProfilerActivity.CUDA]) as prof:
                torch.autograd.grad(y, xr, dF)
                torch.cuda.synchronize()
    per = {}
    for ev in prof.events():
        if ev.device_type == torch.autograd.DeviceType.CUDA:
            per[ev.name] = per.get(ev.name, 0.0) + ev.device_time_total / 1e6
    tot = sum(per.values())
    share = lambda pred: sum(v for k, v in per.items() if pred(k)) / tot
    return dict(samples=n * steps, backward_kernel_s=tot, wgrad_gemm_share=share(lambda k: "wgrad" in k),
                fused_mlp_bwd_share=share(lambda k: "mlp" in k and "bwd" in k),
                bwd_data_kernel_s=sum(v for k, v in per.items() if "patch_embed_bwd_data" in k),
                per_kernel_s=dict(sorted(per.items(), key=lambda kv: -kv[1])))


def oracle_chunk(spec, n, steps, reps):
    sd = {k: v.cuda() for k, v in O.synthetic_state_dict(spec, seed=3).items()}
    xi = torch.randn(n * steps, spec.channels, 8, 8, device="cuda")
    dF = _objective_weights(torch.zeros(n * steps, 8, 8, dtype=torch.int64, device="cuda"), spec.num_classes)

    def run():
        x = xi.detach().requires_grad_(True)
        torch.autograd.grad(O.encoder_forward(x, sd, spec), x, dF)
    run()
    torch.cuda.synchronize()
    ts = []
    for _ in range(reps):
        t0 = time.perf_counter()
        run()
        torch.cuda.synchronize()
        ts.append(time.perf_counter() - t0)
    return dict(samples=n * steps, seconds=statistics.median(ts), samples_per_s=n * steps / statistics.median(ts))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=os.path.join(os.path.dirname(os.path.abspath(__file__)), "r10_attribution.json"))
    ap.add_argument("--reps", type=int, default=3)
    a = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("bench_attribution: needs a CUDA device")
    res = dict(gpu=gpu_info(), kernel={}, scene=[], oracle_fp32_eager=None)
    res["kernel"]["houston"] = kernel_bench("houston", 50)
    res["kernel"]["enmap"] = kernel_bench("enmap", 200)
    print(json.dumps(res["kernel"]), flush=True)
    model, spec = make_model(O.HOUSTON)
    rt = make_scene("houston", (1, 48, 601, 2384))
    B, _, H, W = rt.tiles.shape
    target = torch.zeros(B, H, W, dtype=torch.int64, device="cuda")
    ny, nx = scene_windows(H, W, 8, 8)
    for steps in (16, 32):
        ts = []
        torch.cuda.reset_peak_memory_stats()
        base_mem = torch.cuda.memory_allocated()
        for _ in range(a.reps):
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            attr = attribute_scene(model, rt, target, steps=steps, stride=8)
            torch.cuda.synchronize()
            ts.append(time.perf_counter() - t0)
        peak = torch.cuda.max_memory_allocated()
        inst, split = instrumented(model, rt, steps, 8, 4096)
        s = statistics.median(ts)
        row = dict(scene=[1, 48, H, W], stride=8, steps=steps, windows=ny * nx, samples=ny * nx * steps, seconds=s, all_seconds=ts,
                   samples_per_s=ny * nx * steps / s, split_s=split, instrumented_equal=bool(torch.equal(inst, attr)),
                   peak_mem_bytes=peak, peak_mem_above_start_bytes=peak - base_mem)
        res["scene"].append(row)
        print(json.dumps(row), flush=True)
    res["backward_profile"] = profile_chunk(model, rt, 32, 4096 // 32)
    print(json.dumps({k: v for k, v in res["backward_profile"].items() if k != "per_kernel_s"}), flush=True)
    res["oracle_fp32_eager"] = oracle_chunk(O.Spec(**O.HOUSTON), 4096 // 32, 32, a.reps)
    print(json.dumps(res["oracle_fp32_eager"]), flush=True)
    res["gpu_after"] = gpu_info()
    with open(a.out, "w") as f:
        json.dump(res, f, indent=1)
    print("wrote", a.out)


if __name__ == "__main__":
    main()
