"""Linear-probe fit and prediction throughput (msst_linprobe_grad + msst_linprobe_update, msst_linprobe_predict, csrc/linprobe.cu) against
the same probe in eager PyTorch on the same GPU.

    python profiles/bench_linprobe.py [--out FILE] [--epochs 100] [--reps 3] [--no-baseline]

Fit cases: N in {1e5, 1e6} references, D = 96 (the model's dim), 20 classes, H in {1, 8} heads, batch 4096, --epochs epochs.  The
features are 20 Gaussian blobs (class means N(0, 0.25^2 I), unit noise) from a fixed seed, so the probe learns something.  Per case:
  - fit_ms: host clock around the whole linear_probe_fit call (ending in a device synchronise), and ms per epoch = fit_ms / epochs;
  - launches_per_step from msst_launch_count over the fit (the torch.randperm launches are not ours and not counted);
  - kernel_ms_per_step: CUDA events around --reps x 200 back-to-back grad + update launches on the fit's minibatch shape (no Python
    between them), split into grad and update; ffma_TFLOPs = 4 * batch * D * nc * H (logits and dW, one FMA = 2 FLOP) over the grad
    kernel's time, against the FP32 peak 148 SMs x 128 lanes x 2 FLOP x the maximum SM clock that nvidia-smi reports in this run;
  - the baseline: F.layer_norm, one x @ W_all^T over all heads, per-head F.cross_entropy (summed, so each head gets its own gradient),
    backward, torch.optim.AdamW with one param group per head (betas (0.9, 0.999), eps 1e-8), on the same permutations; its fit_ms
    and the largest |probs| difference between the two fits over the first 65,536 references, every head.
Prediction case: Q = 601 x 2384 = 1,432,784 queries (one Houston2018-sized scene, the query count of r05_knn.json), one head of the
N = 1e5, H = 1 fit: CUDA-event ms (median of --reps after a warm-up), the eager softmax(F.layer_norm(q) @ W^T + b), and the largest
|probs| difference.  The GPU name, power limit and SM clocks are read in the same run.  Needs a CUDA device (no CPU fallback).
"""
import argparse
import ctypes
import json
import os
import statistics
import subprocess
import sys
import time

import torch
import torch.nn.functional as F

sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))
from bench_scene import gpu_info   # noqa: E402  (also puts the repo on sys.path)

from maskedsst_b200 import _lib                                                                # noqa: E402
from maskedsst_b200.inference import _linprobe_dims, _linprobe_grad, _linprobe_update, linear_probe_fit   # noqa: E402

D, NC, BATCH, Q = 96, 20, 4096, 601 * 2384
NS, HS = [10 ** 5, 10 ** 6], [1, 8]


def sm_clocks():
    q = subprocess.run(["nvidia-smi", "--query-gpu=clocks.sm,clocks.max.sm", "--format=csv,noheader,nounits"], capture_output=True, text=True)
    cur, mx = (float(v) for v in q.stdout.strip().splitlines()[0].split(","))
    return cur, mx


def heads_of(H):
    return [(10 ** -(2 + h % 3), 0.01 * (h % 2)) for h in range(H)]


def blobs(N, g):
    means = 0.25 * torch.randn(NC, D, device="cuda", generator=g)
    y = torch.randint(0, NC, (N,), device="cuda", generator=g)
    return means[y] + torch.randn(N, D, device="cuda", generator=g), y


def eager_fit(x, y, heads, epochs, seed):
    N = x.shape[0]
    Ws = [torch.zeros(NC, D, device="cuda", requires_grad=True) for _ in heads]
    bs = [torch.zeros(NC, device="cuda", requires_grad=True) for _ in heads]
    opt = torch.optim.AdamW([dict(params=[W, b], lr=lr, weight_decay=wd) for W, b, (lr, wd) in zip(Ws, bs, heads)], betas=(0.9, 0.999),
                            eps=1e-8)
    g = torch.Generator(device="cuda").manual_seed(seed)
    for _ in range(epochs):
        perm = torch.randperm(N, generator=g, device="cuda")
        for first in range(0, N, BATCH):
            idx = perm[first:first + BATCH]
            logits = F.layer_norm(x[idx], (D,)) @ torch.cat(Ws).T + torch.cat(bs)
            yi = y[idx]
            loss = sum(F.cross_entropy(logits[:, h * NC:(h + 1) * NC], yi) for h in range(len(heads)))
            opt.zero_grad(set_to_none=True)
            loss.backward()
            opt.step()
    return [(W.detach(), b.detach()) for W, b in zip(Ws, bs)]


def eager_probs(x, W, b):
    return torch.softmax(F.layer_norm(x, (D,)) @ W.T + b, -1)


def events_ms(fn, reps):
    fn()
    torch.cuda.synchronize()
    out = []
    for _ in range(reps):
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        fn()
        b.record()
        torch.cuda.synchronize()
        out.append(a.elapsed_time(b))
    return out


def kernel_step_ms(x, y, heads, reps, n_launch=200):
    """(grad ms, update ms) per launch at the fit's minibatch shape, CUDA events around n_launch back-to-back launches."""
    H = len(heads)
    P = NC * D + NC
    params = torch.zeros(H, P, device="cuda")
    m, v = torch.zeros_like(params), torch.zeros_like(params)
    dims = _linprobe_dims(x.shape[0], D, NC, heads, batch=BATCH)
    ws = torch.empty(_lib.lib().msst_linprobe_workspace(ctypes.byref(dims)) // 4, device="cuda")
    loss = torch.empty(H, device="cuda")
    idx = torch.randperm(x.shape[0], device="cuda")[:BATCH]

    def grads():
        for _ in range(n_launch):
            _linprobe_grad(dims, x, y, idx, params, ws)

    def updates():
        for i in range(n_launch):
            dims.step = i + 1
            _linprobe_update(dims, ws, params, m, v, loss)

    return statistics.median(events_ms(grads, reps)) / n_launch, statistics.median(events_ms(updates, reps)) / n_launch


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=None)
    ap.add_argument("--epochs", type=int, default=100)
    ap.add_argument("--reps", type=int, default=3)
    ap.add_argument("--no-baseline", action="store_true")
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("bench_linprobe: needs a CUDA device")
    torch.backends.cuda.matmul.allow_tf32 = False
    L = _lib.lib()
    res = dict(gpu=gpu_info(), dim=D, classes=NC, batch=BATCH, epochs=args.epochs, reps=args.reps, cases=[])
    g = torch.Generator(device="cuda").manual_seed(0)
    pred_probe = None
    for N in NS:
        x, y = blobs(N, g)
        for H in HS:
            heads = heads_of(H)
            val = (x[:4096], y[:4096]) if H > 1 else None
            linear_probe_fit(x[:BATCH], y[:BATCH], num_classes=NC, heads=heads, epochs=1, val=val)   # warm-up (module load, attributes)
            torch.cuda.synchronize()
            n0 = L.msst_launch_count()
            t0 = time.perf_counter()
            probe = linear_probe_fit(x, y, num_classes=NC, heads=heads, epochs=args.epochs, batch_size=BATCH, seed=1, val=val)
            torch.cuda.synchronize()
            fit_ms = (time.perf_counter() - t0) * 1e3
            steps = args.epochs * -(-N // BATCH)
            launches = L.msst_launch_count() - n0 - (H if val is not None else 0)   # minus the validation predictions
            grad_ms, upd_ms = kernel_step_ms(x, y, heads, args.reps)
            cur, mx = sm_clocks()
            peak = 148 * 128 * 2 * mx * 1e6
            flop = 4 * BATCH * D * NC * H
            row = dict(N=N, H=H, fit_ms=round(fit_ms, 1), ms_per_epoch=round(fit_ms / args.epochs, 3), steps=steps,
                       launches_per_step=launches / steps, kernel_ms_per_step=round(grad_ms + upd_ms, 4), grad_kernel_ms=round(grad_ms, 4),
                       update_kernel_ms=round(upd_ms, 4), kernel_share_of_fit=round(steps * (grad_ms + upd_ms) / fit_ms, 3),
                       ffma_flop_per_step=flop, ffma_TFLOPs=round(flop / grad_ms / 1e9, 2), fp32_peak_TFLOPs=round(peak / 1e12, 1),
                       frac_of_fp32_peak=round(flop / (grad_ms / 1e3) / peak, 4), sm_clock_mhz=cur, sm_clock_max_mhz=mx,
                       final_train_loss=[round(float(v), 4) for v in probe.train_loss[-1]])
            if not args.no_baseline:
                eager_fit(x[:BATCH], y[:BATCH], heads, 1, 1)
                torch.cuda.synchronize()
                t0 = time.perf_counter()
                eager = eager_fit(x, y, heads, args.epochs, 1)
                torch.cuda.synchronize()
                base_ms = (time.perf_counter() - t0) * 1e3
                xs = x[:65536]
                diff = max(float((probe.predict(xs, head=h)[0] - eager_probs(xs, *eager[h])).abs().max()) for h in range(H))
                row.update(baseline_fit_ms=round(base_ms, 1), baseline_ms_per_epoch=round(base_ms / args.epochs, 3),
                           speedup=round(base_ms / fit_ms, 2), max_abs_probs_diff=diff)
            print(json.dumps(row), flush=True)
            res["cases"].append(row)
            if N == NS[0] and H == 1:
                pred_probe = probe
        del x, y
        torch.cuda.empty_cache()
    q = torch.randn(Q, D, device="cuda", generator=g)
    times = events_ms(lambda: pred_probe.predict(q), args.reps)
    ms = statistics.median(times)
    cur, mx = sm_clocks()
    flop = 2 * Q * D * NC
    row = dict(case="predict", Q=Q, ms=round(ms, 3), ms_all_reps=[round(t, 3) for t in times], ffma_flop=flop,
               ffma_TFLOPs=round(flop / ms / 1e9, 2), frac_of_fp32_peak=round(flop / (ms / 1e3) / (148 * 128 * 2 * mx * 1e6), 4),
               hbm_bytes=Q * (D + NC) * 4 + Q * 8, hbm_TBps=round((Q * (D + NC) * 4 + Q * 8) / ms / 1e9, 2))
    if not args.no_baseline:
        W, b = pred_probe.W[0], pred_probe.b[0]
        eager_probs(q[:1024], W, b)
        bt = events_ms(lambda: torch.argmax(eager_probs(q, W, b), 1), args.reps)
        row.update(baseline_ms=round(statistics.median(bt), 3), speedup=round(statistics.median(bt) / ms, 2),
                   max_abs_probs_diff=float((pred_probe.predict(q)[0] - eager_probs(q, W, b)).abs().max()))
    print(json.dumps(row), flush=True)
    res["cases"].append(row)
    res["gpu_after"] = gpu_info()
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            json.dump(res, f, indent=1)
    print(json.dumps(dict(gpu=res["gpu"])))


if __name__ == "__main__":
    main()
