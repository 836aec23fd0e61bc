"""k-means throughput (msst_kmeans_seed / _assign / _update, csrc/kmeans.cu) against the same Lloyd iteration in eager PyTorch on the
same GPU.

    python profiles/bench_kmeans.py [--out FILE] [--iters 20] [--reps 3] [--no-baseline]

Cases: n = 601 x 2384 = 1,432,784 rows (one Houston2018-sized scene, the query count of r05_knn.json), R = 8 restarts, normalize on, and
(dim, K) in {(96, 20), (96, 128), (256, 64)}.  The rows are 20 Gaussian blobs (means N(0, 0.5^2 I), unit noise) from a fixed seed.  The
feature matrix (550 MB at dim 96, 1.47 GB at dim 256) is larger than the 126 MB L2, so every pass reads it from HBM; the workspace
partials (R * ceil(n / 4096) * K * dim * 4 B) may stay in L2.  Per case:
  - iter_ms: CUDA events around --iters back-to-back Lloyd iterations (assign + update, no read-back between them), median of --reps;
    assign_ms / update_ms: the same for each launch alone; launches_per_iter from msst_launch_count; assign_no_workspace_ms: the
    assignment launch without a workspace (prediction: labels only, no per-tile fp64 sums, counts, inertia or changed labels), so
    assign_ms - assign_no_workspace_ms is the cost of the sums phase;
  - seed_round_ms: CUDA events around the K k-means++ rounds of all restarts, / K; launches_per_round;
  - fit_ms: host clock around kmeans_fit(iters=--iters) ending in a device synchronise (seeding + iterations + one 4-byte-per-restart
    read-back per iteration), and the iterations it ran;
  - assign kernel rates: it issues 2 FP32 instructions (FADD + FFMA) per row x centroid x feature x restart; fp32_frac = those over
    148 SMs x 128 lanes x the maximum SM clock nvidia-smi reports in this run x assign_ms.  hbm_bytes = n * dim * 4 (rows, read once:
    the restarts of a slice run side by side) + R * n * 16 (labels read and written) + the partials written; hbm_frac against 7.7 TB/s;
  - the baseline: one eager iteration for all restarts, per restart in chunks of 65,536 rows: torch.cdist (fp32, no matmul expansion
    shortcut: compute_mode='donot_use_mm_for_euclid_dist'), argmin, index_add_ of the rows and bincount, then the means; its ms (CUDA
    events, median of --reps) and the fraction of labels it assigns differently from the kernel on the same centroids.
The GPU name, power limit and SM clocks are read in the same run.  Needs a CUDA device (no CPU fallback).
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

from maskedsst_b200 import _lib                                                                               # noqa: E402
from maskedsst_b200.inference import (_kmeans_assign, _kmeans_dims, _kmeans_seed, _kmeans_uniforms, _kmeans_update,   # noqa: E402
                                      kmeans_fit)

N, R = 601 * 2384, 8
CASES = [(96, 20), (96, 128), (256, 64)]
HBM_PEAK = 7.7e12


def sm_clocks():
    q = subprocess.run(["nvidia-smi", "--query-gpu=clocks.sm,clocks.max.sm", "--format=csv,noheader,nounits"], capture_output=True, text=True)
    cur, mx = (float(v) for v in q.stdout.strip().splitlines()[0].split(","))
    return cur, mx


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


def blobs(D, g):
    means = 0.5 * torch.randn(20, D, device="cuda", generator=g)
    y = torch.randint(0, 20, (N,), device="cuda", generator=g)
    return means[y] + torch.randn(N, D, device="cuda", generator=g)


def eager_iter(y, cent, chunk=65536):
    """One Lloyd iteration of every restart in eager torch: labels [R, n] and the new centroids."""
    K, D = cent.shape[1:]
    labels, new = [], []
    for r in range(cent.shape[0]):
        lab = torch.empty(y.shape[0], device=y.device, dtype=torch.int64)
        for a in range(0, y.shape[0], chunk):
            lab[a:a + chunk] = torch.cdist(y[a:a + chunk], cent[r], compute_mode="donot_use_mm_for_euclid_dist").argmin(1)
        s = torch.zeros(K, D, device=y.device).index_add_(0, lab, y)
        cnt = torch.bincount(lab, minlength=K)
        new.append(torch.where(cnt[:, None] > 0, s / cnt[:, None].clamp_min(1), cent[r]))
        labels.append(lab)
    return torch.stack(labels), torch.stack(new)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=None)
    ap.add_argument("--iters", type=int, default=20)
    ap.add_argument("--reps", type=int, default=3)
    ap.add_argument("--no-baseline", action="store_true")
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("bench_kmeans: needs a CUDA device")
    L = _lib.lib()
    res = dict(gpu=gpu_info(), n=N, restarts=R, normalize=True, iters=args.iters, reps=args.reps, hbm_peak_TBps=HBM_PEAK / 1e12, cases=[])
    g = torch.Generator(device="cuda").manual_seed(0)
    for D, K in CASES:
        x = blobs(D, g)
        dims = _kmeans_dims(N, D, K, R, True)
        ws = torch.empty(L.msst_kmeans_workspace(ctypes.byref(dims)), device="cuda", dtype=torch.uint8)
        cent = torch.empty(R, K, D, device="cuda")
        index = torch.empty(R, K, device="cuda", dtype=torch.int64)
        mindist = torch.empty(R, N, device="cuda")
        u = _kmeans_uniforms(1, R, K, x.device)

        def seed_all():
            for j in range(K):
                _kmeans_seed(dims, j, x, u, cent, index, mindist, ws)

        n0 = L.msst_launch_count()
        seed_ms = statistics.median(events_ms(seed_all, args.reps))
        seed_launches = (L.msst_launch_count() - n0) / ((args.reps + 1) * K)
        init = cent.clone()
        labels = torch.full((R, N), -1, device="cuda", dtype=torch.int64)
        inertia = torch.empty(R, device="cuda", dtype=torch.float64)
        changed = torch.empty(R, device="cuda", dtype=torch.int32)
        empty = torch.empty(R, device="cuda", dtype=torch.int32)
        work = init.clone()

        def iters():
            for _ in range(args.iters):
                _kmeans_assign(dims, x, work, labels, workspace=ws)
                _kmeans_update(dims, ws, work, inertia, changed, empty)

        def assigns():
            for _ in range(args.iters):
                _kmeans_assign(dims, x, work, labels, workspace=ws)

        def updates():
            for _ in range(args.iters):
                _kmeans_update(dims, ws, work, inertia, changed, empty)

        n0 = L.msst_launch_count()
        it_ms = statistics.median(events_ms(iters, args.reps)) / args.iters
        launches = (L.msst_launch_count() - n0) / ((args.reps + 1) * args.iters)
        work.copy_(init)
        as_ms = statistics.median(events_ms(assigns, args.reps)) / args.iters
        up_ms = statistics.median(events_ms(updates, args.reps)) / args.iters
        plab = torch.empty(R, N, device="cuda", dtype=torch.int64)

        def predicts():
            for _ in range(args.iters):
                _kmeans_assign(dims, x, work, plab)

        pr_ms = statistics.median(events_ms(predicts, args.reps)) / args.iters
        del plab
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        km = kmeans_fit(x, K, restarts=R, iters=args.iters, seed=1)
        torch.cuda.synchronize()
        fit_ms = (time.perf_counter() - t0) * 1e3
        cur, mx = sm_clocks()
        instr = 2 * N * K * D * R
        S = -(-N // 4096)
        hbm = N * D * 4 + R * N * 16 + R * S * (K * D * 4 + K * 4 + 12)
        row = dict(dim=D, K=K, iter_ms=round(it_ms, 4), assign_ms=round(as_ms, 4), update_ms=round(up_ms, 4), assign_no_workspace_ms=round(pr_ms, 4),
                   launches_per_iter=launches, seed_round_ms=round(seed_ms / K, 4), launches_per_round=seed_launches,
                   fit_ms=round(fit_ms, 1), fit_iterations=km.iterations.tolist(), fit_converged=km.converged.tolist(),
                   assign_fp32_instr=instr, assign_fp32_Tinstr_per_s=round(instr / as_ms / 1e9, 2),
                   fp32_peak_Tinstr_per_s=round(148 * 128 * mx * 1e6 / 1e12, 1), fp32_frac=round(instr / (as_ms / 1e3) / (148 * 128 * mx * 1e6), 4),
                   assign_hbm_bytes=hbm, assign_hbm_TBps=round(hbm / as_ms / 1e9, 3), hbm_frac=round(hbm / (as_ms / 1e3) / HBM_PEAK, 4),
                   sm_clock_mhz=cur, sm_clock_max_mhz=mx)
        if not args.no_baseline:
            y = F.normalize(x, dim=1)
            c0 = init.clone()
            base = statistics.median(events_ms(lambda: eager_iter(y, c0), args.reps))
            blab, _ = eager_iter(y, c0)
            klab = torch.full((R, N), -1, device="cuda", dtype=torch.int64)
            _kmeans_assign(dims, x, c0, klab)
            row.update(baseline_iter_ms=round(base, 3), speedup=round(base / it_ms, 2),
                       baseline_label_mismatch=float((blab != klab).double().mean()))
            del y
        print(json.dumps(row), flush=True)
        res["cases"].append(row)
        del x, ws, mindist, labels
        torch.cuda.empty_cache()
    res["gpu_after"] = gpu_info()
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            json.dump(res, f, indent=1)
    print(json.dumps(dict(gpu=res["gpu"])))


if __name__ == "__main__":
    main()
