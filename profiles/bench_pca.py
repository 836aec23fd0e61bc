"""PCA / RX throughput (msst_moments_mean / _cov / _project, csrc/moments.cu) against the same FP64 arithmetic in eager PyTorch on the
same GPU, and the share of pca_scene / rx_scene that embed_scene takes.

    python profiles/bench_pca.py [--out FILE] [--reps 5] [--no-scene]

Rows: n = 601 x 2384 = 1,432,784 (one Houston2018-sized scene), dim in {50, 96, 256}, correlated Gaussian rows offset by 10 from a fixed
seed (287 MB at dim 50, 1.47 GB at dim 256: larger than the 126 MB L2, so every pass reads them from HBM).  Per dim:
  - mean_ms, cov_ms, project_k3_ms (y only, k = 3: a false-colour map) and project_full_ms (k = dim with the score: RX): CUDA events
    around the launches, median of --reps after one warm-up;
  - fit_ms: host clock around pca_fit (mean, covariance, the 8 * dim^2-byte read-back and numpy's float64 eigh, the copies back) ending
    in a device synchronise, median of --reps;
  - rates: fp64 FMAs the algorithm needs (covariance n * dim (dim + 1) / 2, projection n * k * dim) x 2 FLOP over the kernel time,
    against 37 TFLOP/s FP64, the HGX B200 data sheet's 296 TFLOP/s for eight GPUs divided by eight (a data-sheet figure, not a measured
    peak); HBM bytes the algorithm needs (the rows once, plus y and the score) over the time, against 7.7 TB/s;
  - the baseline: eager torch float64 on the same GPU (x.double(), the mean, the centred c^T c in chunks of 262,144 rows, (c @ W^T) in
    the same chunks), its times by CUDA events, and the largest differences from the kernels (relative to max |cov| and max |y|).
Scenes (--no-scene skips them): bench_scene.py's bf16 Houston model and synthetic int16 601 x 2384 scene at stride 8: host clock
around embed_scene, pca_scene (3 components), rx_scene on the features and rx_scene(None, ...) on the raw spectra, each ending in a
device synchronise; the embed share = embed_scene / pca_scene and / rx_scene.
The GPU name, power limit and SM clocks are read in the same run.  Needs a CUDA device (no CPU fallback).
"""
import argparse
import json
import os
import statistics
import sys
import time

import torch

sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))
from bench_kmeans import events_ms, sm_clocks                                    # noqa: E402
from bench_scene import gpu_info, make_model, make_scene                        # noqa: E402  (also puts the repo on sys.path)

from maskedsst_b200 import _lib                                                 # noqa: E402
from maskedsst_b200.inference import (_moments_cov, _moments_mean, _moments_project, embed_scene, pca_fit, pca_scene,   # noqa: E402
                                      rx_scene)
from oracle import maskedsst_oracle as O                                        # noqa: E402

N = 601 * 2384
DIMS = [50, 96, 256]
FP64_PEAK = 296e12 / 8
HBM_PEAK = 7.7e12
CHUNK = 262144


def rows(D, g):
    mix = torch.randn(D, D, device="cuda", generator=g) / D ** 0.5 + torch.eye(D, device="cuda")
    return (torch.randn(N, D, device="cuda", generator=g) @ mix + 10.0).contiguous()


def eager(x, W):
    """float64 mean, covariance and projection in eager torch."""
    x64_mean = torch.zeros(x.shape[1], device="cuda", dtype=torch.float64)
    for a in range(0, N, CHUNK):
        x64_mean += x[a:a + CHUNK].double().sum(0)
    m = x64_mean / N
    cov = torch.zeros(x.shape[1], x.shape[1], device="cuda", dtype=torch.float64)
    for a in range(0, N, CHUNK):
        c = x[a:a + CHUNK].double() - m
        cov += c.T @ c
    cov /= N - 1
    y = torch.empty(N, W.shape[0], device="cuda", dtype=torch.float64)
    for a in range(0, N, CHUNK):
        y[a:a + CHUNK] = (x[a:a + CHUNK].double() - m) @ W.T
    return m, cov, y


def host_ms(fn, reps):
    fn()
    torch.cuda.synchronize()
    out = []
    for _ in range(reps):
        t0 = time.perf_counter()
        fn()
        torch.cuda.synchronize()
        out.append((time.perf_counter() - t0) * 1e3)
    return statistics.median(out)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=None)
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--no-scene", action="store_true")
    args = ap.parse_args()
    cur, mx = sm_clocks()
    res = dict(gpu=gpu_info(), sm_clock_mhz=cur, sm_clock_max_mhz=mx, n=N, reps=args.reps, fp64_peak_TFLOPs_datasheet=FP64_PEAK / 1e12,
               hbm_peak_TBps=HBM_PEAK / 1e12, cases=[])
    g = torch.Generator(device="cuda").manual_seed(9)
    for D in DIMS:
        x = rows(D, g)
        ws = torch.empty(_lib.lib().msst_moments_workspace(N, D), device="cuda", dtype=torch.uint8)
        mean = torch.empty(D, device="cuda", dtype=torch.float64)
        cov = torch.empty(D, D, device="cuda", dtype=torch.float64)
        _moments_mean(x, ws, mean)
        _moments_cov(x, mean, ws, cov)
        W = torch.linalg.qr(torch.randn(D, D, device="cuda", dtype=torch.float64, generator=g))[0].T.contiguous()
        y3 = torch.empty(N, 3, device="cuda")
        yf = torch.empty(N, D, device="cuda")
        sc = torch.empty(N, device="cuda")
        t = dict(
            mean_ms=statistics.median(events_ms(lambda: _moments_mean(x, ws, mean), args.reps)),
            cov_ms=statistics.median(events_ms(lambda: _moments_cov(x, mean, ws, cov), args.reps)),
            project_k3_ms=statistics.median(events_ms(lambda: _moments_project(x, mean, W[:3].contiguous(), y=y3), args.reps)),
            project_full_ms=statistics.median(events_ms(lambda: _moments_project(x, mean, W, y=yf, score=sc), args.reps)),
            fit_ms=host_ms(lambda: pca_fit(x), args.reps))
        fma_cov, fma_k3, fma_full = N * D * (D + 1) / 2, N * 3 * D, N * D * D
        row = dict(dim=D, workspace_MB=ws.numel() / 1e6, **t,
                   cov_fp64_TFLOPs=2 * fma_cov / t["cov_ms"] / 1e9, cov_fp64_frac=2 * fma_cov / t["cov_ms"] / 1e-3 / FP64_PEAK,
                   project_full_fp64_TFLOPs=2 * fma_full / t["project_full_ms"] / 1e9,
                   project_full_fp64_frac=2 * fma_full / t["project_full_ms"] / 1e-3 / FP64_PEAK,
                   project_k3_fp64_frac=2 * fma_k3 / t["project_k3_ms"] / 1e-3 / FP64_PEAK,
                   mean_hbm_frac=N * D * 4 / t["mean_ms"] / 1e-3 / HBM_PEAK,
                   cov_hbm_frac=N * D * 4 / t["cov_ms"] / 1e-3 / HBM_PEAK,
                   project_k3_hbm_frac=N * (D + 3) * 4 / t["project_k3_ms"] / 1e-3 / HBM_PEAK,
                   project_full_hbm_frac=N * (2 * D + 1) * 4 / t["project_full_ms"] / 1e-3 / HBM_PEAK)
        m64, cov64, y64 = eager(x, W)
        row["eager_fp64_ms"] = statistics.median(events_ms(lambda: eager(x, W), max(1, args.reps // 2)))
        row["eager_max_mean_diff_rel"] = float((mean - m64).abs().max() / m64.abs().max())
        row["eager_max_cov_diff_rel"] = float((cov - cov64).abs().max() / cov64.abs().max())
        _moments_project(x, mean, W, y=yf, score=sc)
        row["eager_max_y_diff_rel"] = float((yf.double() - y64).abs().max() / y64.abs().max())
        row["kernels_ms"] = t["mean_ms"] + t["cov_ms"] + t["project_full_ms"]
        row["speedup_vs_eager"] = row["eager_fp64_ms"] / row["kernels_ms"]
        del m64, cov64, y64, x, ws, yf
        torch.cuda.empty_cache()
        print(json.dumps(row), flush=True)
        res["cases"].append(row)
    if not args.no_scene:
        model, _ = make_model(O.HOUSTON)
        scene = make_scene("houston", (1, 48, 601, 2384))
        reps = max(1, args.reps // 2)
        s = dict(stride=8, dim=model.dim,
                 embed_scene_ms=host_ms(lambda: embed_scene(model, scene, stride=8), reps),
                 pca_scene_ms=host_ms(lambda: pca_scene(model, scene, stride=8), reps),
                 rx_scene_ms=host_ms(lambda: rx_scene(model, scene, stride=8), reps),
                 rx_raw_spectra_ms=host_ms(lambda: rx_scene(None, scene), reps))
        s["embed_share_of_pca_scene"] = s["embed_scene_ms"] / s["pca_scene_ms"]
        s["embed_share_of_rx_scene"] = s["embed_scene_ms"] / s["rx_scene_ms"]
        print(json.dumps(s), flush=True)
        res["scene"] = s
    res["gpu_after"] = gpu_info()
    res["sm_clock_after_mhz"] = sm_clocks()[0]
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            json.dump(res, f, indent=1)
    print(json.dumps(dict(gpu=res["gpu"])))


if __name__ == "__main__":
    main()
