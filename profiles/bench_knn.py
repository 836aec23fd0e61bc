"""k-NN search + vote throughput (msst_knn_topk + msst_knn_vote, csrc/knn.cu) against the same-GPU PyTorch baseline.

    python profiles/bench_knn.py [--out FILE] [--reps 3] [--no-baseline]

Cases: D = 96 (the model's dim), k = 20, 20 classes, Q in {601 * 2384 (one Houston2018-sized scene), 65,536} queries against
N in {1e4, 1e5, 1e6} references.  Features are N(0, 1) rows from a fixed seed.  Per case:
  - ms of one msst_knn_topk + msst_knn_vote over all queries (CUDA events, median of --reps after one warm-up call), inputs already
    prepared; msst_knn_prepare of the queries is timed on its own;
  - tensor FLOP/s counting the products actually issued, 6 bf16 products x 2 * D per (query, reference) pair over the 128 x 128 tiles
    (padding included), against the 2,250 TFLOP/s dense BF16 data-sheet figure of one HGX B200 GPU;
  - the baseline: F.normalize, torch.mm in chunks of queries with TF32 off, torch.topk(k + 1), timed the same way (one call, after a
    one-chunk warm-up), and the agreement of the two: largest |score difference| over all k columns, and the share of queries whose index
    sets are equal among those where the baseline's k-th and (k+1)-th scores differ by more than 1e-4.
The GPU name and power limit are read in the same run.  Needs a CUDA device (no CPU fallback).
"""
import argparse
import ctypes
import json
import os
import statistics
import sys

import torch
import torch.nn.functional as F

sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))
from bench_scene import gpu_info   # noqa: E402  (also puts the repo on sys.path)

from maskedsst_b200 import _lib                      # noqa: E402
from maskedsst_b200.inference import _knn_prepare   # noqa: E402

BF16_PEAK = 2.25e15   # FLOP/s, HGX B200 data sheet, one GPU, dense
D, K, NC = 96, 20, 20
QS = [601 * 2384, 65536]
NS = [10 ** 4, 10 ** 5, 10 ** 6]


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


def baseline(ref, query, k, chunk):
    """F.normalize + chunked fp32 torch.mm (TF32 off) + torch.topk(k + 1) -> (scores [Q, k + 1], index [Q, k + 1])."""
    r = F.normalize(ref, dim=1, eps=1e-12)
    s_out = torch.empty(query.shape[0], k + 1, device=ref.device)
    i_out = torch.empty(query.shape[0], k + 1, device=ref.device, dtype=torch.int64)
    for a in range(0, query.shape[0], chunk):
        q = F.normalize(query[a:a + chunk], dim=1, eps=1e-12)
        s_out[a:a + chunk], i_out[a:a + chunk] = torch.topk(torch.mm(q, r.T), k + 1, dim=1)
    return s_out, i_out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=None)
    ap.add_argument("--reps", type=int, default=3)
    ap.add_argument("--no-baseline", action="store_true")
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("bench_knn: needs a CUDA device")
    torch.backends.cuda.matmul.allow_tf32 = False
    L = _lib.lib()
    res = dict(gpu=gpu_info(), dim=D, k=K, classes=NC, reps=args.reps, bf16_peak_flops=BF16_PEAK, cases=[])
    g = torch.Generator(device="cuda").manual_seed(0)
    stream = torch.cuda.current_stream().cuda_stream
    for Q in QS:
        query = torch.randn(Q, D, device="cuda", generator=g)
        qp = _knn_prepare(query)
        prep_ms = events_ms(lambda: _knn_prepare(query), args.reps)
        for N in NS:
            ref = torch.randn(N, D, device="cuda", generator=g)
            labels = torch.randint(0, NC, (N,), device="cuda", generator=g)
            rp = _knn_prepare(ref)
            scores = torch.empty(Q, K, device="cuda")
            index = torch.empty(Q, K, device="cuda", dtype=torch.int64)
            probs = torch.empty(Q, NC, device="cuda")
            pred = torch.empty(Q, device="cuda", dtype=torch.int64)
            dims = _lib.KnnDims(N, Q, D, K)

            def run():
                _lib.check(L.msst_knn_topk(ctypes.byref(dims), rp.data_ptr(), qp.data_ptr(), scores.data_ptr(), index.data_ptr(), stream))
                _lib.check(L.msst_knn_vote(Q, K, N, scores.data_ptr(), index.data_ptr(), labels.data_ptr(), NC, 0.07, probs.data_ptr(),
                                           pred.data_ptr(), stream))

            times = events_ms(run, args.reps)
            ms = statistics.median(times)
            issued = 6 * 2 * D * (-(-Q // 128) * 128) * (-(-N // 128) * 128)
            row = dict(Q=Q, N=N, ms=round(ms, 3), ms_all_reps=[round(t, 3) for t in times], query_prepare_ms=round(statistics.median(prep_ms), 3),
                       issued_tensor_flop=issued, tensor_TFLOPs=round(issued / ms / 1e9, 1), frac_of_bf16_peak=round(issued / (ms / 1e3) / BF16_PEAK, 3))
            if not args.no_baseline:
                chunk = max(1, min(Q, (2 << 30) // (4 * N)))     # <= 2 GiB of fp32 scores per chunk
                baseline(ref, query[:chunk], K, chunk)
                torch.cuda.synchronize()
                a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                a.record()
                bs, bi = baseline(ref, query, K, chunk)
                b.record()
                torch.cuda.synchronize()
                bms = a.elapsed_time(b)
                sep = (bs[:, K - 1] - bs[:, K]) > 1e-4
                same = (torch.sort(index, 1).values == torch.sort(bi[:, :K], 1).values).all(1)
                row.update(baseline_ms=round(bms, 3), baseline_chunk=chunk, speedup=round(bms / ms, 2),
                           max_abs_score_diff=float((scores - bs[:, :K]).abs().max()), separated_queries=int(sep.sum()),
                           index_sets_equal_where_separated=float(same[sep].float().mean()) if bool(sep.any()) else None)
                del bs, bi
            print(json.dumps(row), flush=True)
            res["cases"].append(row)
            del ref, rp, scores, index, probs, pred
            torch.cuda.empty_cache()
        del query, qp
    res["gpu_after"] = gpu_info()
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            json.dump(res, f, indent=1)
    print(json.dumps(dict(gpu=res["gpu"])))


if __name__ == "__main__":
    main()
