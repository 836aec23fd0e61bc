#!/usr/bin/env python
"""bench.py -- SimMIM pre-training step throughput (samples/s) of the B200-native MaskedSST hot path.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--batch B] [--precision bf16|fp32] [--impl reference] [--no-extra]
                    [--dump-outputs DIR]

Headline workload (BASELINE.json configs[1]): one SimMIM masked-pretraining step = forward + backward + AdamW (+ the reference's
grad clamp) of ViTSpatialSpectral(dim 96, depth 4+4, heads 8, mlp 64, dropout 0.1) on synthetic Houston2018-shaped
cubes [B, 50, 8, 8] (bands 48-49 zero), tube masking ratio 0.7 / mask patch 4, blockwise decoder, lr .008 wd .05
(configs/config.yaml, configs/pretrain_config.yaml of the reference).  Random-init weights, synthetic data; every step
starts from the same initial weights (Workload.w0), so its inputs and outputs are the same from run to run.

Prints ONE JSON line (rank 0).  `value` = whole-job samples/s with inputs (cubes + masks) resident in HBM;
`e2e` = the same step through the public nn.Module API with HOST inputs: pinned cube -> H2D, masks drawn inside model(img),
loss read back D2H every step.  The same line also carries (default invocation):
  extra               BASELINE configs[2]/[3] shapes and the reference's default batch, each timed like the headline:
                      EnMAP pretrain (B = 256/GPU), EnMAP finetune CE/Adam (B = 512/GPU), Houston B = 64 (eager and CUDA graph);
                      for N > 1 also strong-scaling legs (global batch 1024 / 4096 fixed) and the exposed all-reduce time
  gpu_eager_baseline  the reference algorithm (oracle port = plain torch ops) in stock PyTorch eager ON THIS GPU, fp32 and TF32
  cpu_baseline        the same port on the host cores (all cores, and the 4 threads the reference pins, pretrain.py:4-9)
  dp_parity           (N > 1) data-parallel step == single-process step on the gathered batch, checked before the timed region
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

FLOP_PER_SAMPLE_TRAIN = {"houston": 3.754e9, "enmap": 15.49e9}   # SURVEY.md §8(d): 3 x forward GEMM+attention FLOPs
SHAPES = {"houston": (50, 20, 5, 320), "enmap": (200, 8, 20, 1280)}   # channels, classes, C, T


def parse():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--batch", type=int, default=None, help="per-GPU batch (default 1024 ours / 32 reference)")
    ap.add_argument("--precision", default=os.environ.get("MSST_BENCH_PRECISION", "bf16"))
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--dataset", default="houston", choices=["houston", "enmap"])
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-extra", action="store_true", help="headline line only (no extra configs / eager baseline / parity legs)")
    ap.add_argument("--dropout", type=float, default=0.1)
    ap.add_argument("--workload", default="pretrain", choices=["pretrain", "finetune"],
                    help="pretrain = BASELINE configs[1] (default); finetune = CE classification step with Adam (configs[2])")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="after the timed steps, write what the last one computed (loss, updated parameters, gradients) as "
                         "DIR/<name>.npy.  The inputs (data, masks, dropout seeds, the weights every step starts from) are "
                         "seeded and the same every run, so two runs or two builds agree to rounding (float-atomic gradient "
                         "reductions: up to 6e-7 relative on a B200 at a 1000 W power limit)")
    a = ap.parse_args()
    if a.steps < 1:
        ap.error("--steps must be at least 1")
    if a.dump_outputs and a.impl != "ours":
        ap.error("--dump-outputs is written by --impl ours only")
    return a


def dist_env():
    return int(os.environ.get("RANK", 0)), int(os.environ.get("LOCAL_RANK", 0)), int(os.environ.get("WORLD_SIZE", 1))


# ------------------------------------------------------------------------------------------------------------
# Reference algorithm in stock PyTorch (the oracle port): CPU legs (cpu_baseline, --impl reference) and the same-box
# GPU-eager leg.  This is the ONLY place outside tests/ and smoke() that executes oracle/ -- as a baseline, never as product.
# ------------------------------------------------------------------------------------------------------------
def port_step_time(dataset, batch, steps, warmup, dropout, budget_s=25.0, device="cpu", threads=None, tf32=False):
    import numpy as np
    import torch
    from oracle import maskedsst_oracle as O
    cores = threads or os.cpu_count() or 1
    if device == "cpu":
        torch.set_num_threads(cores)
    else:
        torch.backends.cuda.matmul.allow_tf32 = tf32
        torch.backends.cudnn.allow_tf32 = tf32
    spec = O.Spec(**(O.HOUSTON if dataset == "houston" else O.ENMAP))
    sd = O.synthetic_state_dict(spec, seed=5, simmim=True)
    params = {k: v.clone().to(device).requires_grad_(True) for k, v in sd.items()}
    opt = torch.optim.AdamW(list(params.values()), lr=0.008, weight_decay=0.05)
    gen = O.MaskGen(spec.image_size, 4, 1, 0.7)
    x = O.synthetic_cube(spec, batch, seed=5, zero_pad_bands=2 if dataset == "houston" else 0).to(device)
    nm = int(0.7 * spec.T)
    np.random.seed(5)
    sync = (lambda: torch.cuda.synchronize()) if device != "cpu" else (lambda: None)
    times = []
    t_start = time.perf_counter()
    for it in range(warmup + steps):
        sync()
        t0 = time.perf_counter()
        mask, idx = gen.batch(batch, spec.C, nm, tube=True)         # host numpy generator, as the reference does every step
        mask, idx = mask.to(device), idx.to(device)
        opt.zero_grad()
        loss = O.simmim_forward(x, params, spec, mask, idx, drop=dropout)
        loss.backward()
        for p in params.values():            # pretrain.py:71-73 elementwise clamp
            if p.grad is not None:
                p.grad.clamp_(-1, 1)
        opt.step()
        loss.item()
        sync()
        dt = time.perf_counter() - t0
        if it >= warmup:
            times.append(dt)
        if it >= warmup and time.perf_counter() - t_start > budget_s and len(times) >= 2:
            break
    times.sort()
    med = times[len(times) // 2]
    if device != "cpu":
        torch.backends.cuda.matmul.allow_tf32 = False
        torch.backends.cudnn.allow_tf32 = False
    return med, cores, len(times)


def run_reference(args):
    rank, _, world = dist_env()
    if rank != 0:
        return
    batch = args.batch or 32
    med, cores, n = port_step_time(args.dataset, batch, args.steps, min(args.warmup, 2), args.dropout, budget_s=120.0)
    v = batch / med
    line = {
        "impl": "reference", "metric": "simmim_pretrain_samples_per_sec", "value": v, "unit": "samples/s",
        "n_gpus": args.gpus, "steps": n, "warmup": min(args.warmup, 2), "ms_per_step": med * 1e3, "higher_is_better": True,
        "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": {"workload": f"SimMIM pretrain step (fwd+bwd+AdamW+clamp), ViTSpatialSpectral {args.dataset} shape, CPU",
                   "per_gpu_batch": batch, "dropout": args.dropout},
        "cpu_baseline": {"value": v, "unit": "samples/s", "cores": cores, "kind": "port",
                         "sample": f"{n} timed steps of batch {batch} (median), torch CPU fp32 oracle port of the reference"},
        "e2e": {"value": v, "unit": "samples/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
    }
    print(json.dumps(line), flush=True)


# ------------------------------------------------------------------------------------------------------------
# clocks sampler (nvidia-smi during the timed region)
# ------------------------------------------------------------------------------------------------------------
class Clocks:
    Q = "clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown," \
        "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap"

    def __init__(self, index):
        self.rows, self.proc, self.index = [], None, index

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--id={self.index}", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits",
                                          "-lms", "100"], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            threading.Thread(target=self._read, daemon=True).start()
        except Exception:
            self.proc = None

    def _read(self):
        for ln in self.proc.stdout:
            self.rows.append([c.strip() for c in ln.split(",")])

    def stop(self):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.15)
        self.proc.terminate()
        sm = sorted(int(float(r[0])) for r in self.rows if len(r) >= 7 and r[0].replace(".", "").isdigit())
        mx = [int(float(r[1])) for r in self.rows if len(r) >= 7 and r[1].replace(".", "").isdigit()]
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        reasons = [n for k, n in enumerate(names) if any(len(r) >= 7 and r[3 + k].lower().startswith("active") for r in self.rows)]
        return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_max_mhz": max(mx) if mx else None, "reasons": reasons,
                "samples": len(sm)}


# ------------------------------------------------------------------------------------------------------------
# one workload = (dataset shape, pretrain | finetune, per-GPU batch): model + optimiser + synthetic inputs + the two step functions
# ------------------------------------------------------------------------------------------------------------
class Workload:
    def __init__(self, ds, workload, B, dev, rank, world, precision, dropout, overlap=True, capturable=False):
        import numpy as np
        import torch
        import maskedsst_b200 as M
        from maskedsst_b200.optim import FusedAdam
        from maskedsst_b200.dp import GradSync, stage_boundaries
        self.ds, self.kind, self.B, self.dev, self.world = ds, workload, B, dev, world
        channels, ncls, _, _ = SHAPES[ds]
        self.channels = channels
        torch.manual_seed(5)
        np.random.seed(5 + rank)
        enc = M.ViTSpatialSpectral(image_size=8, spatial_patch_size=1, spectral_patch_size=10, num_classes=ncls, dim=96, depth=4,
                                   heads=8, mlp_dim=64, dropout=dropout, emb_dropout=dropout, channels=channels,
                                   spectral_pos_embed=False, blockwise_patch_embed=True, spectral_pos=list(range(channels // 10)),
                                   precision=precision)
        if workload == "finetune":   # finetune.py:116-135: Adam + L2, head lr .005 / rest .0005, CE(ignore_index=-1)
            self.model = enc.to(dev).train()
            head = [p for n, p in self.model.named_parameters() if "mlp_head" in n]
            rest = [p for n, p in self.model.named_parameters() if "mlp_head" not in n]
            self.opt = FusedAdam([{"params": head, "lr": 0.005}, {"params": rest, "lr": 0.0005}], lr=0.0005, weight_decay=0.005,
                                 decoupled=False, grad_scale=1.0 / world, capturable=capturable)
        else:
            self.model = M.SimMIMSpatialSpectral(encoder=enc, masking_ratio=0.7, mask_patch_size=4, tube_masking=True,
                                                 to_pixels_per_spectral_block=True).to(dev).train()
            self.opt = FusedAdam(self.model.parameters(), lr=0.008, weight_decay=0.05, decoupled=True, clamp=1.0, grad_scale=1.0 / world,
                                 capturable=capturable)
        # synthetic inputs: a pool of pinned host batches (per step a different one) + their masks / labels
        self.pool = pool = 4
        g = torch.Generator().manual_seed(1234 + rank)
        self.host_x = [torch.randn(B, channels, 8, 8, generator=g).pin_memory() for _ in range(pool)]
        if ds == "houston":
            for t in self.host_x:
                t[:, 48:] = 0
        self.dev_x = [t.to(dev) for t in self.host_x]
        if workload == "finetune":
            self.host_y = [torch.randint(-1, ncls, (B, 8, 8), generator=g).pin_memory() for _ in range(pool)]
            self.dev_y = [t.to(dev) for t in self.host_y]
        else:
            self.dev_masks = [self.model.draw_masks(B, dev) for _ in range(pool)]
        self.sync = GradSync(self.opt.arena, overlap=overlap, boundaries=stage_boundaries(self.model)) if world > 1 else None
        # Every step starts from these weights (the optimiser moments carry over).  The weight-gradient kernels reduce with
        # float atomics, so a step's gradients vary in the last bits from run to run; training on would feed that back and
        # amplify it (to ~20% of the parameters after 25 steps on a B200 at a 1000 W power limit).  From fixed weights each step's inputs are the same every run,
        # what it computes agrees to rounding, and the kernels do the same work as in training.
        self.w0 = self.opt.param_arena.clone()

    def restore_weights(self):
        self.opt.param_arena.copy_(self.w0)
        if self.opt.bf16_arena is not None:
            self.opt.bf16_arena.copy_(self.w0)

    def step_resident(self, i):
        from maskedsst_b200.dp import cross_entropy_dp
        self.restore_weights()
        self.opt.zero_grad()
        k = i % self.pool
        if self.kind == "finetune":
            loss = cross_entropy_dp(self.model(self.dev_x[k]), self.dev_y[k], ignore_index=-1)
        else:
            loss = self.model(self.dev_x[k], masks=self.dev_masks[k])
        loss.backward()
        if self.sync is not None:
            self.sync.finish()                                   # bucketed all-reduce overlapped with backward (hooks); this only drains it
        self.opt.step()
        return loss

    def step_e2e(self, i):
        from maskedsst_b200.dp import cross_entropy_dp
        k = i % self.pool
        x = self.host_x[k].to(self.dev, non_blocking=True)       # H2D from pinned memory, inside the timed region
        self.restore_weights()
        self.opt.zero_grad()
        if self.kind == "finetune":
            loss = cross_entropy_dp(self.model(x), self.host_y[k].to(self.dev, non_blocking=True), ignore_index=-1)
        else:
            loss = self.model(x)                                  # public API: model(img); masks drawn inside (see mask_backend)
        loss.backward()
        if self.sync is not None:
            self.sync.finish()
        self.opt.step()
        return loss.item()                                        # D2H read of the step's result

    def close(self):
        if self.sync is not None:
            self.sync.remove()


def barrier(world):
    import torch
    import torch.distributed as dist
    if world > 1:
        dist.barrier()
    torch.cuda.synchronize()


def max_over_ranks(x, dev, world):
    import torch
    import torch.distributed as dist
    t = torch.tensor([x], device=dev, dtype=torch.float64)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    return float(t.item())


def time_resident(w, steps, warmup):
    """W untimed warm-up steps, then exactly `steps` steps between barriers, CUDA events on the launching stream, max over ranks."""
    import torch
    from maskedsst_b200 import _lib
    for i in range(warmup):
        w.step_resident(i)
    barrier(w.world)
    n0 = _lib.lib().msst_launch_count()
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    ev0.record()
    for i in range(steps):
        loss = w.step_resident(i)
    ev1.record()
    barrier(w.world)
    launches = _lib.lib().msst_launch_count() - n0
    ms = max_over_ranks(ev0.elapsed_time(ev1), w.dev, w.world)
    return ms, launches, float(loss.item())


def dump_outputs(out_dir, model, loss):
    """What the timed step hands its caller, as of its last step: the loss, every updated parameter and every gradient, in
    float32.  The bench models have under 2 M parameters, so the whole set (< 16 MB) fits the 64 MB budget unsampled."""
    import numpy as np
    arrays = {"loss": np.asarray(loss, dtype=np.float32)}
    for name, p in model.named_parameters():
        arrays["param." + name] = p.detach().float().cpu().numpy()
        if p.grad is not None:
            arrays["grad." + name] = p.grad.detach().float().cpu().numpy()
    total = sum(a.nbytes for a in arrays.values())
    if total > 64 << 20:
        raise RuntimeError(f"--dump-outputs: {total} bytes exceed the 64 MB budget")
    os.makedirs(out_dir, exist_ok=True)
    for name, a in arrays.items():
        np.save(os.path.join(out_dir, name + ".npy"), a)


def time_e2e(w, steps, backend="device"):
    if hasattr(w.model, "mask_backend"):
        w.model.mask_backend = backend
    for i in range(2):
        w.step_e2e(i)
    barrier(w.world)
    t0 = time.perf_counter()
    for i in range(steps):
        w.step_e2e(i)
    barrier(w.world)
    return max_over_ranks(time.perf_counter() - t0, w.dev, w.world)


def extra_config(name, ds, kind, B, dev, rank, world, args, steps=8, warmup=3, graph=False, overlap=True):
    """One `extra` entry, timed like the headline (resident + e2e), fewer steps."""
    import torch
    w = Workload(ds, kind, B, dev, rank, world, args.precision, args.dropout, overlap=overlap, capturable=graph)
    out = {"name": name, "dataset": ds, "workload": kind, "per_gpu_batch": B, "global_batch": B * world, "steps": steps, "warmup": warmup}
    try:
        if graph:
            from maskedsst_b200.graph import GraphedStep
            inputs = (w.dev_x[0],) if kind == "pretrain" else (w.dev_x[0], w.dev_y[0])
            g = GraphedStep(w.model, w.opt, inputs)
            for i in range(warmup):
                g(*inputs)
            torch.cuda.synchronize()
            ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            ev0.record()
            for i in range(steps):
                g(w.dev_x[i % w.pool])
            ev1.record()
            torch.cuda.synchronize()
            ms = ev0.elapsed_time(ev1)
            out.update({"mode": "CUDA graph replay of the whole step (maskedsst_b200.graph.GraphedStep), masks drawn on the device"})
        else:
            ms, launches, loss = time_resident(w, steps, warmup)
            out.update({"gpu_launches_per_step": launches / steps, "final_loss": loss})
        sps = world * B * steps / (ms / 1e3)
        out.update({"ms_per_step": ms / steps, "samples_per_s": sps, "model_tflops_per_s": sps * FLOP_PER_SAMPLE_TRAIN[ds] / 1e12})
        if not graph:
            e2e_steps = 5
            s = time_e2e(w, e2e_steps)
            out["e2e_samples_per_s"] = world * B * e2e_steps / s
            out["h2d_bytes_per_step"] = w.host_x[0].numel() * 4
    finally:
        w.close()
        del w
        torch.cuda.empty_cache()
    return out


def dp_parity_check(dev, rank, world):
    """SURVEY §8(e): an N-rank data-parallel step (bucketed all-reduce, 1/world + clamp inside the optimiser) must equal the
    single-process step on the gathered global batch.  fp32 mode, dropout 0, 2 steps, per-rank batch 8: parameters are compared
    (a) across ranks (bit-equal: every rank applies the same reduced gradient) and (b) on rank 0 against the single-process run."""
    import torch
    import torch.distributed as dist
    import maskedsst_b200 as M
    from maskedsst_b200.optim import FusedAdam
    from maskedsst_b200.dp import GradSync, stage_boundaries
    Bl = 8

    def build():
        torch.manual_seed(11)
        enc = M.ViTSpatialSpectral(image_size=8, spatial_patch_size=1, spectral_patch_size=10, num_classes=20, dim=96, depth=2,
                                   heads=8, mlp_dim=64, dropout=0.0, emb_dropout=0.0, channels=50, spectral_pos_embed=False,
                                   blockwise_patch_embed=True, spectral_pos=list(range(5)), precision="fp32")
        return M.SimMIMSpatialSpectral(encoder=enc, masking_ratio=0.7, mask_patch_size=4, tube_masking=True,
                                       to_pixels_per_spectral_block=True).to(dev).train()

    g = torch.Generator().manual_seed(77)
    xs = torch.randn(2, world * Bl, 50, 8, 8, generator=g).to(dev)          # the same global batches on every rank
    m = build()
    masks_g = []
    for _ in range(2):                                                       # rank 0's draw is THE global mask pair
        mk, ix = m.draw_masks(world * Bl, dev)
        mk8, ix = mk.to(torch.uint8).contiguous(), ix.contiguous()
        dist.broadcast(mk8, 0)
        dist.broadcast(ix, 0)
        masks_g.append((mk8.bool(), ix))
    opt = FusedAdam(m.parameters(), lr=0.008, weight_decay=0.05, clamp=1.0, grad_scale=1.0 / world)
    sync = GradSync(opt.arena, boundaries=stage_boundaries(m))
    for s in range(2):
        sl = slice(rank * Bl, (rank + 1) * Bl)
        opt.zero_grad()
        m(xs[s, sl], masks=(masks_g[s][0][sl], masks_g[s][1][sl])).backward()
        sync.finish()
        opt.step()
    sync.remove()
    mine = opt.param_arena.clone()
    ref0 = mine.clone()
    dist.broadcast(ref0, 0)
    bit_equal = torch.tensor([int(torch.equal(mine, ref0))], device=dev)
    dist.all_reduce(bit_equal, op=dist.ReduceOp.MIN)
    res = {"ranks": world, "steps": 2, "per_rank_batch": Bl, "precision": "fp32", "params_bit_equal_across_ranks": bool(bit_equal.item())}
    if rank == 0:
        m1 = build()
        o1 = FusedAdam(m1.parameters(), lr=0.008, weight_decay=0.05, clamp=1.0)
        for s in range(2):
            o1.zero_grad()
            m1(xs[s], masks=masks_g[s]).backward()
            o1.step()
        err = float((o1.param_arena - mine).norm() / o1.param_arena.norm())
        res["rel_l2_vs_single_process_global_batch"] = err
        res["tolerance"] = 1e-5
        res["ok"] = bool(res["params_bit_equal_across_ranks"] and err <= 1e-5)
    okt = torch.tensor([int(res.get("ok", True))], device=dev)
    dist.broadcast(okt, 0)
    res["ok"] = bool(okt.item())
    return res


# ------------------------------------------------------------------------------------------------------------
def run_ours(args):
    import torch
    import torch.distributed as dist

    rank, local_rank, world = dist_env()
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)
    B = args.batch or 1024
    ds = args.dataset
    default_run = args.batch is None and ds == "houston" and args.workload == "pretrain" and not args.no_extra

    dp_parity = None
    if world > 1 and not args.no_extra:
        dp_parity = dp_parity_check(dev, rank, world)
        if not dp_parity["ok"]:
            if rank == 0:
                print(json.dumps({"error": "data-parallel parity check failed", "dp_parity": dp_parity}), flush=True)
            dist.destroy_process_group()
            sys.exit(3)

    w = Workload(ds, args.workload, B, dev, rank, world, args.precision, args.dropout)
    clocks = Clocks(local_rank)
    for i in range(args.warmup):
        w.step_resident(i)
    barrier(world)
    clocks.start()
    ms, launches, final_loss = time_resident(w, args.steps, 0)
    clk = clocks.stop()
    if args.dump_outputs and rank == 0:                          # before the e2e legs below train the model further
        dump_outputs(args.dump_outputs, w.model, final_loss)
    # e2e leg: (a) masks drawn on the device (module option mask_backend="device"), (b) the reference-compatible host generator
    e2e_steps = max(3, min(args.steps, 10))
    e2e_res = {b: time_e2e(w, e2e_steps, b) for b in (("device", "host") if args.workload == "pretrain" else ("device",))}
    h2d = w.host_x[0].numel() * 4
    channels = w.channels
    w.close()
    del w
    torch.cuda.empty_cache()

    extra = []
    if default_run:
        extra.append(extra_config("enmap_pretrain_b256", "enmap", "pretrain", 256, dev, rank, world, args))
        extra.append(extra_config("enmap_finetune_b512", "enmap", "finetune", 512, dev, rank, world, args))
        extra.append(extra_config("houston_pretrain_b64_reference_default_batch", "houston", "pretrain", 64, dev, rank, world, args, steps=20))
        if world == 1:
            extra.append(extra_config("houston_pretrain_b64_cuda_graph", "houston", "pretrain", 64, dev, rank, world, args, steps=20, graph=True))
        else:
            # all-reduce exposed time: the same step with the buckets reduced AFTER backward instead of overlapped with it
            a = extra_config("houston_pretrain_b1024_allreduce_after_backward", "houston", "pretrain", 1024, dev, rank, world, args, overlap=False)
            a["allreduce_exposed_ms"] = a["ms_per_step"] - ms / args.steps
            extra.append(a)
            for gb in (1024, 4096):                              # strong scaling: global batch fixed (SURVEY §8(d) config 4)
                if gb % world == 0:
                    extra.append(extra_config(f"houston_pretrain_strong_global{gb}", "houston", "pretrain", gb // world, dev, rank, world, args))

    if rank != 0:
        if world > 1:
            dist.destroy_process_group()
        return

    peaks = {}
    try:
        peaks = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
    except Exception:
        pass
    value = world * B * args.steps / (ms / 1e3)
    roof = roofline(args, B, dev, peaks)
    tf = value * FLOP_PER_SAMPLE_TRAIN[ds] / 1e12
    roof["step_tensor_frac"] = tf / world / peaks.get("bf16_tflops_sustained", 1400.0)
    roof["step_tensor_frac_note"] = "model TFLOP/s per GPU (3 x forward GEMM + attention FLOPs, recomputation not credited) / sustained bf16 peak"
    line = {
        "metric": "simmim_pretrain_samples_per_sec" if args.workload == "pretrain" else "finetune_samples_per_sec",
        "value": value, "unit": "samples/s", "n_gpus": world, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": ms / args.steps, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
        "dtype": "bf16" if args.precision == "bf16" else "f32", "data": "synthetic",
        "config": {"workload": ("SimMIM pretrain step (fwd+bwd+AdamW+clamp)" if args.workload == "pretrain" else
                                "finetune step (fwd+CE+bwd+Adam, 2 lr groups)") + f", ViTSpatialSpectral {ds} shape "
                               f"[B,{channels},8,8], dim 96 depth 4+4 heads 8 mlp 64, dropout {args.dropout}, tube mask 0.7/4",
                   "per_gpu_batch": B, "global_batch": B * world, "parallelism": f"dp{world}",
                   "l2_policy": "per-step working set (saved activations ~%.1f GB) exceeds the 126 MB L2; input pool of 4 batches"
                                % (B * SHAPES[ds][3] * 8 * 2.3e3 / 1e9),
                   "model_tflops_per_s": tf, "final_loss": final_loss},
        "e2e": {"value": world * B * e2e_steps / e2e_res["device"], "unit": "samples/s",
                "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": 4, "steps": e2e_steps,
                "masks": "drawn on the device inside model(img) (mask_backend='device')"},
        "gpu_launches": int(launches), "clocks": clk, "roofline": roof,
    }
    if "host" in e2e_res:
        line["e2e"]["value_host_masks"] = world * B * e2e_steps / e2e_res["host"]
        line["e2e"]["host_masks_note"] = "reference-compatible numpy generator on the host: +B*(T + 8*nm) H2D bytes per step"
    if extra:
        line["extra"] = extra
    if dp_parity is not None:
        line["dp_parity"] = dp_parity
    if not args.no_cpu_baseline and world == 1 and args.workload == "pretrain":
        med, cores, n = port_step_time(ds, 32, 8, 1, args.dropout, budget_s=15.0)
        line["cpu_baseline"] = {"value": 32 / med, "unit": "samples/s", "cores": cores, "kind": "port",
                                "sample": f"{n} timed steps of batch 32 (median) of the same step, torch CPU fp32 oracle port"}
        if default_run:
            med4, _, n4 = port_step_time(ds, 32, 4, 1, args.dropout, budget_s=12.0, threads=4)
            line["cpu_baseline_4_threads"] = {"value": 32 / med4, "unit": "samples/s", "cores": 4, "kind": "port",
                                              "sample": f"{n4} timed steps of batch 32, 4 threads as the reference pins (pretrain.py:4-9)"}
            line["gpu_eager_baseline"] = gpu_eager_baseline(ds, args.dropout, value, extra)
    print(json.dumps(line), flush=True)
    if world > 1:
        dist.destroy_process_group()


def gpu_eager_baseline(ds, dropout, ours_b1024, extra):
    """'The kernel to beat on the same box' (SURVEY §2.4): the reference algorithm (oracle port: the same torch ops the reference
    module issues, einsum instead of its per-block python loops -- generous to the baseline) in stock PyTorch eager on this GPU,
    torch.optim.AdamW (foreach), masks from the reference's host generator.  bf16 autocast is not possible for the reference
    (BlockwiseToPixels dtype crash, SURVEY C15), so fp32 and TF32."""
    import torch
    rows = []
    ours = {1024: ours_b1024}
    for e in extra:
        if e["name"].startswith("houston_pretrain_b64_reference"):
            ours[64] = e["samples_per_s"]
    for tf32 in (False, True):
        for b in (32, 64, 1024):
            try:
                med, _, n = port_step_time(ds, b, 6, 2, dropout, budget_s=6.0, device="cuda", tf32=tf32)
                r = {"precision": "tf32" if tf32 else "fp32", "batch": b, "ms_per_step": med * 1e3, "samples_per_s": b / med, "steps": n}
                if b in ours:
                    r["ours_over_eager"] = ours[b] / (b / med)
                rows.append(r)
            except Exception as e:   # noqa
                rows.append({"precision": "tf32" if tf32 else "fp32", "batch": b, "error": str(e)[:200]})
            torch.cuda.empty_cache()
    return {"what": "oracle port of the reference SimMIM step in stock PyTorch eager on cuda:0 (a baseline, not product code)", "rows": rows}


def _time_launch(fn, reps=10):
    import torch
    for _ in range(3):
        fn()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    torch.cuda.synchronize()
    e0.record()
    for _ in range(reps):
        fn()
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) / 1e3 / reps


def _traffic(kernel, R):
    """dram__bytes_read.sum + dram__bytes_write.sum per launch from the committed `ncu --set full` capture of this kernel at this
    shape (profiles/r02_ncu_traffic.json, written by profiles/ncu_traffic.py from the raw ncu CSV); None when no capture matches."""
    try:
        tab = json.load(open(os.path.join(ROOT, "profiles", "r02_ncu_traffic.json")))
        return tab.get(f"{kernel}@R={R}")
    except Exception:
        return None


def roofline(args, B, dev, peaks):
    """Roofline of the DOMINANT kernel of the step (largest share of the ncu launch list, profiles/r02_launches_*.summary.txt): the
    fused projection + attention BACKWARD kernel (attn_block_bwd_kernel: tcgen05 / TMEM / TMA), timed alone with CUDA events on the
    launching stream at the step's spatial-stack shape.  Its algorithmic HBM bytes per launch: R*(D*2 [h] + I*2 [dO] + H*4 [lse]) in,
    R*(3I*2 [dqkv] + D*4 [dh]) out; its tensor work: recomputation 2*R*D*3I + five 64x64x64 contractions per (64-token sequence,
    head) + data gradient 2*R*3I*D.  Both fractions are reported; `bound` names the larger.  `other_kernels`: the same kernel at the
    spectral-stack shape, the fused forward (with its out-projection / residual / LayerNorm tail, as the step runs it) at both shapes,
    and the weight-gradient GEMM that reads dqkv."""
    import ctypes as C
    import torch
    from maskedsst_b200 import _lib
    lib = _lib.lib()
    st = torch.cuda.current_stream().cuda_stream
    if args.precision != "bf16":
        return {"note": "roofline legs are measured for the bf16 (tcgen05) mode only"}
    Cb, T = SHAPES[args.dataset][2], SHAPES[args.dataset][3]
    R, H, I, D = B * T, 8, 512, 96
    hbm_peak = peaks.get("hbm_gbs", 6650.0)
    tc_peak = peaks.get("bf16_tflops", 1590.0)
    src = "measured (MEASURED_PEAKS.json)" if peaks else "fallback"
    out, others = {}, []
    try:
        h = torch.randn(R, D, device=dev).bfloat16()
        w = (torch.randn(3 * I, D, device=dev) * D ** -0.5).bfloat16()
        wt = w.t().contiguous()
        o = torch.empty(R, I, device=dev, dtype=torch.bfloat16)
        lse = torch.empty(R, H, device=dev)
        do = torch.randn(R, I, device=dev).bfloat16()
        dqkv = torch.empty(R, 3 * I, device=dev, dtype=torch.bfloat16)
        dh = torch.empty(R, D, device=dev)
        flush = torch.empty(256 << 20, device=dev, dtype=torch.uint8)
        bwd_bytes = R * (D * 2 + I * 2 + H * 4) + R * (3 * I * 2 + D * 4)
        # forward incl. its fused tail (out-projection + residual + LN2): h, x in; o, lse, xmid, h2, stats2 out
        fwd_bytes = R * (D * 2 + D * 4) + R * (I * 2 + H * 4 + D * 4 + D * 2 + 8)
        w_out = (torch.randn(D, I, device=dev) * I ** -0.5).bfloat16()
        b_out = torch.randn(D, device=dev); xres = torch.randn(R, D, device=dev); xmid = torch.empty(R, D, device=dev)
        h2 = torch.empty(R, D, device=dev, dtype=torch.bfloat16); stats2 = torch.empty(R, 2, device=dev)
        ln_w = torch.ones(D, device=dev); ln_b = torch.zeros(D, device=dev)

        def timed(fn):
            for _ in range(3):
                fn()
            tot = 0.0
            for _ in range(8):
                flush.zero_()                                    # L2 flush between timed launches
                e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                e0.record(); fn(); e1.record(); torch.cuda.synchronize()
                tot += e0.elapsed_time(e1)
            return tot / 8 / 1e3

        for shape, (n_seq, N, inner) in (("spatial", (B * Cb, 64, 1)), ("spectral", (B * 64, Cb, 64))):
            ad = _lib.AttnDims(n_seq, N, inner, H, 64, float(args.dropout), 1234, 16, _lib.PREC_BF16, None)
            fwd = lambda: _lib.check(lib.msst_attn_block_out_fwd(C.byref(ad), D, h.data_ptr(), w.data_ptr(), o.data_ptr(), lse.data_ptr(), w_out.data_ptr(),
                                                                 b_out.data_ptr(), xres.data_ptr(), xmid.data_ptr(), ln_w.data_ptr(), ln_b.data_ptr(),
                                                                 h2.data_ptr(), stats2.data_ptr(), 17, st))
            bwd = lambda: _lib.check(lib.msst_attn_block_bwd(C.byref(ad), D, h.data_ptr(), w.data_ptr(), wt.data_ptr(), do.data_ptr(), lse.data_ptr(),
                                                             dqkv.data_ptr(), dh.data_ptr(), st))
            sec_f, sec_b = timed(fwd), timed(bwd)
            fl_f = 2.0 * R * D * 3 * I + 2 * 2.0 * N * 64 * R * H + 2.0 * R * I * D
            fl_b = 2 * 2.0 * R * D * 3 * I + 5 * 2.0 * N * 64 * R * H
            for tag, sec, byts, fl, kern in (("backward", sec_b, bwd_bytes, fl_b, "attn_block_bwd_kernel"), ("forward", sec_f, fwd_bytes, fl_f, "attn_block_fwd_kernel")):
                hb, tc = byts / sec / 1e9 / hbm_peak, fl / sec / 1e12 / tc_peak
                what = "fused QKV projection + attention backward" if tag == "backward" else "fused QKV projection + attention + out-projection + residual + LN2 forward"
                row = {"kernel": f"{what} ({kern}, tcgen05/TMEM/TMA), {shape} stack shape",
                       "bound": "hbm" if hb >= tc else "tensor", "achieved": byts / sec / 1e9 if hb >= tc else fl / sec / 1e12,
                       "peak": hbm_peak if hb >= tc else tc_peak, "unit": "GB/s" if hb >= tc else "TFLOP/s", "frac": max(hb, tc),
                       "hbm_frac": hb, "tensor_frac": tc, "traffic": _traffic(f"{kern}:{shape}", R), "algorithmic_bytes": byts,
                       "algorithmic_flops": fl, "us_per_launch": sec * 1e6, "peak_source": src}
                if tag == "backward" and shape == "spatial":
                    out = row
                else:
                    others.append(row)
        x = h
        dW = torch.zeros(3 * I, D, device=dev)
        ld = _lib.LinearDims(R, 3 * I, D, 0, 0.0, 0, 0, _lib.PREC_BF16, None, 0)
        sec = timed(lambda: _lib.check(lib.msst_linear_bwd_weight(C.byref(ld), dqkv.data_ptr(), x.data_ptr(), dW.data_ptr(), None, st)))
        gb = R * (3 * I + D) * 2
        others.append({"kernel": "Wqkv weight-gradient GEMM dqkv^T h (gemm_wgrad_kernel: tcgen05, MN-major operands)", "bound": "hbm",
                       "achieved": gb / sec / 1e9, "peak": hbm_peak, "unit": "GB/s", "frac": gb / sec / 1e9 / hbm_peak,
                       "traffic": _traffic("gemm_wgrad_kernel:wqkv", R), "algorithmic_bytes": gb, "us_per_launch": sec * 1e6})
    except Exception as e:   # noqa
        out["error"] = str(e)
    out["other_kernels"] = others
    return out


if __name__ == "__main__":
    a = parse()
    if a.impl == "reference":
        run_reference(a)
    else:
        run_ours(a)
