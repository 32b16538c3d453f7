#!/usr/bin/env python
"""bench.py -- throughput of the MonoDETR hot path on B200 (see DESIGN.md "Measurement").

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl b200|reference] [--workload model|msda|infer]
                    [--dump-outputs DIR]

Prints ONE JSON line (rank 0).  Workloads:
  model : full MonoDETR forward+backward, ResNet-50, 1280x384 synthetic images, train mode
          (BASELINE.json configs[2] at N=1: batch 8; configs[3] at N>1: batch 16 per GPU)
  msda  : the MSDeformAttn core alone, forward+backward, encoder shape (B=8, Lq=10200, 4 levels,
          8 heads x 32 ch, 4 points) -- BASELINE.json configs[1] family
`--impl reference` times the reference's CPU implementation of the same workload (the oracle port; the
Python reference itself cannot travel to the GPU box) on all host cores, rank 0 only.
`--dump-outputs DIR` (b200 arm, rank 0) writes what the last timed step computed as DIR/<name>.npy (see dump_outputs), so
that two builds run with the same arguments -- hence the same seeded inputs and weights -- can be compared output for output.
"""
import argparse
import json
import os
import statistics
import subprocess
import sys
import tempfile
import time
import zlib

import torch

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

FULL_SHAPES = [(48, 160), (24, 80), (12, 40), (6, 20)]   # feature levels of a 1280x384 image
METRIC = "images/sec (1280x384, fwd+bwd)"


# ------------------------------------------------------------------------------------------------
# helpers
# ------------------------------------------------------------------------------------------------
def peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        d = json.load(open(p))
        return {"hbm_gbs": d["hbm_gbs"], "bf16_tflops": d["bf16_tflops"],
                "bf16_tflops_sustained": d.get("bf16_tflops_sustained", d["bf16_tflops"]), "source": "measured"}
    return {"hbm_gbs": 6650.0, "bf16_tflops": 1590.0, "bf16_tflops_sustained": 1400.0, "source": "fallback"}


class ClockSampler:
    """nvidia-smi sampler running DURING the timed region (B200_PROFILING.md, clocks line)."""
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,"
         "clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, index=0):
        self.index = index
        self.f = tempfile.NamedTemporaryFile("w+", suffix=".csv", delete=False)
        self.p = None

    def start(self):
        try:
            self.p = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits",
                                       "-lms", "100", "-i", str(self.index)], stdout=self.f, stderr=subprocess.DEVNULL)
        except Exception:
            self.p = None

    def stop(self):
        out = {"sm_mhz": None, "sm_max_mhz": None, "reasons": [], "samples": 0}
        if self.p is None:
            return out
        time.sleep(0.15)
        self.p.terminate()
        try:
            self.p.wait(timeout=5)
        except Exception:
            self.p.kill()
        self.f.flush()
        rows = [r.strip().split(", ") for r in open(self.f.name).read().strip().splitlines() if r.strip()]
        os.unlink(self.f.name)
        sm, mx, reasons = [], [], set()
        for r in rows:
            if len(r) < 9:
                continue
            try:
                sm.append(float(r[1])); mx.append(float(r[2]))
            except ValueError:
                continue
            for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), r[5:9]):
                if v.strip().lower().startswith("active"):
                    reasons.add(name)
        if sm:
            out.update(sm_mhz=statistics.median(sm), sm_max_mhz=max(mx), reasons=sorted(reasons), samples=len(sm))
        return out


DUMP_LIMIT_BYTES = 64 * 1024 * 1024


def sampled(t, k, name):
    """`t` itself if it has at most k elements, else k of its (flattened) elements at fixed positions: the first k of a
    permutation seeded by crc32(name), in ascending order.  The same name and shape always select the same elements."""
    if t.numel() <= k:
        return t
    g = torch.Generator().manual_seed(zlib.crc32(name.encode()))
    idx = torch.randperm(t.numel(), generator=g)[:k].sort().values
    return t.detach().reshape(-1)[idx.to(t.device)]


def dump_outputs(path, arrays):
    """Write every tensor of `arrays` (name -> tensor) as path/<name>.npy: float64 tensors as float64, all others as float32.
    Refuses to write more than DUMP_LIMIT_BYTES in all."""
    import numpy as np
    host = {n: t.detach().to("cpu", torch.float64 if t.dtype == torch.float64 else torch.float32) for n, t in arrays.items()}
    total = sum(t.numel() * t.element_size() for t in host.values())
    if total > DUMP_LIMIT_BYTES:
        raise RuntimeError(f"--dump-outputs: {total} bytes exceed the {DUMP_LIMIT_BYTES}-byte limit")
    os.makedirs(path, exist_ok=True)
    for n, t in host.items():
        np.save(os.path.join(path, n + ".npy"), t.numpy())


def dist_info():
    ws = int(os.environ.get("WORLD_SIZE", "1"))
    return int(os.environ.get("RANK", "0")), int(os.environ.get("LOCAL_RANK", "0")), ws


def make_msda_inputs(B, Lq, seed, realistic=True, device="cpu"):
    """SURVEY.md 8(d) config 2.  realistic=True: reference grid + pixel-scale offsets like the module's
    offset-bias initialisation (ops/modules/ms_deform_attn.py:108-114); False: uniform [0,1] (cache-worst case)."""
    g = torch.Generator().manual_seed(seed)
    shapes = torch.as_tensor(FULL_SHAPES, dtype=torch.long)
    lsi = torch.cat((shapes.new_zeros((1,)), shapes.prod(1).cumsum(0)[:-1]))
    S = int(shapes.prod(1).sum())
    value = torch.randn(B, S, 8, 32, generator=g)
    if realistic:
        ref = torch.rand(B, Lq, 1, 1, 1, 2, generator=g)
        if Lq == S:   # encoder: one query per pixel, reference point = its own pixel centre
            pts = []
            for (H, W) in FULL_SHAPES:
                ys, xs = torch.meshgrid((torch.arange(H) + 0.5) / H, (torch.arange(W) + 0.5) / W, indexing="ij")
                pts.append(torch.stack((xs.reshape(-1), ys.reshape(-1)), -1))
            ref = torch.cat(pts, 0).view(1, S, 1, 1, 1, 2).expand(B, -1, -1, -1, -1, -1)
        wh = torch.as_tensor([(w, h) for h, w in FULL_SHAPES], dtype=torch.float32).view(1, 1, 1, 4, 1, 2)
        off = torch.randn(B, Lq, 8, 4, 4, 2, generator=g) * 2.0          # a couple of pixels at every level
        loc = (ref + off / wh).contiguous()
    else:
        loc = torch.rand(B, Lq, 8, 4, 4, 2, generator=g)
    attn = torch.softmax(torch.randn(B, Lq, 8, 16, generator=g), -1).view(B, Lq, 8, 4, 4)
    grad_out = torch.randn(B, Lq, 256, generator=g)
    ts = [value, shapes, lsi, loc, attn, grad_out]
    return [t.to(device) for t in ts]


def msda_bytes(B, Lq, S=10200, M=8, D=32, L=4, P=4):
    """Algorithmic bytes per launch (SURVEY.md 8d): forward reads value+loc+attn, writes out."""
    fwd = B * (S * M * D * 4 + Lq * M * L * P * 3 * 4 + Lq * M * D * 4)
    bwd = B * (2 * S * M * D * 4 + Lq * M * L * P * 3 * 4 * 2 + Lq * M * D * 4)
    return fwd, bwd


# ------------------------------------------------------------------------------------------------
# workload: msda (ours)
# ------------------------------------------------------------------------------------------------
def run_msda_b200(args, rank, local_rank, ws):
    import torch.distributed as dist
    from monodetr_b200 import _lib
    from monodetr_b200.msda import ms_deform_attn_backward, ms_deform_attn_forward
    dev = torch.device("cuda", local_rank)
    torch.cuda.set_device(dev)
    B, Lq = args.batch or 8, args.lq
    host = make_msda_inputs(B, Lq, seed=rank, realistic=not args.uniform_loc)
    pinned = [t.pin_memory() for t in host]
    dv = [t.to(dev) for t in host]
    flush = torch.empty(256 * 1024 * 1024 // 4, device=dev)
    fwd_bytes, bwd_bytes = msda_bytes(B, Lq)

    def step_device():
        out = ms_deform_attn_forward(*dv[:5], 64)
        gv, gl, ga = ms_deform_attn_backward(*dv[:5], dv[5], 64)
        return out, gv, gl, ga

    def barrier():
        if ws > 1:
            dist.barrier()
        torch.cuda.synchronize()

    for _ in range(args.warmup):
        step_device()
    barrier()
    sampler = ClockSampler(local_rank) if rank == 0 else None
    if sampler:
        sampler.start()
    evs = [[torch.cuda.Event(enable_timing=True) for _ in range(3)] for _ in range(args.steps)]
    lc0 = _lib.launch_count()
    for i in range(args.steps):
        grads = None                 # released before the step allocates, as when the step discards them
        flush.zero_()
        evs[i][0].record()
        out = ms_deform_attn_forward(*dv[:5], 64)
        evs[i][1].record()
        grads = ms_deform_attn_backward(*dv[:5], dv[5], 64)
        evs[i][2].record()
    barrier()
    launches = _lib.launch_count() - lc0
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, {n: sampled(t, 1 << 21, n) for n, t in
                                         zip(("out", "grad_value", "grad_loc", "grad_attn"), (out,) + tuple(grads))})
    del grads
    clocks = sampler.stop() if sampler else None
    t_fwd = [evs[i][0].elapsed_time(evs[i][1]) for i in range(args.steps)]
    t_bwd = [evs[i][1].elapsed_time(evs[i][2]) for i in range(args.steps)]
    total_ms = sum(t_fwd) + sum(t_bwd)
    tt = torch.tensor([total_ms], device=dev, dtype=torch.float64)
    if ws > 1:
        dist.all_reduce(tt, op=dist.ReduceOp.MAX)
    total_ms = float(tt.item())

    # end-to-end through the public op API with HOST buffers: H2D of the step's inputs + D2H of its results
    stage = [torch.empty_like(t, device=dev) for t in host]
    res_host = [torch.empty(B, Lq, 256).pin_memory(), torch.empty_like(host[3]).pin_memory(),
                torch.empty_like(host[4]).pin_memory()]
    def step_e2e():
        for s, p in zip(stage, pinned):
            s.copy_(p, non_blocking=True)
        out = ms_deform_attn_forward(*stage[:5], 64)
        gv, gl, ga = ms_deform_attn_backward(*stage[:5], stage[5], 64)
        res_host[0].copy_(out, non_blocking=True)
        res_host[1].copy_(gl, non_blocking=True)
        res_host[2].copy_(ga, non_blocking=True)
        return gv
    step_e2e()
    barrier()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(args.steps):
        step_e2e()
    e1.record()
    barrier()
    te = torch.tensor([e0.elapsed_time(e1)], device=dev, dtype=torch.float64)
    if ws > 1:
        dist.all_reduce(te, op=dist.ReduceOp.MAX)
    e2e_ms = float(te.item())
    h2d = sum(t.numel() * t.element_size() for t in host)
    d2h = sum(t.numel() * t.element_size() for t in res_host)

    if rank != 0:
        return None
    pk = peaks()
    fwd_ms = statistics.mean(t_fwd)
    ach = fwd_bytes / (fwd_ms * 1e-3) / 1e9
    line = {
        "metric": METRIC, "value": B * ws * args.steps / (total_ms * 1e-3), "unit": "images/sec",
        "n_gpus": ws, "steps": args.steps, "warmup": args.warmup, "ms_per_step": total_ms / args.steps,
        "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": {"workload": f"msda core fwd+bwd, B={B}/GPU, Lq={Lq}, 4 levels (1280x384), 8 heads x 32, 4 points, "
                               f"loc={'uniform' if args.uniform_loc else 'ref+N(0,2px)'}",
                   "timing": "CUDA events per step; 256 MiB L2 flush (untimed) between steps"},
        "e2e": {"value": B * ws * args.steps / (e2e_ms * 1e-3), "unit": "images/sec",
                "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": d2h},
        "gpu_launches": launches,
        "clocks": clocks,
        "roofline": {"kernel": "msda_fwd_d32_kernel", "bound": "hbm", "achieved": ach, "peak": pk["hbm_gbs"],
                     "unit": "GB/s", "frac": ach / pk["hbm_gbs"], "traffic": None, "peak_source": pk["source"],
                     "algorithmic_bytes": fwd_bytes, "avg_ms": fwd_ms},
        "roofline_bwd": {"kernel": "msda_bwd_vec_kernel<8,4>(+memset)", "bound": "hbm",
                         "achieved": bwd_bytes / (statistics.mean(t_bwd) * 1e-3) / 1e9, "peak": pk["hbm_gbs"],
                         "unit": "GB/s", "frac": bwd_bytes / (statistics.mean(t_bwd) * 1e-3) / 1e9 / pk["hbm_gbs"],
                         "algorithmic_bytes": bwd_bytes, "avg_ms": statistics.mean(t_bwd)},
    }
    if ws == 1:
        line["cpu_baseline"] = cpu_baseline_msda(Lq, budget_s=12.0)
        line["reference_cuda_kernel"] = time_reference_cuda_kernels(dv, flush, args.steps)
    return line


def time_reference_cuda_kernels(dv, flush, steps):
    """The reference's own SIMT kernels recompiled for sm_100a (oracle/_ref), same inputs: the kernel to beat."""
    from oracle import ref_gpu
    if not ref_gpu.available():
        return None
    for _ in range(2):
        ref_gpu.forward(*dv[:5]); ref_gpu.backward(*dv)
    torch.cuda.synchronize()
    tf, tb = [], []
    for _ in range(steps):
        flush.zero_()
        e = [torch.cuda.Event(enable_timing=True) for _ in range(3)]
        e[0].record(); ref_gpu.forward(*dv[:5]); e[1].record(); ref_gpu.backward(*dv); e[2].record()
        torch.cuda.synchronize()
        tf.append(e[0].elapsed_time(e[1])); tb.append(e[1].elapsed_time(e[2]))
    return {"fwd_ms": statistics.mean(tf), "bwd_ms": statistics.mean(tb), "note": "not a CPU line"}


def cpu_baseline_msda(Lq, budget_s=12.0, threads=None):
    """Reference CPU path of the op (oracle port of ms_deform_attn_core_pytorch) on a bounded sample."""
    from oracle.msda_torch import msda_core_torch
    threads = threads or os.cpu_count()
    torch.set_num_threads(threads)
    Bs = 2 if Lq > 1000 else 8
    value, shapes, lsi, loc, attn, grad_out = make_msda_inputs(Bs, Lq, seed=0)

    def one_pass():
        v, lo, a = (t.clone().requires_grad_(True) for t in (value, loc, attn))
        out = msda_core_torch(v, shapes, lo, a)
        torch.autograd.grad(out, (v, lo, a), grad_out)

    one_pass()                      # warm-up
    n, t0 = 0, time.time()
    while n < 1 or (time.time() - t0 < budget_s and n < 20):
        one_pass()
        n += 1
    dt = time.time() - t0
    return {"value": Bs * n / dt, "unit": "images/sec", "cores": threads, "kind": "port",
            "sample": f"msda core fwd+bwd (grid_sample port of ms_deform_attn_core_pytorch), B={Bs}, Lq={Lq}, {n} passes"}


def cpu_baseline_model():
    """CPU port of the reference model path (oracle/monodetr_torch.py), train shapes, fwd+bwd, bounded sample."""
    from oracle import monodetr_torch as om

    class A:
        steps, warmup, cpu_batch = 1, 0, 1
    val, dt, sample, threads, cfg = om.bench_reference_model(A)
    return {"value": val, "unit": "images/sec", "cores": threads, "kind": "port", "sample": sample + f", {A.steps} timed steps"}


# ------------------------------------------------------------------------------------------------
# reference arm (CPU)
# ------------------------------------------------------------------------------------------------
def run_reference(args, rank, ws):
    if rank != 0:
        return None
    if args.workload == "msda":
        from oracle.msda_torch import msda_core_torch
        threads = os.cpu_count()
        torch.set_num_threads(threads)
        Bs = 2
        value, shapes, lsi, loc, attn, grad_out = make_msda_inputs(Bs, args.lq, seed=0, realistic=not args.uniform_loc)
        def step():
            v, lo, a = (t.clone().requires_grad_(True) for t in (value, loc, attn))
            out = msda_core_torch(v, shapes, lo, a)
            torch.autograd.grad(out, (v, lo, a), grad_out)
        for _ in range(min(args.warmup, 2)):
            step()
        t0 = time.time()
        for _ in range(args.steps):
            step()
        dt = time.time() - t0
        val = Bs * args.steps / dt
        sample = f"B={Bs} per step (bounded sample of the B=8 workload), Lq={args.lq}"
        cfg = {"workload": f"msda core fwd+bwd, Lq={args.lq}, reference CPU path (grid_sample) port"}
    else:
        from oracle import monodetr_torch as om
        args.cpu_batch = 1
        val, dt, sample, threads, cfg = om.bench_reference_model(args)
    return {"impl": "reference", "metric": METRIC, "value": val, "unit": "images/sec", "n_gpus": ws,
            "steps": args.steps, "warmup": args.warmup, "ms_per_step": dt / args.steps * 1e3,
            "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "config": cfg,
            "cpu_baseline": {"value": val, "unit": "images/sec", "cores": threads, "kind": "port", "sample": sample},
            "e2e": {"value": val, "unit": "images/sec", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--workload", default=os.environ.get("MDB_BENCH_WORKLOAD", "model"), choices=["model", "msda", "infer"])
    ap.add_argument("--batch", type=int, default=0, help="per-GPU batch (default: 8 at N=1, 16 at N>1 for model)")
    ap.add_argument("--lq", type=int, default=10200)
    ap.add_argument("--uniform-loc", action="store_true")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="b200 arm: write the results of the last timed step as DIR/<name>.npy (float32/float64, <= 64 MiB; "
                         "arrays above a size cap as a fixed seeded sample)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "b200":
        ap.error("--dump-outputs needs --impl b200")
    args.warmup = max(args.warmup, 3) if args.impl == "b200" else args.warmup
    rank, local_rank, ws = dist_info()

    if args.impl == "reference":
        line = run_reference(args, rank, ws)
        if line is not None:
            print(json.dumps(line), flush=True)
        return

    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device (the hot path has no CPU fallback)")
    if ws > 1:
        import torch.distributed as dist
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        torch.cuda.set_device(local_rank)
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))
    if args.workload == "msda":
        line = run_msda_b200(args, rank, local_rank, ws)
    else:
        from monodetr_b200 import bench_model
        quick = bool(os.environ.get("MDB_BENCH_QUICK"))      # A/B runs: the timed step and e2e only (no probes, batch-16 point, CPU arm, extras)
        line = bench_model.run(args, rank, local_rank, ws, infer=(args.workload == "infer"), extras=not quick,
                               dump_dir=args.dump_outputs)
        if line is not None and ws == 1 and args.workload == "model" and not quick:
            if not args.batch and not os.environ.get("MDB_BENCH_NO_B16"):
                # the N > 1 runs use batch 16 per GPU (BASELINE configs[3]): the like-for-like single-GPU point for scaling
                import gc
                gc.collect(); torch.cuda.empty_cache()
                b16 = bench_model.run(args, rank, local_rank, ws, batch_override=16, extras=False)
                line["batch16"] = {"value": b16["value"], "unit": "images/sec", "ms_per_step": b16["ms_per_step"],
                                   "e2e": b16["e2e"]["value"], "note": "same step at batch 16/GPU (the per-GPU batch of the N>1 runs): "
                                   "use this value, not `value`, as the 1-GPU point of a like-for-like scaling efficiency"}
            line["cpu_baseline"] = cpu_baseline_model()
            if not args.batch and not os.environ.get("MDB_BENCH_NO_EXTRAS"):
                # SURVEY.md 8(f): criterion / post-process / pre-process beside their CPU restatements, and the complete
                # training iteration (forward + criterion + backward + AdamW) in one CUDA graph.  Extras, never the headline.
                import gc
                import bench_extras
                gc.collect(); torch.cuda.empty_cache()
                dev = torch.device("cuda", local_rank)
                try:
                    line["next_rows"] = bench_extras.next_rows_probe(dev)
                    flush = torch.empty(256 * 1024 * 1024 // 4, device=dev)
                    line["full_training_iteration"] = bench_extras.full_train_step_probe(dev, 8, args.steps, flush)
                except Exception as e:
                    line["extras_error"] = f"{type(e).__name__}: {e}"
    if line is not None:
        print(json.dumps(line), flush=True)
    if ws > 1:
        import torch.distributed as dist
        dist.barrier()
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
