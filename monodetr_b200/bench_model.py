"""bench.py --workload model: full MonoDETR forward+backward (train mode: 550 queries, group self-attention, dropout
0.1), ResNet-50, 1280x384 synthetic images, surrogate loss sum_k mean(out_k^2) (SURVEY.md 8d), one flat-bucket NCCL
all-reduce of the gradients per step when world_size > 1.  The step is captured once in a CUDA graph (fwd + loss +
bwd; the all-reduce is launched right after the replay on the same stream) so the timed region is GPU-bound.
"""
import json
import os
import statistics
import time

import torch
import torch.distributed as dist

from . import _lib, kernels as K, tc
from . import build_monodetr
from .ddp import FlatGradBucket, broadcast_parameters
from .monodetr import DEFAULT_MODEL_CFG

METRIC = "images/sec (1280x384, fwd+bwd)"
TRAIN_FLOPS_PER_IMAGE = 363.5e9          # matmul+conv fwd+bwd, SURVEY.md 8d
FULL_S = 10200


def surrogate_loss(out):
    """sum_k mean(out_k^2) over every head output incl. the aux levels (SURVEY.md 8d), as one fused launch."""
    from . import functional as Fn
    ts = []
    for k, v in out.items():
        if k == "aux_outputs":
            for aux in v:
                ts.extend(aux.values())
        else:
            ts.append(v)
    return Fn.sum_mean_squares(ts)


def synthetic_batch(B, seed):
    g = torch.Generator().manual_seed(seed)
    images = torch.randn(B, 3, 384, 1280, generator=g)
    calibs = torch.zeros(B, 3, 4)
    calibs[:, 0, 0] = calibs[:, 1, 1] = 721.5377
    calibs[:, 0, 2] = 609.5593; calibs[:, 1, 2] = 172.854; calibs[:, 0, 3] = 44.85728
    sizes = torch.tensor([[1242., 375.]]).repeat(B, 1)
    return images, calibs, sizes


class MsdaProbe:
    """CUDA-event timing of the MSDeformAttn forward launches (events recorded immediately around the C call inside
    monodetr_b200.msda, eager steps only)."""

    def __enter__(self):
        from . import msda as _m
        self._m = _m
        self.events = []
        _m.PROBE = self.events
        return self

    def __exit__(self, *a):
        self._m.PROBE = None

    def encoder_ms(self):
        ts = [e0.elapsed_time(e1) for e0, e1, _, lq in self.events if lq == FULL_S]
        return statistics.mean(ts) if ts else None


def gemm_probe(dev, flush):
    """`roofline_gemm`: the dominant kernel family (tc_conv_gemm_kernel: ~50 % of the step) timed alone with CUDA events on
    the three shapes that carry most of its FLOPs at batch 8 -- a ResNet 3x3 convolution (layer3), the encoder-sized linear
    (M = 81 600, N = K = 256: value_proj / output_proj / FFN of the three encoder layers) forward, and that linear's weight
    gradient.  Useful FLOPs (2 M N K, one product per MAC although the bf16x3 arithmetic issues three) / launch time."""
    g = torch.Generator(device=dev).manual_seed(0)
    out = []
    x = torch.randn(8, 24, 80, 256, device=dev, generator=g)
    w = torch.randn(256, 256, 3, 3, device=dev, generator=g) / 48.0
    xl = torch.randn(81600, 256, device=dev, generator=g)
    wl = torch.randn(256, 256, device=dev, generator=g) / 16.0
    dyl = torch.randn(81600, 256, device=dev, generator=g)
    sw = tc.split_weights([w])[0] if tc.get_precision() == "bf16x3" else tc.pack_weight(w)
    swl = tc.split_weights([wl])[0] if tc.get_precision() == "bf16x3" else wl
    cases = [("conv3x3 256->256 @ 8x24x80 fwd", 2.0 * 8 * 24 * 80 * 256 * 256 * 9, lambda: tc.conv2d_forward(x, sw, None, None, 3, 3, 1, 1)),
             ("linear 81600x256x256 fwd", 2.0 * 81600 * 256 * 256, lambda: tc.linear_forward(xl, swl)),
             ("linear 81600x256x256 wgrad", 2.0 * 81600 * 256 * 256, lambda: tc.linear_wgrad(dyl, xl))]
    for name, flops, fn in cases:
        for _ in range(3):
            fn()
        ts = []
        for _ in range(5):
            flush.zero_()
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record(); fn(); e1.record()
            torch.cuda.synchronize()
            ts.append(e0.elapsed_time(e1))
        ms = statistics.mean(ts)
        out.append({"shape": name, "avg_ms": ms, "tflops": flops / (ms * 1e-3) / 1e12})
    return out


def run(args, rank, local_rank, ws, infer=False, batch_override=None, extras=True, dump_dir=None):
    """infer=False: BASELINE configs[2]/[3] (train step).  infer=True: configs[4], eval-mode forward only, batch 32,
    no gradients, N>1 = independent replicas (no collective).  dump_dir: rank 0 writes the last timed step's results there
    (bench.dump_outputs): the surrogate loss, every output head, and (train) every parameter gradient."""
    dev = torch.device("cuda", local_rank)
    torch.cuda.set_device(dev)
    B = batch_override or args.batch or (32 if infer else (8 if ws == 1 else 16))
    precision = os.environ.get("MDB_PRECISION", "bf16x3")
    tc.set_precision(precision)
    torch.manual_seed(0)
    model, _ = build_monodetr(DEFAULT_MODEL_CFG)
    model = model.to(dev)
    model = model.eval() if infer else model.train()
    broadcast_parameters(model)
    bucket = None if infer else FlatGradBucket(model)

    host = [t.pin_memory() for t in synthetic_batch(B, seed=1000 + rank)]
    images, calibs, sizes = (t.to(dev) for t in host)
    loss_buf = torch.zeros((), device=dev)
    loss_host = torch.zeros(()).pin_memory()

    last = {}      # the latest call's outputs; in graph mode the captured tensors, which every replay rewrites

    def fwd_bwd():
        last.clear()
        if infer:
            with torch.no_grad():
                out = model(images, calibs, None, sizes)
                loss_buf.copy_(surrogate_loss(out))          # checksum over every output head = the step's result
            last["out"] = out
            return
        bucket.zero()
        out = model(images, calibs, None, sizes)
        loss = surrogate_loss(out)
        loss.backward()
        loss_buf.copy_(loss.detach())
        last["out"] = out

    def barrier():
        if ws > 1:
            dist.barrier()
        torch.cuda.synchronize()

    # ---- warm-up (eager) then capture --------------------------------------------------------------------
    side = torch.cuda.Stream()
    side.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(side):
        for _ in range(2):
            fwd_bwd()
    torch.cuda.current_stream().wait_stream(side)
    torch.cuda.synchronize()
    lc0 = _lib.launch_count()
    graph = None
    use_graph = os.environ.get("MDB_NO_GRAPH", "0") != "1"
    if use_graph:
        try:
            graph = torch.cuda.CUDAGraph()
            with torch.cuda.graph(graph):
                fwd_bwd()
            if bucket is not None:
                bucket.freeze_sources()
        except Exception as e:          # capture is an optimisation of launch overhead only: same kernels either way
            if rank == 0:
                print(f"[bench_model] CUDA graph capture failed ({type(e).__name__}: {e}); running eager", flush=True)
            graph = None
            torch.cuda.synchronize()
            lc0 = _lib.launch_count()
            fwd_bwd()
    else:
        fwd_bwd()
    launches_per_step = _lib.launch_count() - lc0

    def step():
        if graph is not None:
            graph.replay()
        else:
            fwd_bwd()
        if bucket is not None:
            bucket.all_reduce()

    for _ in range(max(args.warmup, 3)):
        step()
    barrier()

    from bench import ClockSampler, peaks, msda_bytes          # bench.py is the entry script (already imported)
    sampler = ClockSampler(local_rank) if rank == 0 else None
    if sampler:
        sampler.start()
    flush = torch.empty(256 * 1024 * 1024 // 4, device=dev)
    evs = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(args.steps)]
    for i in range(args.steps):
        flush.zero_()
        evs[i][0].record()
        step()
        evs[i][1].record()
    barrier()
    clocks = sampler.stop() if sampler else None
    total_ms = sum(a.elapsed_time(b) for a, b in evs)
    tt = torch.tensor([total_ms], device=dev, dtype=torch.float64)
    if ws > 1:
        dist.all_reduce(tt, op=dist.ReduceOp.MAX)
    total_ms = float(tt.item())
    if dump_dir is not None and rank == 0:
        from bench import dump_outputs, sampled
        arrays = {"loss": loss_buf}
        for k, v in last["out"].items():
            for name, t in ([(f"out.aux{i}.{kk}", vv) for i, aux in enumerate(v) for kk, vv in aux.items()] if k == "aux_outputs"
                            else [(f"out.{k}", v)]):
                arrays[name] = sampled(t, 1 << 21, name)
        for n, p in model.named_parameters():
            if p.grad is not None:
                arrays[f"grad.{n}"] = sampled(p.grad, 1 << 14, f"grad.{n}")
        dump_outputs(dump_dir, arrays)

    # ---- exposed all-reduce (N > 1): the flat-bucket pack + ncclAllReduce + divide run after the graph replay, not overlapped
    allreduce_ms = None
    if bucket is not None and ws > 1:
        barrier()
        a0, a1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a0.record()
        for _ in range(args.steps):
            bucket.all_reduce()
        a1.record()
        barrier()
        ta = torch.tensor([a0.elapsed_time(a1) / args.steps], device=dev, dtype=torch.float64)
        dist.all_reduce(ta, op=dist.ReduceOp.MAX)
        allreduce_ms = float(ta.item())

    # ---- end to end through the public API with HOST inputs: H2D of the batch + D2H of the loss every step ------
    # Input feeding is double-buffered the way a data loader would do it: a copy stream moves batch i+1 from pinned host
    # memory into a staging buffer while step i runs; the step's own stream waits for the copy, takes the batch with a
    # device-to-device copy, and hands the staging buffer back.  All K host->device copies are inside the timed region
    # (the first one is not hidden by anything).
    copy_stream = torch.cuda.Stream()
    stage = [torch.empty_like(t) for t in (images, calibs, sizes)]

    def prefetch(after=None):
        with torch.cuda.stream(copy_stream):
            if after is not None:
                copy_stream.wait_event(after)            # the staging buffer has been consumed
            for d, h in zip(stage, host):
                d.copy_(h, non_blocking=True)
            ev = torch.cuda.Event()
            ev.record(copy_stream)
        return ev

    def run_e2e(n):
        main = torch.cuda.current_stream()
        ev = prefetch()
        for i in range(n):
            main.wait_event(ev)
            images.copy_(stage[0]); calibs.copy_(stage[1]); sizes.copy_(stage[2])
            consumed = torch.cuda.Event()
            consumed.record(main)
            if i + 1 < n:
                ev = prefetch(consumed)
            step()
            loss_host.copy_(loss_buf, non_blocking=True)

    run_e2e(2)
    barrier()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    run_e2e(args.steps)
    e1.record()
    barrier()
    te = torch.tensor([e0.elapsed_time(e1)], device=dev, dtype=torch.float64)
    if ws > 1:
        dist.all_reduce(te, op=dist.ReduceOp.MAX)
    e2e_ms = float(te.item())
    h2d = sum(t.numel() * t.element_size() for t in host)

    # ---- MSDA kernel duration in situ (eager steps, events around the launches; real sampling locations) --------
    enc_ms = None
    if extras:
        with MsdaProbe() as probe:
            for _ in range(3):
                fwd_bwd()
            torch.cuda.synchronize()
            enc_ms = probe.encoder_ms()
    loss_val = float(loss_buf.item())
    gemm = gemm_probe(dev, flush) if (extras and rank == 0 and not infer) else None

    if rank != 0:
        return None
    pk = peaks()
    fwd_bytes, _ = msda_bytes(B, FULL_S)
    ms_step = total_ms / args.steps
    flops_img = TRAIN_FLOPS_PER_IMAGE / 3 if infer else TRAIN_FLOPS_PER_IMAGE
    line = {
        "metric": "images/sec (1280x384, fwd only)" if infer else METRIC, "value": B * ws * args.steps / (total_ms * 1e-3), "unit": "images/sec", "n_gpus": ws,
        "steps": args.steps, "warmup": max(args.warmup, 3), "ms_per_step": ms_step, "higher_is_better": True,
        "scaling": "weak", "vs_baseline": None, "dtype": {"tf32x3": "f32 (3xTF32)", "bf16x3": "f32 (BF16x3: error-compensated bf16 tensor-core products, fp32 accumulate)", "tf32": "tf32"}[precision],
        "data": "synthetic",
        "config": {"workload": (f"MonoDETR inference forward, ResNet-50, batch {B}/GPU, 1280x384 synthetic, eval mode (50 queries), "
                                f"{'independent replicas, ' if ws > 1 else ''}fp32 storage, tensor-core math = " if infer else
                                f"full MonoDETR fwd+bwd, ResNet-50, batch {B}/GPU, 1280x384 synthetic, train mode (550 queries, dropout 0.1), "
                                f"surrogate loss, {'flat-bucket NCCL all-reduce, ' if ws > 1 else ''}fp32 storage, tensor-core math = ")
                               + {"tf32x3": "error-compensated 3xTF32 (fp32-equivalent)", "tf32": "single-pass TF32",
                                  "bf16x3": "error-compensated BF16x3 (hi/lo split operands, fp32 accumulate) for forward, data-gradient and weight-gradient GEMMs and attention"}[precision],
                   "parallelism": f"dp{ws}", "global_batch": B * ws,
                   "timing": "CUDA events per step; 256 MiB L2 flush (untimed) between steps; " + ("CUDA graph replay" if graph is not None else "eager launches")
                             + "; e2e: batch double-buffered from pinned host memory on a copy stream, every step's H2D + loss D2H inside the timed "
                               "region, NO L2 flush between its steps (which is why e2e can exceed `value` by the cold-L2 penalty of a step)"},
        "e2e": {"value": B * ws * args.steps / (e2e_ms * 1e-3), "unit": "images/sec", "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": 4},
        "gpu_launches": launches_per_step * args.steps,
        "clocks": clocks,
        "loss": loss_val,
        "model_tflops": flops_img * B / (ms_step * 1e-3) / 1e12,
        "tensor_frac_of_measured_bf16_peak": flops_img * B / (ms_step * 1e-3) / 1e12 / pk["bf16_tflops_sustained"],
    }
    if allreduce_ms is not None:
        line["allreduce_ms_exposed"] = allreduce_ms
    if gemm:
        best = max(gemm, key=lambda c: c["tflops"])
        line["roofline_gemm"] = {"kernel": "tc_conv_gemm_kernel (tcgen05 BF16x3 implicit GEMM; " + best["shape"] + ")", "bound": "tensor",
                                 "achieved": best["tflops"], "peak": pk["bf16_tflops"], "unit": "TFLOP/s", "frac": best["tflops"] / pk["bf16_tflops"],
                                 "traffic": None, "peak_source": pk["source"] + " (burst: kernel timed alone)",
                                 "note": "useful FLOPs; the error-compensated arithmetic issues 3 tensor-core products per MAC, so 1/3 is the ceiling of this ratio",
                                 "shapes": gemm}
    if enc_ms:
        ach = fwd_bytes / (enc_ms * 1e-3) / 1e9
        line["roofline"] = {"kernel": "msda_fwd_d32_kernel<fused pre-processing> (encoder call, Lq=10200, in situ)", "bound": "hbm", "achieved": ach,
                            "peak": pk["hbm_gbs"], "unit": "GB/s", "frac": ach / pk["hbm_gbs"],
                            # dram__bytes_read.sum + dram__bytes_write.sum of this launch at B=8 from the committed ncu --set full
                            # capture of the fused kernel inside the step, profiles/r02_msda_fused_fwd_step_ncu.txt
                            # (242.4 MB + 73.2 MB); scaled with the batch
                            "traffic": int(315.52e6 * B / 8),
                            "peak_source": pk["source"], "algorithmic_bytes": fwd_bytes, "avg_ms": enc_ms}
    return line
