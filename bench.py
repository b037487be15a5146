#!/usr/bin/env python
"""bench.py -- N-pair fwd+bwd samples/sec (BASELINE.json metric: B=8192, D=512 on 1/2/4/8 B200).

  python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--config HL|C2|C3|C4|C5]
                  [--precision fp16x2|bf16x3|bf16] [--mining config|usage|rand|relative] [--dump-outputs DIR]

One "step" = Forward_gpu + Backward_gpu of the NPairMultiClassLoss layer (reference npair_multi_class_loss.cu:207-402, :420-499)
over one batch of synthetic L2-normalised embeddings (B/2 classes x 2 images, SURVEY 8d seeds), the global batch sharded by anchor
over the N ranks (strong scaling: Q = B/N rows per rank against all B columns).  --config picks one of BASELINE.json's named
configurations (HL = the headline metric, usage-block mining of usage/def.prototxt:137-146).

  value    : whole-job samples/sec with the inputs resident in HBM, through the C ABI (npair_forward_backward: both passes enqueued,
             one wait for the five host scalars; includes the feature exchange and the row-record exchange), CUDA-event timed, max
             over ranks.  step_call_other: the same through npair_forward + npair_backward (--two-call makes that the headline).
  e2e      : the same metric through the reference-facing plugin surface (the Caffe-style layer in npairloss_b200/caffe_shim)
             with HOST bottoms: every timed step copies that step's batch host->device from pinned memory (on a copy stream,
             double-buffered like Caffe's prefetching data layers) and reads the five tops device->host.  e2e_serial is the same
             without overlap (copy, then compute); e2e_serial_grad_d2h additionally copies the gradient back every step.
  roofline : the dominant kernel, live CUDA-event duration from a profiled pass, algorithmic flops of SURVEY 8d.
  cpu_baseline : the oracle (a "port": the reference has no CPU path and cannot be compiled here) on a bounded sample.
  parity_check (N > 1): the NCCL path against an emulation of all ranks on rank 0's GPU through the external-collectives ABI
             (bitwise), and against the CPU oracle on a small sharded shape.

--impl reference times the CPU oracle (faithful sorts, one thread per physical core, pinned) on the same config; rank 0 only.
"""
from __future__ import annotations

import os

# The CPU arm's OpenMP threads stay on their cores (set before anything loads libgomp).  ONLY in a single-process run: with
# OMP_PROC_BIND set libgomp also binds the INITIAL thread to the first place, so under torchrun every rank's main thread landed on
# core 0 and the eight busy-polling ranks took turns on it -- 32.5 ms per step at N = 8 whatever the configuration (round 2, first
# 8-GPU run; profiles/r02_experiments.md).  Sharded runs never set it; their reference arm (rank 0 only) runs unpinned.
if int(os.environ.get("WORLD_SIZE", "1")) == 1:
    os.environ.setdefault("OMP_PROC_BIND", "close")
    os.environ.setdefault("OMP_PLACES", "cores")

import argparse  # noqa: E402
import ctypes as C  # noqa: E402
import json  # noqa: E402
import subprocess  # noqa: E402
import sys  # noqa: E402
import threading  # noqa: E402
import time  # noqa: E402

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)
sys.dont_write_bytecode = True          # the benchmark leaves the source tree as it found it (it may be read-only)

import numpy as np  # noqa: E402

PRECS = {"bf16x3": 0, "bf16": 1, "fp16x2": 2}
MMA_PASSES = {"bf16x3": 6, "bf16": 1, "fp16x2": 3}
DTYPE_DESC = {"fp16x2": "f32 (3-pass fp16-split tcgen05, f32 accumulate)", "bf16x3": "f32 (6-pass bf16-split tcgen05, f32 accumulate)",
              "bf16": "bf16 (f32 accumulate)"}


def load_peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        d = json.load(open(p))
        return dict(hbm_gbs=d["hbm_gbs"], tf_burst=d["bf16_tflops"], tf_sustained=d.get("bf16_tflops_sustained", d["bf16_tflops"]),
                    sm_max_mhz=d.get("sm_max_mhz"), source="measured (MEASURED_PEAKS.json)")
    return dict(hbm_gbs=6650.0, tf_burst=1590.0, tf_sustained=1400.0, sm_max_mhz=1965.0, source="fallback (B200_PROFILING.md)")


class ClockSampler:
    """nvidia-smi clocks / throttle reasons DURING the timed region (B200_PROFILING.md recipe)."""
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index=0):
        self.rows, self.proc, self.gpu = [], None, gpu_index

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits", "-lms", "25",
                                          "-i", str(self.gpu)], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.t = threading.Thread(target=self._read, daemon=True)
            self.t.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append(line.strip())

    def stop(self):
        if not self.proc:
            return dict(sm_mhz=None, sm_max_mhz=None, reasons=["nvidia-smi unavailable"])
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except Exception:
            pass
        sm, mx, reasons = [], [], set()
        for r in self.rows:
            f = [x.strip() for x in r.split(",")]
            if len(f) < 9:
                continue
            try:
                sm.append(float(f[1])); mx.append(float(f[2]))
            except ValueError:
                continue
            for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), f[5:9]):
                if v.lower().startswith("active"):
                    reasons.add(name)
        if not sm:
            return dict(sm_mhz=None, sm_max_mhz=None, reasons=["no samples"])
        return dict(sm_mhz=float(np.median(sm)), sm_max_mhz=float(max(mx)), reasons=sorted(reasons), samples=len(sm))


def host_threads():
    """Threads for the CPU oracle: one per physical core (the sort-heavy oracle loses 4x with SMT oversubscription:
    683 vs 2690 samples/s on the 128-thread gpurun box).  torchrun exports OMP_NUM_THREADS=1, so never rely on the default."""
    n = os.cpu_count() or 1
    return max(1, n // 2) if n >= 32 else n


def resolve_workload(args):
    """(name, B, D, mining, mining_desc, noise, seed, precision) of the run."""
    from npairloss_b200 import synth
    c = synth.CONFIGS[args.config]
    B = args.batch or c["B"]
    D = args.dim or c["D"]
    mining, desc = dict(c["mining"]), None
    if args.mining == "usage":
        mining = dict(synth.USAGE_MINING)
    elif args.mining == "rand":
        mining = dict(synth.DEFAULT_MINING)
    elif args.mining == "relative":
        mining = dict(synth.USAGE_MINING, ap_region=synth.LOCAL, ap_method=synth.RELATIVE_HARD, an_region=synth.LOCAL,
                      an_method=synth.RELATIVE_HARD, identsn=-0.3, diffsn=-0.3, margin_diff=0.0)
    reg, met = {0: "GLOBAL", 1: "LOCAL"}, {0: "HARD", 1: "EASY", 2: "RAND", 3: "RELATIVE_HARD", 4: "RELATIVE_EASY"}
    desc = (f"AP {reg[mining['ap_region']]} {met[mining['ap_method']]} (identsn {mining['identsn']}, margin_ident {mining['margin_ident']}), "
            f"AN {reg[mining['an_region']]} {met[mining['an_method']]} (diffsn {mining['diffsn']}, margin_diff {mining['margin_diff']})")
    if mining == synth.USAGE_MINING:
        desc = "usage-block mining of usage/def.prototxt:137-146: " + desc
    prec = args.precision or ("bf16" if args.config == "C3" else "fp16x2")
    return args.config, B, D, mining, desc, c["noise"], 20171225 + c["idx"], prec


def metric_name(B, D):
    return f"N-pair fwd+bwd samples/sec at B={B},D={D}"


def oracle_sample(B, D, mining, x, lab, world_s, threads):
    """The oracle state for the bounded CPU sample: rank 0's block of a world_s-way anchor sharding, faithful sorts, fp32 accumulate."""
    from oracle import oracle_lib as o
    Qs = B // world_s
    cfg = o.make_config(Qs, D, world=world_s, rank=0, accum_double=0, faithful_sorts=1, num_threads=threads, **mining)
    L = o.lib()
    buf = np.zeros(L.npo_state_floats(C.byref(cfg)), dtype=np.float32)
    st = o.NpoState()
    L.npo_state_bind(C.byref(cfg), o._fp(buf), C.byref(st))
    tops = np.zeros(5, np.float32)
    ld = np.zeros((Qs, D), np.float32)
    td = np.zeros((B, D), np.float32)

    def step():
        e = L.npo_forward(C.byref(cfg), o._fp(x), o._fp(lab), None, C.byref(st), o._fp(tops))
        e2 = L.npo_backward_partial(C.byref(cfg), o._fp(x), C.byref(st), C.c_float(1.0), o._fp(ld), o._fp(td))
        assert e == 0 and e2 == 0
    step.keep = (buf, ld, td, tops)
    return step, Qs


def cpu_sample_world(B):
    """The CPU sample is rank 0's block of this sharding (about 1024 anchors per step, whatever the batch)."""
    return max(1, B // 1024)


def run_reference(args, wl):
    """CPU baseline arm: the oracle with the reference's unconditional sorts on the host cores, on the SAME workload as the GPU arm
    (the k = 1 shape: B anchors x B database); --cpu-sample (and B > 16384) time rank 0's block of an anchor sharding with ~1024
    anchors instead."""
    from npairloss_b200 import synth
    name, B, D, mining, desc, noise, seed, prec = wl
    x, lab = synth.make_inputs(B, D, seed, noise=noise)
    cores = host_threads()
    # the true k = 1 shape whenever the oracle's five B x B fp32 arrays fit comfortably (HL: 1.3 GB, ~2 s per step on 64 cores);
    # C5 (B = 65536: 86 GB) is timed on the bounded sample
    world_s = cpu_sample_world(B) if (args.cpu_sample or B > 16384) and not args.cpu_full else 1
    step, Qs = oracle_sample(B, D, mining, x, lab, world_s, cores)
    for _ in range(args.warmup):
        step()
    times = []
    for _ in range(args.steps):
        t0 = time.perf_counter()
        step()
        times.append(time.perf_counter() - t0)
    dt = float(np.median(times))
    val = Qs / dt
    sample = (f"{'the full k=1 shape' if world_s == 1 else f'rank-0 block of a {world_s}-way anchor sharding'}: {Qs} anchors x {B} database x D={D}, "
              "faithful unconditional sorts, fp32 accumulate, OpenMP pinned (OMP_PROC_BIND=close), median of the timed steps")
    out = {"metric": metric_name(B, D), "impl": "reference", "value": val, "unit": "samples/s", "n_gpus": args.gpus, "steps": args.steps,
           "warmup": args.warmup, "ms_per_step": dt * 1e3, "higher_is_better": True, "scaling": "strong", "vs_baseline": None,
           "dtype": "f32", "data": "synthetic",
           "config": {"workload": f"{name}: B={B}, D={D}, {B // 2} classes x 2, {desc}, loss_weight 1", "global_batch": B, "feature_dim": D,
                      "noise": noise, "step_spread": {"min_ms": min(times) * 1e3, "max_ms": max(times) * 1e3}},
           "cpu_baseline": {"value": val, "unit": "samples/s", "cores": cores, "kind": "port", "sample": sample},
           "e2e": {"value": val, "unit": "samples/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
           "gpu_launches": 0}
    emit(out)


DUMP_BYTES = 64 << 20


def dump_outputs(path, tops, grad, world, rank):
    """Writes what the step call returned in the last timed step, as float32 .npy files under `path` (rank 0):
      tops.npy  (world, 5)  loss, top1, top5, top10, feature_asum of every rank
      dx.npy    (B, D)      the gradient of the whole batch, rank blocks in order
    When dx would exceed the size cap, a fixed, seeded sample of its rows is written instead, as dx_sample.npy, with the row
    indices in dx_sample_rows.npy (float64).  The inputs depend only on the arguments, so two builds run with the same
    arguments can be compared file by file."""
    import torch
    import torch.distributed as dist
    t = torch.tensor(tops, dtype=torch.float32, device=grad.device).reshape(1, 5)
    if world > 1:
        ts = [torch.empty_like(t) for _ in range(world)]
        gs = [torch.empty_like(grad) for _ in range(world)]
        dist.all_gather(ts, t)
        dist.all_gather(gs, grad)
        t, grad = torch.cat(ts), torch.cat(gs)
    if rank != 0:
        return
    os.makedirs(path, exist_ok=True)
    np.save(os.path.join(path, "tops.npy"), t.cpu().numpy())
    B, D = grad.shape
    cap = DUMP_BYTES - (1 << 20)                         # the rest is room for tops.npy and the .npy headers
    if B * D * 4 <= cap:
        np.save(os.path.join(path, "dx.npy"), grad.cpu().numpy())
        return
    rows = np.sort(np.random.default_rng(20171225).choice(B, size=cap // (4 * D + 8), replace=False))
    np.save(os.path.join(path, "dx_sample.npy"), grad[torch.from_numpy(rows).to(grad.device)].cpu().numpy())
    np.save(os.path.join(path, "dx_sample_rows.npy"), rows.astype(np.float64))


_REAL_STDOUT = None


def emit(obj):
    """The contract is ONE JSON line on stdout; libraries (NCCL's version banner, torchrun) also write to fd 1, so the
    process's stdout is pointed at stderr for the whole run and the result goes to the saved descriptor."""
    line = (json.dumps(obj) + "\n").encode()
    os.write(_REAL_STDOUT if _REAL_STDOUT is not None else 1, line)


def main():
    global _REAL_STDOUT
    sys.stdout.flush()
    _REAL_STDOUT = os.dup(1)
    os.dup2(2, 1)
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=50)
    ap.add_argument("--warmup", type=int, default=10)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--config", default="HL", choices=["HL", "C2", "C3", "C4", "C5"])
    ap.add_argument("--precision", default=None, choices=list(PRECS))
    ap.add_argument("--batch", type=int, default=0)
    ap.add_argument("--dim", type=int, default=0)
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--cpu-full", action="store_true", help="reference arm: time the true k = 1 shape even when it is huge")
    ap.add_argument("--cpu-sample", action="store_true", help="reference arm: time the bounded rank-0 block sample instead of the k = 1 shape")
    # SURVEY 8(d): "config" = the named configuration's own mining; rand (RAND/RAND, cheapest) and relative (LOCAL RELATIVE_HARD on
    # both sides, diffsn -0.3: a radix select per row and side, costliest) are the two other settings it asks to be reported
    ap.add_argument("--mining", default="config", choices=["config", "usage", "rand", "relative"])
    ap.add_argument("--no-extras", action="store_true", help="skip the other_minings / e2e variants / parity_check legs")
    ap.add_argument("--two-call", action="store_true", help="device-resident step through npair_forward + npair_backward (the host returns to the "
                    "caller between the passes) instead of npair_forward_backward; the other form is always reported as `step_call_other`")
    ap.add_argument("--no-flush", action="store_true", help="diagnostic: never flush the L2 between steps (sharded runs)")
    ap.add_argument("--cfg-flags", type=int, default=0, help="npair_config.flags (NPAIR_FLAG_*), e.g. 24 = exchange through NCCL instead of peer memory")
    ap.add_argument("--grad-chunk", type=int, default=0, help="npair_config.grad_chunk_cols (0 = library default)")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="after the timed steps, write the tops and the gradient of the last timed step as DIR/<name>.npy (float32, "
                         "at most 64 MB: a seeded sample of the rows of a larger gradient), to compare two builds output for output")
    args = ap.parse_args()
    if args.dump_outputs and args.impl != "ours":
        ap.error("--dump-outputs writes the outputs of the GPU step (--impl ours)")

    from npairloss_b200 import synth
    wl = resolve_workload(args)
    name, B, D, mining, mining_desc, noise, seed, precision = wl
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))

    if args.impl == "reference":
        if rank == 0:
            run_reference(args, wl)
        return

    import torch
    import torch.distributed as dist
    from npairloss_b200 import capi

    assert torch.cuda.is_available(), "bench.py needs a B200 (the product path has no CPU fallback)"
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    host_affinity = None
    if world > 1:
        # one busy-polling host thread per rank: make sure an inherited OMP_PROC_BIND / taskset has not parked all ranks on one core
        try:
            if len(os.sched_getaffinity(0)) < world:
                os.sched_setaffinity(0, range(os.cpu_count()))
            host_affinity = len(os.sched_getaffinity(0))
        except (AttributeError, OSError):
            pass
        dist.init_process_group("nccl", device_id=dev)
    assert world == args.gpus, f"--gpus {args.gpus} but WORLD_SIZE={world}"
    assert B % world == 0
    Q = B // world
    N = B
    peaks = load_peaks()

    # identical bytes on every rank; each rank keeps its own row block
    x, lab = synth.make_inputs(B, D, seed, noise=noise)
    xl = np.ascontiguousarray(x[rank * Q:(rank + 1) * Q])
    ll = np.ascontiguousarray(lab[rank * Q:(rank + 1) * Q])

    def new_nccl_id():
        if world == 1:
            return None
        idt = torch.zeros(128, dtype=torch.uint8, device=dev)
        if rank == 0:
            idt.copy_(torch.frombuffer(bytearray(capi.nccl_unique_id()), dtype=torch.uint8))
        dist.broadcast(idt, 0)
        return bytes(idt.cpu().numpy().tobytes())

    def make_ctx(m, Qr=Q, Dr=D, **kw):
        return capi.Context(capi.make_config(Qr, Dr, world=world, rank=rank, sim_precision=PRECS[precision], device=local_rank,
                                             flags=args.cfg_flags, grad_chunk_cols=args.grad_chunk, **m, **kw), new_nccl_id())

    ctx = make_ctx(mining)
    stream = torch.cuda.current_stream()
    d_x = torch.from_numpy(xl).to(dev)
    d_l = torch.from_numpy(ll).to(dev)
    d_g = torch.empty_like(d_x)

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def step_two_call(c=None):
        c = c or ctx
        tops = c.forward(d_x, d_l)
        c.backward(1.0, d_g)
        return tops

    def step_fused(c=None):
        return (c or ctx).forward_backward(d_x, d_l, 1.0, d_g)

    step_device = step_two_call if args.two_call else step_fused
    step_other = step_fused if args.two_call else step_two_call

    # L2 rule: the step's working set is dominated by the Q x N fp32 similarity block.  When it is larger than twice the 126 MB
    # L2 nothing survives from one step to the next (N = 1: 268 MB); otherwise (sharded runs) a 252 MB device buffer is rewritten
    # before every step and the steps are timed one by one with their own event pair (the flush is outside the pairs).
    L2_BYTES = 126 << 20
    need_flush = 4 * Q * N < 2 * L2_BYTES and not args.no_flush
    flush_buf = torch.empty(2 * L2_BYTES, dtype=torch.uint8, device=dev) if need_flush else None

    def timed_steps(c, steps, fn=None):
        """ms per step (this rank), kernel launches inside the region, the tops of the last step."""
        fn = fn or step_device
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        barrier()
        if not need_flush:
            e0.record(stream)
            l0 = capi.kernel_launches()
            for _ in range(steps):
                t = fn(c)
            nl = capi.kernel_launches() - l0
            e1.record(stream)
            barrier()
            return e0.elapsed_time(e1) / steps, nl, t
        pairs = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(steps)]
        l0 = capi.kernel_launches()
        for ea, eb in pairs:
            flush_buf.fill_(1)                 # same stream as the step: ordered before it, evicts the whole L2
            ea.record(stream)
            t = fn(c)
            eb.record(stream)
        nl = capi.kernel_launches() - l0
        barrier()
        return float(sum(ea.elapsed_time(eb) for ea, eb in pairs)) / steps, nl, t

    def max_over_ranks(v):
        t = torch.tensor([v], dtype=torch.float64, device=dev)
        if world > 1:
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return t.item()

    # ---------------- device-resident timed region ----------------
    sampler = ClockSampler(local_rank)
    if rank == 0:
        sampler.start()            # nvidia-smi takes ~0.1 s to produce its first line: start it ahead of the warm-up
    for _ in range(args.warmup):
        tops = step_device()
    barrier()
    n_before = len(sampler.rows)
    ms_mine, launches_timed, tops_timed = timed_steps(ctx, args.steps)
    grad_timed = d_g.clone() if args.dump_outputs else None      # later legs reuse d_g
    clocks = None
    if rank == 0:
        in_region = len(sampler.rows) - n_before
        # a 50-step timed region lasts ~20 ms, shorter than nvidia-smi's sampling period: keep the SAME load running
        # (untimed) until a handful of samples exist, and say how many fell inside the timed region itself
        t_top = time.perf_counter()
        while len(sampler.rows) - n_before < 6 and time.perf_counter() - t_top < 2.0 and world == 1:
            step_device()
        clocks = sampler.stop()
        clocks["samples_in_timed_region"] = in_region
        clocks["note"] = "sampled with nvidia-smi -lms 25 from warm-up through the timed region and an untimed continuation of the same load"
    ms_step = max_over_ranks(ms_mine)
    value = B / (ms_step * 1e-3)
    # the other form of the step call, timed the same way (flush rule included)
    for _ in range(3):
        step_other()
    ms_other = max_over_ranks(timed_steps(ctx, args.steps, step_other)[0])
    tops = step_device()
    torch.cuda.synchronize()
    grad_dev = d_g.cpu().numpy()

    # ---------------- sharded runs: the same step without the per-step L2 flush, and through npair_forward_backward ----------------
    variants = None
    if world > 1 and not args.no_extras:
        def plain_loop(fn, steps):
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            for _ in range(3):
                fn()
            barrier()
            e0.record(stream)
            for _ in range(steps):
                fn()
            e1.record(stream)
            barrier()
            return max_over_ranks(e0.elapsed_time(e1) / steps)
        ms_nf = plain_loop(lambda: step_device(), args.steps)
        ms_ot = plain_loop(lambda: step_other(), args.steps)
        variants = {"no_l2_flush": {"ms_per_step": ms_nf, "value": B / (ms_nf * 1e-3), "note": "the headline step call back to back, one event pair around the loop, L2 not flushed"},
                    "other_call_no_l2_flush": {"ms_per_step": ms_ot, "value": B / (ms_ot * 1e-3),
                                               "note": ("npair_forward_backward" if args.two_call else "npair_forward + npair_backward (the host returns to the caller between the passes)")}}

    # ---------------- end-to-end through the plugin surface with host buffers ----------------
    # The Caffe-style layer (npairloss_b200/caffe_shim) on HOST blobs: a data layer hands a new batch through mutable_cpu_data()
    # (-> H2D of features + labels from pinned memory), Forward (five tops read on the host), Backward.  The gradient stays in
    # bottom[0]'s device diff, where the upstream layer consumes it in a net; it is fetched once after the loop for the check.
    from npairloss_b200 import caffe_layer
    layer = caffe_layer.Layer(caffe_layer.layer_prototxt(mining, 5), Q, D, 1, 1, world=world, rank=rank, nccl_id=new_nccl_id(),
                              sim_precision=PRECS[precision])
    layer.bottom_data(0)[:] = xl.ravel()
    layer.bottom_data(1)[:] = ll
    h2d = Q * D * 4 + Q * 4
    d2h = 5 * 4 + 4                       # five tops + the error word, read from mapped pinned memory by Forward
    nw = max(3, args.warmup // 2)

    def wall_loop(fn, steps):
        barrier()
        t0 = time.perf_counter()
        for _ in range(steps):
            fn()
        barrier()
        return max_over_ranks(time.perf_counter() - t0) / steps

    e2e_variants = {}
    # (1) double-buffered bottoms, the copy of batch k+1 runs on a copy stream under step k (Caffe's BasePrefetchingDataLayer)
    layer.prefetch_enable()
    for sset in (0, 1):
        layer.set_data(sset, 0)[:] = xl.ravel()
        layer.set_data(sset, 1)[:] = ll
    layer.prefetch(0)
    kk = [0]

    def pf_step():
        layer.prefetch((kk[0] + 1) & 1)                 # one H2D (of the NEXT step's batch) is issued inside every timed step
        t = layer.step_set(kk[0] & 1)
        kk[0] += 1
        return t
    for _ in range(nw + 1):
        tops_p = pf_step()
    s_pf = wall_loop(pf_step, args.steps)
    grad_p = layer.set_diff((kk[0] - 1) & 1).copy()
    e2e_consistent = bool(np.linalg.norm(grad_p - grad_dev) <= 1e-6 * max(np.linalg.norm(grad_dev), 1e-30))
    e2e = {"value": B / s_pf, "unit": "samples/s", "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": d2h,
           "api": ("caffe_shim NPairMultiClassLossLayer (prototxt-configured): Layer::Forward + Layer::Backward on two host bottom sets; "
                   "SyncedMemory::async_gpu_push of the next batch on a copy stream while the current step computes; tops read on the "
                   "host every step, gradient left in bottom[0]'s device diff"),
           "timing": "host wall clock around the loop, device synchronised and ranks barriered on both sides, max over ranks",
           "gradient_matches_device_path": e2e_consistent, "loss": tops_p[0]}
    if not args.no_extras and world == 1:
        # (2) serial: copy, then compute; (3) serial + the gradient copied back to the host every step
        for _ in range(nw):
            layer.step_host(read_gradient=False)
        s_ser = wall_loop(lambda: layer.step_host(read_gradient=False), args.steps)
        s_grad = wall_loop(lambda: layer.step_host(read_gradient=True), args.steps)
        e2e_variants = {"e2e_serial": {"value": B / s_ser, "unit": "samples/s", "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": d2h,
                                       "note": "same layer, one bottom set: H2D of the batch, then Forward + Backward (no overlap)"},
                        "e2e_serial_grad_d2h": {"value": B / s_grad, "unit": "samples/s", "h2d_bytes_per_step": h2d,
                                                "d2h_bytes_per_step": d2h + Q * D * 4,
                                                "note": "as e2e_serial, plus bottom[0]'s diff read on the host every step (cpu_diff)"}}
    layer.close()
    torch.cuda.synchronize()

    # ---------------- profiled pass: per-phase CUDA events (roofline of the dominant kernel) ----------------
    def profile_phases(c, n):
        c.profile_enable(True)
        ph = np.zeros(9)
        for _ in range(n):
            if need_flush:
                flush_buf.fill_(1)
            step_device(c)
            ph += np.array(c.profile_read())
        c.profile_enable(False)
        return ph / n

    phases = profile_phases(ctx, min(args.steps, 10))
    sim_ms, grad_ms = float(phases[2]), float(phases[6])
    flops_alg = 2.0 * Q * N * D                                   # one Q x N x D contraction per launch (SURVEY 8d), both GEMMs
    peak_tf = peaks["tf_sustained"]
    passes = MMA_PASSES[precision]
    # tiles the similarity kernel really issues: world == 1 computes only the 128 x 256 tiles that touch the upper triangle
    tm, tn = (Q + 127) // 128, (N + 255) // 256
    sym_frac = (sum(tn - mb // 2 for mb in range(tm)) / float(tm * tn)) if world == 1 else 1.0

    def tensor_roofline(kernel, ms, issued_factor, extra):
        ach = flops_alg / (ms * 1e-3) / 1e12 if ms > 0 else 0.0
        return {"kernel": kernel, "bound": "tensor", "achieved": ach, "peak": peak_tf, "unit": "TFLOP/s", "frac": ach / peak_tf,
                "mma_passes": passes, "issued_tflops": ach * issued_factor, "frac_of_issued_mma": ach * issued_factor / peak_tf,
                "peak_source": peaks["source"] + ", sustained bf16 (kernel timed inside a long step)",
                "duration_ms": ms, "traffic": None,
                "note": "achieved = algorithmic 2*Q*N*D flops / live CUDA-event duration of the phase; the fp32-faithful modes issue "
                        "mma_passes bf16-rate MMA passes per algorithmic flop; issued_tflops / frac_of_issued_mma count the MMA work "
                        "the kernel really issues (" + extra + ")"}

    r_sim = tensor_roofline("split_gemm_kernel<EPI_SIM*> CTA-pair tcgen05 similarity GEMM + fused row statistics", sim_ms, passes * sym_frac,
                            f"passes x {sym_frac:.3f} of the tiles: symmetric tile list" if world == 1 else "passes x all tiles")
    r_grad = tensor_roofline("fused_grad_kernel CTA-pair tcgen05 gradient GEMM, weights produced into tensor memory, chunked accumulation",
                             grad_ms, passes, "passes x all tiles; includes the split-K reduce when Q = B/world leaves few tiles")
    # DRAM bytes per launch from the committed ncu --set full capture, when it is this workload
    try:
        with open(os.path.join(ROOT, "profiles", "r02_traffic.json")) as f:
            tr = json.load(f)
        w = tr["workload"]
        if (w["B"], w["D"], w["precision"], w["world"]) == (B, D, precision, world):
            r_sim["traffic"] = tr["kernels"]["sim_gemm"]["dram_bytes"]
            r_grad["traffic"] = tr["kernels"]["grad_gemm"]["dram_bytes"]
            r_sim["traffic_source"] = r_grad["traffic_source"] = "profiles/r02_traffic.json (ncu --set full, bytes per launch)"
    except Exception:
        pass
    roofline = r_grad if grad_ms >= sim_ms else r_sim              # the dominant kernel of the step
    roofline_other = [r_sim if grad_ms >= sim_ms else r_grad]
    phase_names = ["fwd_allgather", "operand_prep", "sim_gemm", "thresholds_select", "row_pass_finalize", "weight_build", "grad_gemm",
                   "grad_gemm_T", "bwd_exchange"]
    phase_ms = {n: float(v) for n, v in zip(phase_names, phases)}
    sbytes = 4.0 * Q * N                                           # memory-bound kernels: one fp32 pass over the Q x N block

    def gbs(ms):
        return sbytes / (ms * 1e-3) / 1e9 if ms > 0 else None
    hbm = {"row_pass_GBs": gbs(phases[4]), "row_pass_frac": (gbs(phases[4]) or 0) / peaks["hbm_gbs"],
           "weight_build_GBs": gbs(phases[5]), "hbm_peak_GBs": peaks["hbm_gbs"], "algorithmic_bytes": sbytes}

    # ---------------- the two other mining settings of SURVEY 8d (short runs, N = 1 or sharded alike) ----------------
    other = None
    if not args.no_extras and args.mining == "config" and name in ("HL", "C4") and world == 1:
        other = {}
        for mname, m in (("rand", dict(synth.DEFAULT_MINING)),
                         ("relative", dict(synth.USAGE_MINING, ap_region=synth.LOCAL, ap_method=synth.RELATIVE_HARD, an_region=synth.LOCAL,
                                           an_method=synth.RELATIVE_HARD, identsn=-0.3, diffsn=-0.3, margin_diff=0.0))):
            c2 = make_ctx(m)
            for _ in range(3):
                step_device(c2)
            ms2 = timed_steps(c2, args.steps)[0]
            ms2 = max_over_ranks(ms2)
            ph2 = profile_phases(c2, 5)
            c2.close()
            sel_ms = float(ph2[3])
            other[mname] = {"ms_per_step": ms2, "value": B / (ms2 * 1e-3), "thresholds_select_ms": sel_ms,
                            "select_GBs_per_S_pass": (gbs(sel_ms) if mname == "relative" else None),
                            "select_frac_of_hbm_peak": ((gbs(sel_ms) or 0) / peaks["hbm_gbs"] if mname == "relative" else None),
                            "row_pass_ms": float(ph2[4])}

    # ---------------- N > 1: the NCCL path against an emulation of every rank on one GPU, and against the oracle ----------------
    parity = None
    if world > 1 and not args.no_extras:
        t_all = [torch.empty(5, device=dev) for _ in range(world)]
        dist.all_gather(t_all, torch.tensor(tops, device=dev, dtype=torch.float32))
        parity = {}
        if rank == 0:
            xt, lt = torch.from_numpy(x).to(dev), torch.from_numpy(lab).to(dev)
            rs = torch.empty((world, Q, 8), dtype=torch.float32, device=dev)
            emu_tops, ctx0 = [], None
            for r in range(world):
                ce = capi.Context(capi.make_config(Q, D, world=world, rank=r, sim_precision=PRECS[precision], device=local_rank,
                                                   grad_chunk_cols=args.grad_chunk, **mining))
                emu_tops.append(ce.forward_gathered(xt, lt))
                ce.row_scalars(rs[r])
                if r == 0:
                    ctx0 = ce
                else:
                    ce.close()
            g0 = torch.empty_like(d_g)
            ctx0.backward_gathered(1.0, rs, g0)
            torch.cuda.synchronize()
            ctx0.close()
            got = torch.stack(t_all).cpu().numpy()
            emu = np.array(emu_tops, np.float32)
            gd = g0.cpu().numpy()
            parity["emulated_ranks"] = {
                "what": "rank 0's GPU runs all ranks through npair_forward_gathered / npair_row_scalars / npair_backward_gathered (no NCCL) on the same batch",
                "tops_max_abs_diff_all_ranks": float(np.abs(got - emu).max()), "tops_bitwise_equal": bool(np.array_equal(got, emu)),
                "rank0_gradient_max_abs_diff": float(np.abs(gd - grad_dev).max()), "rank0_gradient_bitwise_equal": bool(np.array_equal(gd, grad_dev)),
                "rank0_gradient_norm": float(np.linalg.norm(grad_dev))}
            del xt, lt, rs, g0
        # small sharded shape against the CPU oracle (the role of tests/test_multi_gpu.py inside the scaling run)
        Bs, Ds = 256 * world, 128
        xs, ls = synth.make_inputs(Bs, Ds, seed=Bs + Ds, noise=2.5)
        Qs = Bs // world
        cs = make_ctx(synth.USAGE_MINING, Qr=Qs, Dr=Ds)
        dxs = torch.from_numpy(np.ascontiguousarray(xs[rank * Qs:(rank + 1) * Qs])).to(dev)
        dls = torch.from_numpy(np.ascontiguousarray(ls[rank * Qs:(rank + 1) * Qs])).to(dev)
        dgs = torch.full_like(dxs, float("nan"))
        ts = cs.forward(dxs, dls)
        cs.backward(0.7, dgs)
        torch.cuda.synchronize()
        Ss = torch.from_numpy(cs.debug_read(0, Qs * Bs).reshape(Qs, Bs)).to(dev)
        cs.close()
        S_all = [torch.empty_like(Ss) for _ in range(world)]
        g_all = [torch.empty_like(dgs) for _ in range(world)]
        ts_all = [torch.empty(5, device=dev) for _ in range(world)]
        dist.all_gather(S_all, Ss); dist.all_gather(g_all, dgs)
        dist.all_gather(ts_all, torch.tensor(ts, device=dev, dtype=torch.float32))
        if rank == 0:
            from oracle import oracle_lib as o
            ocfg = o.make_config(Qs, Ds, world=world, faithful_sorts=0, **synth.USAGE_MINING)
            tops_o, dx_o = o.step_world(xs, ls, ocfg, 0.7, S_inject_all=torch.cat(S_all).cpu().numpy())
            dxg = torch.cat(g_all).cpu().numpy()
            tg = torch.stack(ts_all).cpu().numpy()
            grel = float(np.linalg.norm(dxg - dx_o) / max(np.linalg.norm(dx_o), 1e-30))
            lrel = float(np.abs(tg[:, 0] - tops_o[:, 0]).max() / max(np.abs(tops_o[:, 0]).max(), 1e-30))
            parity["oracle_small"] = {"shape": f"B={Bs} (Q={Qs} per rank), D={Ds}, usage-block mining, loss_weight 0.7",
                                      "loss_max_rel_err": lrel, "gradient_normwise_rel_err": grel,
                                      "retrieval_max_row_diff": float(np.abs(tg[:, 1:4] - tops_o[:, 1:4]).max() * Qs),
                                      "pass": bool(np.isfinite(dxg).all() and grel <= 1e-5 and lrel <= 1e-5)}
        barrier()

    # ---------------- CPU baseline (rank 0, bounded sample) ----------------
    cpu = None
    if rank == 0 and not args.no_cpu_baseline:
        ws = cpu_sample_world(B)
        step, Qs = oracle_sample(B, D, mining, x, lab, ws, host_threads())
        step()                                                    # warm-up (page faults, thread pool)
        times, t_all0 = [], time.perf_counter()
        while len(times) < 3 or (time.perf_counter() - t_all0 < 12 and len(times) < 12):
            t0 = time.perf_counter()
            step()
            times.append(time.perf_counter() - t0)
        dt = float(np.median(times))
        cpu = {"value": Qs / dt, "unit": "samples/s", "cores": host_threads(), "kind": "port",
               "sample": f"rank-0 block of a {ws}-way anchor sharding: {Qs} anchors x {B} database x D={D}, median of {len(times)} reps "
                         f"(min {min(times) * 1e3:.0f} ms, max {max(times) * 1e3:.0f} ms), faithful unconditional sorts, fp32 accumulate, OpenMP, "
                         "one pinned thread per physical core"}

    if rank == 0:
        out = {"metric": metric_name(B, D), "value": value, "unit": "samples/s", "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
               "ms_per_step": ms_step, "higher_is_better": True, "scaling": "strong", "vs_baseline": None,
               "dtype": DTYPE_DESC[precision], "data": "synthetic",
               "config": {"workload": f"{name}: B={B}, D={D}, {B // 2} classes x 2, {mining_desc}, loss_weight 1",
                          "global_batch": B, "feature_dim": D, "rows_per_rank": Q, "sharding": f"anchor-sharded x{world}",
                          "precision": precision, "noise": noise, "seed": seed, "cfg_flags": args.cfg_flags,
                          "host_cpus_allowed_per_rank": host_affinity,
                          "exchange": (None if world == 1 else ("NCCL all-gathers" if args.cfg_flags & 24 == 24 else "peer-memory pushes over NVLink (cudaIpc), NCCL only for bootstrap")),
                          "step_call": "npair_forward + npair_backward" if args.two_call else "npair_forward_backward (both passes enqueued, one wait for the five tops)",
                          "l2": (f"flushed: a {2 * L2_BYTES >> 20} MB device buffer is rewritten before every timed step (per-rank S = "
                                 f"{4 * Q * N / 1e6:.0f} MB fp32 would otherwise stay in the 126 MB L2); steps timed one by one, flush excluded"
                                 if need_flush else
                                 f"not flushed: per-step working set (S {4 * Q * N / 1e6:.0f} MB fp32 + operand pieces) is more than twice the 126 MB L2")},
               "clocks": clocks, "roofline": roofline, "roofline_other": roofline_other, "phase_ms": phase_ms, "hbm_kernels": hbm,
               "step_call_other": {"call": ("npair_forward_backward" if args.two_call else "npair_forward + npair_backward"), "ms_per_step": ms_other,
                                   "value": B / (ms_other * 1e-3), "note": "the other form of the step call, timed like the headline"},
               "other_minings": other, "sharded_variants": variants, "parity_check": parity, "cpu_baseline": cpu, "e2e": e2e, **e2e_variants,
               "gpu_launches": launches_timed,
               "tops": {"loss": tops[0], "top1": tops[1], "top5": tops[2], "top10": tops[3], "feature_asum": tops[4]}}
        emit(out)
    if args.dump_outputs:
        dump_outputs(args.dump_outputs, tops_timed, grad_timed, world, rank)
    ctx.close()
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
