#!/usr/bin/env python
"""bench.py - headline metric of BASELINE.json: clips/sec forward on synthetic clips.

Workload at every N: SlowFast-8x8-R50 eval forward, batch 8 per GPU, 3x32x224x224 synthetic clips
(slow 8 + fast 32 frames) - BASELINE.json configs[1].  One "step" = one forward pass over one
batch; weak scaling (per-GPU batch fixed), clips sharded across ranks, one NCCL all-gather of the
[8,400] logits per step.

  python bench.py [--gpus N] [--steps K] [--warmup W] [--impl b200|reference] [--workload NAME] [--dump-outputs DIR]

Prints ONE JSON line on rank 0 (see the contract in the task statement): value = whole-job
clips/s with inputs resident in HBM; e2e = same through the public model call with pinned HOST
inputs (H2D + D2H inside the timed region); roofline for the dominant kernel
(conv3d_igemm_kernel, tensor-bound) from per-launch CUDA-event times; cpu_baseline = the oracle
port of the reference forward timed on this box's host cores (bounded sample).
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

import torch  # noqa: E402

WORKLOADS = {
    # name: (hub builder, per-GPU batch, T, H, W, slowfast?)
    "slowfast_r50": ("slowfast_r50", 8, 32, 224, 224, True),
    "x3d_m": ("x3d_m", 32, 16, 224, 224, False),
    "x3d_xs": ("x3d_xs", 8, 4, 160, 160, False),
    "slow_r50": ("slow_r50", 8, 8, 224, 224, False),
    "csn_r101": ("csn_r101", 8, 32, 224, 224, False),
    "r2plus1d_r50": ("r2plus1d_r50", 8, 16, 224, 224, False),
    "mvit_base_16x4": ("mvit_base_16x4", 8, 16, 224, 224, False),
}
METRIC = "clips/sec forward (synthetic 3xTx224^2)"


def load_peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        d = json.load(open(p))
        return {"hbm_gbs": d.get("hbm_gbs", 6650.0), "tflops_burst": d.get("bf16_tflops", 1590.0),
                "tflops_sustained": d.get("bf16_tflops_sustained", 1400.0), "source": "measured"}
    return {"hbm_gbs": 6650.0, "tflops_burst": 1590.0, "tflops_sustained": 1400.0, "source": "fallback"}


class ClockSampler:
    """SM clock + throttle reasons sampled DURING the timed region (B200_PROFILING.md clocks line).
    NVML in a thread every ~5 ms (the timed region is ~0.1 s, too short for `nvidia-smi -lms`);
    falls back to an `nvidia-smi -lms 100` child process if pynvml is unavailable."""

    REASONS = {0x8: "hw_slowdown", 0x40: "hw_thermal_slowdown", 0x20: "sw_thermal_slowdown", 0x4: "sw_power_cap"}

    def __init__(self, index):
        self.index, self.proc, self.lines = index, None, []
        self.samples, self.bits, self.mx, self.stop_flag, self.thr = [], 0, None, False, None

    def _nvml_loop(self, nv, h):
        while not self.stop_flag:
            try:
                self.samples.append(float(nv.nvmlDeviceGetClockInfo(h, nv.NVML_CLOCK_SM)))
                try:
                    self.bits |= int(nv.nvmlDeviceGetCurrentClocksEventReasons(h))
                except Exception:
                    self.bits |= int(nv.nvmlDeviceGetCurrentClocksThrottleReasons(h))
            except Exception:
                pass
            time.sleep(0.005)

    def start(self):
        try:
            import pynvml as nv
            nv.nvmlInit()
            idx = self.index
            vis = os.environ.get("CUDA_VISIBLE_DEVICES")
            if vis:
                idx = int(vis.split(",")[self.index])
            h = nv.nvmlDeviceGetHandleByIndex(idx)
            self.mx = float(nv.nvmlDeviceGetMaxClockInfo(h, nv.NVML_CLOCK_SM))
            self.thr = threading.Thread(target=self._nvml_loop, args=(nv, h), daemon=True)
            self.thr.start()
            return
        except Exception:
            self.thr = None
        q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
             "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
             "clocks_event_reasons.sw_power_cap")
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.index), "--query-gpu=" + q,
                                          "--format=csv,noheader,nounits", "-lms", "100"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.t = threading.Thread(target=self._read, daemon=True)
            self.t.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.lines.append(line.strip())

    def stop(self):
        if self.thr is not None:
            self.stop_flag = True
            self.thr.join(timeout=2)
            sm = sorted(self.samples)
            med = sm[len(sm) * 3 // 4] if sm else None     # upper-quartile ~ clocks under load (idle samples drag the median down)
            reasons = sorted(name for bit, name in self.REASONS.items() if self.bits & bit)
            return {"sm_mhz": med, "sm_max_mhz": self.mx, "reasons": reasons, "samples": len(sm), "source": "nvml"}
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        try:
            self.proc.wait(timeout=5)
        except Exception:
            self.proc.kill()
        sm, mx, reasons = [], None, set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for ln in self.lines:
            f = [v.strip() for v in ln.split(",")]
            if len(f) < 7:
                continue
            try:
                sm.append(float(f[0]))
                mx = float(f[1])
            except ValueError:
                continue
            for name, v in zip(names, f[3:7]):
                if v.lower().startswith("active"):
                    reasons.add(name)
        sm.sort()
        # median of the upper half ~ clocks under load (idle samples before/after drag the median down)
        med = sm[len(sm) * 3 // 4] if sm else None
        return {"sm_mhz": med, "sm_max_mhz": mx, "reasons": sorted(reasons), "samples": len(sm), "source": "nvidia-smi"}


def build_model_and_inputs(workload, batch_override=None):
    import pytorchvideo_b200.models.hub as H
    from pytorchvideo_b200 import testing as TS
    hub, B, T, Hh, W, is_sf = WORKLOADS[workload]
    if batch_override:
        B = batch_override
    model = TS.randomize_model(getattr(H, hub)(), seed=1234).eval()
    return model, B, T, Hh, W, is_sf


def make_inputs(B, T, H, W, is_sf, seed):
    from pytorchvideo_b200 import testing as TS
    clip = TS.synthetic_clip(B, T, H, W, seed=seed)
    return TS.slowfast_inputs(clip) if is_sf else clip


def dump_outputs(dirname, arrays):
    """--dump-outputs: write what the timed path returned in its last step as DIR/<name>.npy (float32).  Inputs and
    weights come from fixed seeds, so two builds run with the same arguments can be compared output for output."""
    import numpy as np
    os.makedirs(dirname, exist_ok=True)
    for name, t in arrays.items():
        np.save(os.path.join(dirname, name + ".npy"), t.detach().float().cpu().numpy())


def pick_cpu_threads(model, T, H, W, is_sf):
    """The reference (ATen/oneDNN conv3d) does not scale to every core of a 128-thread host at these
    sizes - pick the thread count that is actually fastest (candidates <= visible cores)."""
    from oracle.interp import oracle_forward
    cores = os.cpu_count() or 1
    cands = sorted(set(c for c in (8, 16, 32, 64, cores) if c <= cores))
    inp = make_inputs(1, T, H, W, is_sf, seed=7)
    best, best_t = cands[0], None
    for c in cands:
        torch.set_num_threads(c)
        if best_t is None:
            oracle_forward(model, inp)          # warm-up (allocator, oneDNN primitives)
        t0 = time.perf_counter()
        oracle_forward(model, inp)
        dt = time.perf_counter() - t0
        if best_t is None or dt < best_t:
            best, best_t = c, dt
        if dt > 4 * best_t:
            break                               # more threads only get slower from here
    torch.set_num_threads(best)
    return best, best_t


def cpu_baseline(model, T, H, W, is_sf, budget_s=20.0):
    """Oracle port of the reference forward on the host cores: bounded sample, the faster of one clip per
    forward and a small batch per forward (on a many-core host oneDNN's conv3d is fastest at batch 1)."""
    from oracle.interp import oracle_forward
    cores, one = pick_cpu_threads(model, T, H, W, is_sf)
    results = []
    for b in (1, max(1, min(8, int(budget_s / max(one, 1e-3) / 4)))):
        if results and b == results[0][1]:
            continue
        inp = make_inputs(b, T, H, W, is_sf, seed=7)
        reps = 3 if one * b * 3 < budget_s / 2 else 1
        best = None
        for _ in range(reps):
            t0 = time.perf_counter()
            oracle_forward(model, inp)
            dt = time.perf_counter() - t0
            best = dt if best is None else min(best, dt)
        results.append((b / best, b, reps))
    v, b, reps = max(results)
    return {"value": v, "unit": "clips/s", "cores": cores, "kind": "port",
            "sample": "%d clip(s) per forward, best of %d, torch fp32 CPU, %d threads (tried batch sizes %s)" % (
                b, reps, cores, [r[1] for r in results])}


def run_reference(args, rank, world):
    """--impl reference: the reference's CPU implementation of the path (oracle port; the reference
    itself is a Python library that cannot travel to this box).  Rank 0 only."""
    if rank != 0:
        return
    model, B, T, H, W, is_sf = build_model_and_inputs(args.workload)
    from oracle.interp import oracle_forward
    cores, _ = pick_cpu_threads(model, T, H, W, is_sf)
    b = 1   # bounded sample: one clip per step
    inp = make_inputs(b, T, H, W, is_sf, seed=7)
    for _ in range(max(1, min(args.warmup, 1))):
        oracle_forward(model, inp)
    t0 = time.perf_counter()
    for _ in range(args.steps):
        out = oracle_forward(model, inp)
    dt = time.perf_counter() - t0
    if args.dump_outputs:
        dump_outputs(args.dump_outputs, {"logits": out})
    v = b * args.steps / dt
    line = {"impl": "reference", "metric": METRIC, "value": v, "unit": "clips/s", "n_gpus": args.gpus,
            "steps": args.steps, "warmup": args.warmup, "ms_per_step": dt / args.steps * 1e3,
            "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            # the b200 arm's workload; each reference step is a bounded SAMPLE of it (batch_per_step clips of the batch)
            "config": {"workload": args.workload, "clip": [3, T, H, W], "batch_per_gpu": B, "global_batch": B * max(1, args.gpus),
                       "parallelism": "dp%d" % max(1, args.gpus), "batch_per_step": b,
                       "note": "reference CPU forward restated in oracle/interp.py (bit-exact vs the reference in the authoring container); "
                               "each step = %d clip of the %d-clip batch on the host cores" % (b, B)},
            "cpu_baseline": {"value": v, "unit": "clips/s", "cores": cores, "kind": "port",
                             "sample": "%d clip per step x %d steps" % (b, args.steps)},
            "e2e": {"value": v, "unit": "clips/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
            "gpu_launches": 0}
    print(json.dumps(line), flush=True)


def run_torch_gpu(args, rank, world):
    """--impl torch-gpu: CONTEXT number, not a product path and not the reference arm - the oracle interpreter
    (plain torch.nn.functional calls) on the same B200 in f16 with channels_last_3d inputs, i.e. stock
    cuDNN / cuBLAS / ATen kernels (SURVEY section 2: "beat stock PyTorch on the same B200" is the per-op bar)."""
    if rank != 0:
        return
    from oracle.interp import Oracle
    dev = torch.device("cuda", 0)
    model, B, T, H, W, is_sf = build_model_and_inputs(args.workload)
    model = model.to(dev).half()
    inp = make_inputs(B, T, H, W, is_sf, seed=42)
    inp = [t.to(dev).half().contiguous(memory_format=torch.channels_last_3d) for t in inp] if is_sf else \
        inp.to(dev).half().contiguous(memory_format=torch.channels_last_3d)
    torch.backends.cudnn.benchmark = True
    orc = Oracle()

    def step():
        with torch.no_grad():
            return orc.run(model, list(inp) if is_sf else inp)
    for _ in range(max(args.warmup, 3)):
        step()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(args.steps):
        out = step()
    e1.record()
    torch.cuda.synchronize()
    if args.dump_outputs:
        dump_outputs(args.dump_outputs, {"logits": out})
    ms = e0.elapsed_time(e1) / args.steps
    print(json.dumps({"impl": "torch-gpu", "metric": METRIC, "value": B / (ms / 1e3), "unit": "clips/s", "n_gpus": 1,
                      "steps": args.steps, "warmup": args.warmup, "ms_per_step": ms, "higher_is_better": True,
                      "dtype": "f16", "data": "synthetic",
                      "config": {"workload": args.workload, "clip": [3, T, H, W], "batch_per_gpu": B,
                                 "note": "stock PyTorch %s eager (cuDNN/cuBLAS) f16 channels_last_3d, cudnn.benchmark; context only" % torch.__version__}}),
          flush=True)


def load_traffic(kernel):
    """DRAM bytes per launch of `kernel`, measured offline with ncu (profiles/r02_traffic.json, written by
    tools/summarize_profiles.py from `ncu --metrics dram__bytes_read.sum,dram__bytes_write.sum`)."""
    p = os.path.join(ROOT, "profiles", "r02_traffic.json")
    try:
        return json.load(open(p)).get(kernel)
    except Exception:
        return None


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference", "torch-gpu"])
    ap.add_argument("--workload", default="slowfast_r50", choices=sorted(WORKLOADS))
    ap.add_argument("--precision", default="f16", choices=["f16", "f32"])
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--resident-only", action="store_true", help="A/B runs: time the resident step only and print a short line")
    ap.add_argument("--dump-kernels", default=None, help="write per-launch times (JSON) to this path")
    ap.add_argument("--dump-outputs", default=None, metavar="DIR",
                    help="write the logits of the last timed step to DIR/logits.npy (float32)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    args.warmup = max(args.warmup, 3)

    from pytorchvideo_b200 import parallel as PAR
    rank, local_rank, world = PAR.env_world()
    if args.impl == "reference":
        run_reference(args, rank, world)
        return
    if args.impl == "torch-gpu":
        run_torch_gpu(args, rank, world)
        return

    import torch.distributed as dist
    from pytorchvideo_b200 import _lib
    from pytorchvideo_b200.engine import compile_model
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    _lib.require_device()
    numa = None
    if world > 1:
        numa = PAR.bind_to_gpu_numa(local_rank)      # before any pinned allocation (first touch on the GPU's socket)
        PAR.init_process_group("nccl")

    model, B, T, H, W, is_sf = build_model_and_inputs(args.workload)
    host_in = make_inputs(B, T, H, W, is_sf, seed=42 + rank)          # this rank's shard of the global batch
    host_list = host_in if is_sf else [host_in]
    pinned = [t.pin_memory() for t in host_list]
    dev_in = [t.to(dev) for t in host_list]
    cm = compile_model(model, dev_in if is_sf else dev_in[0], dtype=args.precision, use_graph=True)
    num_classes = cm.out_shape[1]
    gathered = torch.empty((world * B, num_classes), dtype=torch.float32, device=dev)

    def step_resident():
        out = cm(dev_in if is_sf else dev_in[0])
        if world > 1:
            dist.all_gather_into_tensor(gathered, out)
            return gathered
        return out

    host_out = torch.empty((B, num_classes), dtype=torch.float32).pin_memory()

    def step_e2e_serial():
        # the plain public call with HOST inputs: H2D of the clips, forward, D2H of the logits, in sequence
        out = cm(pinned if is_sf else pinned[0])
        if world > 1:
            dist.all_gather_into_tensor(gathered, out)
        host_out.copy_(out, non_blocking=True)
        torch.cuda.current_stream().synchronize()

    # the serving call: same copies every step, but batch i+1's H2D overlaps batch i's forward
    pipe = cm.pipeline(depth=2)
    if world > 1:
        def _gather(out):
            dist.all_gather_into_tensor(gathered, out)
            return gathered
        pipe.post = _gather
    tickets = []

    def step_e2e():
        tickets.append(pipe.submit(pinned if is_sf else pinned[0]))
        if len(tickets) > 1:
            pipe.result(tickets.pop(0))          # logits of the previous batch are on the host now

    def drain_e2e():
        while tickets:
            pipe.result(tickets.pop(0))

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    last = {}

    def timed(fn, steps, drain=None):
        barrier()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(steps):
            last["out"] = fn()
        if drain is not None:
            drain()                              # every step's result is read inside the timed region
        e1.record()
        barrier()
        ms = e0.elapsed_time(e1)
        if world > 1:
            t = torch.tensor([ms], device=dev)
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
            ms = float(t.item())
        return ms

    for _ in range(args.warmup):
        step_resident()
    sampler = ClockSampler(local_rank)
    if rank == 0:
        sampler.start()
        time.sleep(0.02)
    launches_before = _lib.launch_count()
    ms = timed(step_resident, args.steps)
    clocks = sampler.stop() if rank == 0 else None
    if args.dump_outputs and rank == 0:
        # the step returns a view of the plan's static output buffer: copy it before the e2e passes below reuse the plan
        dump_outputs(args.dump_outputs, {"logits": last["out"]})
    ms_per_step = ms / args.steps
    value = world * B * args.steps / (ms / 1e3)

    if args.resident_only:
        if rank == 0:
            print(json.dumps({"workload": args.workload, "ms_per_step": ms_per_step, "value": value, "n_gpus": world,
                              "launches_per_step": cm.plan.num_launches(), "resident_only": True,
                              "env": {k: v for k, v in os.environ.items() if k.startswith("PVB200_")}}), flush=True)
        if world > 1:
            dist.destroy_process_group()
        return
    for _ in range(2):
        step_e2e_serial()
    ms_e2e_serial = timed(step_e2e_serial, args.steps)
    for _ in range(3):
        step_e2e()
    drain_e2e()
    ms_e2e = timed(step_e2e, args.steps, drain_e2e)
    e2e_value = world * B * args.steps / (ms_e2e / 1e3)
    h2d = sum(t.numel() * t.element_size() for t in pinned)
    d2h = host_out.numel() * host_out.element_size()

    # The fp32 host clips make the e2e number PCIe-bound (SlowFast: 193 MB per step at ~53 GB/s = 3.6 ms > the forward).
    # Same serving loop with f16 pinned host clips (what a decoder + fused transform hands over): reported beside it.
    e2e16 = None
    if args.precision == "f16":
        pinned16 = [t.half().pin_memory() for t in host_list]
        cm16 = compile_model(model, [t.to(dev) for t in pinned16] if is_sf else pinned16[0].to(dev), dtype="f16", use_graph=True)
        pipe16 = cm16.pipeline(depth=2)
        if world > 1:
            pipe16.post = _gather
        t16 = []

        def step16():
            t16.append(pipe16.submit(pinned16 if is_sf else pinned16[0]))
            if len(t16) > 1:
                pipe16.result(t16.pop(0))

        def drain16():
            while t16:
                pipe16.result(t16.pop(0))
        for _ in range(3):
            step16()
        drain16()
        ms16 = timed(step16, args.steps, drain16)
        e2e16 = {"value": world * B * args.steps / (ms16 / 1e3), "ms_per_step": ms16 / args.steps,
                 "h2d_bytes_per_step": sum(t.numel() * t.element_size() for t in pinned16)}
        del cm16, pipe16

    # ---- roofline of the dominant kernel (per-launch CUDA events, eager replay on torch's stream)
    per_op = cm.plan.profile(iters=3)
    kinds = {}
    for m, t in zip(cm.plan.meta, per_op):
        k = kinds.setdefault(m["kind"], {"ms": 0.0, "flops": 0.0, "bytes": 0.0, "n": 0})
        k["ms"] += t; k["flops"] += m["flops"]; k["bytes"] += m["bytes"]; k["n"] += 1
    total_ms = sum(per_op)
    peaks = load_peaks()
    dom = max(kinds, key=lambda k: kinds[k]["ms"])
    kd = kinds[dom]
    # The per-launch CUDA events come from an eager single-stream replay; the benchmarked step is a CUDA graph with
    # PDL-overlapped launches and concurrent lanes, so the launches' summed eager time exceeds the step time.  The
    # kernel's time INSIDE the benchmarked step is its share of the launch time x the measured step time.
    share = kd["ms"] / total_ms
    in_step_ms = share * ms_per_step
    kname = {"tcgen05": "conv3d_igemm_kernel", "attention": "attention_mma_kernel", "depthwise": "dwconv3d_tile_kernel"}.get(dom, dom)
    traffic = load_traffic(kname)
    if dom in ("tcgen05", "attention"):
        achieved = kd["flops"] / (in_step_ms * 1e-3) / 1e12
        peak = peaks["tflops_sustained"]
        roof = {"bound": "tensor", "kernel": kname, "achieved": achieved, "peak": peak,
                "unit": "TFLOP/s", "frac": achieved / peak, "traffic": traffic,
                "launches": kd["n"], "avg_launch_us": in_step_ms / kd["n"] * 1e3,
                "avg_launch_us_eager": kd["ms"] / kd["n"] * 1e3, "achieved_eager": kd["flops"] / (kd["ms"] * 1e-3) / 1e12,
                "share_of_step": share, "peak_source": peaks["source"] + " (sustained cuBLAS bf16)",
                "algorithmic_gflop_per_launch": kd["flops"] / kd["n"] / 1e9,
                "timing": "share of per-launch CUDA-event time (eager replay) x measured graph step time"}
    else:
        achieved = kd["bytes"] / (in_step_ms * 1e-3) / 1e9
        peak = peaks["hbm_gbs"]
        roof = {"bound": "hbm", "kernel": kname, "achieved": achieved, "peak": peak, "unit": "GB/s",
                "frac": achieved / peak, "traffic": traffic, "launches": kd["n"],
                "avg_launch_us": in_step_ms / kd["n"] * 1e3, "avg_launch_us_eager": kd["ms"] / kd["n"] * 1e3,
                "achieved_eager": kd["bytes"] / (kd["ms"] * 1e-3) / 1e9, "share_of_step": share,
                "algorithmic_mb_per_launch": kd["bytes"] / kd["n"] / 1e6,
                "peak_source": peaks["source"],
                "timing": "share of per-launch CUDA-event time (eager replay) x measured graph step time"}
    # Two more views of the same kernel, beside the primary one: (1) its launches judged as an HBM stream (many of them are:
    # conv_c + residual moves 231 MB for 6.6 GFLOP); (2) every launch against ITS OWN binding roofline,
    # sum_i max(flops_i / tensor peak, bytes_i / HBM peak) / time in the step - the fraction of the per-launch speed of light.
    dom_ops = [(m, t) for m, t in zip(cm.plan.meta, per_op) if m["kind"] == dom]
    ideal_ms = sum(max(m["flops"] / (peaks["tflops_sustained"] * 1e12), m["bytes"] / (peaks["hbm_gbs"] * 1e9)) for m, _ in dom_ops) * 1e3
    roof["hbm_view"] = {"achieved": kd["bytes"] / (in_step_ms * 1e-3) / 1e9, "peak": peaks["hbm_gbs"], "unit": "GB/s",
                        "frac": kd["bytes"] / (in_step_ms * 1e-3) / 1e9 / peaks["hbm_gbs"],
                        "algorithmic_mb_per_launch": kd["bytes"] / kd["n"] / 1e6}
    roof["per_launch_roofline_frac"] = ideal_ms / in_step_ms
    roof["launches_hbm_bound"] = sum(1 for m, _ in dom_ops
                                     if m["bytes"] / (peaks["hbm_gbs"] * 1e9) > m["flops"] / (peaks["tflops_sustained"] * 1e12))
    model_flops = sum(m["flops"] for m in cm.plan.meta)
    whole = {"model_gflop_per_clip": model_flops / B / 1e9,
             "model_tflops_achieved": model_flops / (ms_per_step * 1e-3) / 1e12,
             "frac_of_tensor_peak": model_flops / (ms_per_step * 1e-3) / 1e12 / peaks["tflops_sustained"],
             "kernel_ms_by_kind": {k: round(v["ms"], 4) for k, v in kinds.items()},
             "sum_kernel_ms": round(total_ms, 4)}
    if args.dump_kernels and rank == 0:
        json.dump([{**m, "ms": t} for m, t in zip(cm.plan.meta, per_op)], open(args.dump_kernels, "w"), indent=0)

    if rank == 0:
        cpu = None
        if world == 1 and not args.no_cpu_baseline:
            cpu = cpu_baseline(model, T, H, W, is_sf)
        line = {"metric": METRIC, "value": value, "unit": "clips/s", "n_gpus": world, "steps": args.steps,
                "warmup": args.warmup, "ms_per_step": ms_per_step, "higher_is_better": True, "scaling": "weak",
                "vs_baseline": None, "dtype": "f16" if args.precision == "f16" else "f32", "data": "synthetic",
                "config": {"workload": args.workload, "clip": [3, T, H, W], "batch_per_gpu": B, "global_batch": B * world,
                           "parallelism": "dp%d" % world, "numa_bound": numa is not None, "l2": "inputs (%.0f MB/step) larger than L2; CUDA-graph replay" % (h2d / 1e6),
                           "weights": "random (seeded), BN stats randomised"},
                "e2e": {"value": e2e_value, "unit": "clips/s", "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": d2h,
                        "ms_per_step": ms_e2e / args.steps, "mode": "double-buffered H2D/compute/D2H (engine/pipeline.py)",
                        "serial_ms_per_step": ms_e2e_serial / args.steps, "host_dtype": "f32 pinned clips (PCIe-bound)",
                        "f16_host_clips": e2e16},
                "gpu_launches": args.steps * cm.plan.num_launches(),
                "launches_per_step": cm.plan.num_launches(),
                "roofline": roof, "whole_model": whole, "clocks": clocks}
        if cpu is not None:
            line["cpu_baseline"] = cpu
        print(json.dumps(line), flush=True)
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
