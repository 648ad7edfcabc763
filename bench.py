#!/usr/bin/env python
"""Benchmark of the CFP fusion + cross-zone propagation path (BASELINE.json metric:
"CFP fusion frames/s @416x544, 8x8 zones").

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl cfp|reference] [--dump-outputs DIR]

One *step* = one pass of the hot path (histogram encoder + the three TransformerFusion
calls) over one batch of synthetic frames.  Workload = BASELINE.json configs[2]:
combine1 layer list, bf16, 64 frames per GPU, 416x544 input with 8x8 zones of 48 px.
Launched under torchrun for N>1: one process per GPU, frames sharded by batch, no
data-path collective (weak scaling); the time is the max over ranks.

``--impl reference`` times the reference's CPU algorithm (the oracle port of the PyTorch
modules, oracle/cfp_oracle.py) on the host cores, on a bounded sample of the same workload.

``--dump-outputs DIR`` writes what the last timed step returned (rank 0's fused maps) as float32
DIR/fused3.npy, fused2.npy, fused1.npy, so that two builds can be compared output for output:
the inputs, weights and positional-encoding crops are seeded, identical from run to run.
"""
from __future__ import annotations

import argparse
import json
import os
import statistics
import subprocess
import sys
import threading
import time

import torch

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

from cfpnet_b200 import synth  # noqa: E402

METRIC = "CFP fusion frames/s @416x544, 8x8 zones"
GEOMETRY = "G416"
# SURVEY.md §8d / BASELINE.md §3 (combine1, 416x544): algorithmic work per frame
FLOP_PER_FRAME = 13.22e9
DENSE_FLOP_PER_FRAME = 11.26e9
ELEMS_PER_FRAME = 15.43e6
DUMP_BYTES = 64 * 10**6             # --dump-outputs: every file together, .npy headers included


def dump_outputs(out_dir, named):
    """Write each (name, tensor) as float32 ``out_dir/<name>.npy``.  When the arrays together exceed DUMP_BYTES, every
    one is cut to the same share of its elements: flat positions drawn by a fixed seed, in increasing order (a 1-D
    array), so that runs with the same arguments store the same positions."""
    import numpy as np
    os.makedirs(out_dir, exist_ok=True)
    total = sum(t.numel() for _, t in named)
    share = min(1.0, (DUMP_BYTES - 1024 * len(named)) / (4 * total))
    for name, t in named:
        t = t.detach().float().cpu()
        if share < 1.0:
            idx = torch.randperm(t.numel(), generator=torch.Generator().manual_seed(0))[: int(t.numel() * share)]
            t = t.reshape(-1)[idx.sort().values]
        np.save(os.path.join(out_dir, name + ".npy"), t.numpy())
    return share


def load_peaks():
    try:
        with open(os.path.join(ROOT, "MEASURED_PEAKS.json")) as fh:
            p = json.load(fh)
        return {"hbm_gbs": float(p["hbm_gbs"]), "bf16_tflops": float(p["bf16_tflops"]),
                "bf16_tflops_sustained": float(p.get("bf16_tflops_sustained", p["bf16_tflops"])),
                "source": "measured (MEASURED_PEAKS.json)"}
    except Exception:
        return {"hbm_gbs": 6650.0, "bf16_tflops": 1590.0, "bf16_tflops_sustained": 1400.0,
                "source": "fallback (B200_PROFILING.md)"}


def bind_host_to_gpu(index):
    """Pin this process to the CPU cores NVML reports as local to GPU `index` (its NUMA node) BEFORE the pinned host
    buffers are allocated, so that first-touch places them on that node and the copy engine does not cross the socket
    interconnect.  Returns a short description for the JSON line (or why nothing was done)."""
    try:
        import pynvml
        pynvml.nvmlInit()
        h = pynvml.nvmlDeviceGetHandleByIndex(index)
        ncpu = os.cpu_count() or 1
        words = pynvml.nvmlDeviceGetCpuAffinity(h, (ncpu + 63) // 64)
        cpus = [w * 64 + b for w, word in enumerate(words) for b in range(64) if (word >> b) & 1 and w * 64 + b < ncpu]
        allowed = sorted(set(cpus) & set(os.sched_getaffinity(0)))
        if not allowed:
            return "nvml affinity empty / outside the cgroup: not bound"
        os.sched_setaffinity(0, allowed)
        try:
            numa = pynvml.nvmlDeviceGetNumaNodeId(h)
        except Exception:
            numa = None
        return f"bound to {len(allowed)} cpus [{allowed[0]}..{allowed[-1]}] (NVML affinity of GPU {index}, numa {numa})"
    except Exception as e:                                  # noqa: BLE001
        return f"not bound ({type(e).__name__}: {e})"


def probe_host_link(dev, nbytes_in, nbytes_out, barrier, reps=6):
    """Host<->device copy ceiling of THIS run: every rank copies `nbytes_in` host->device and `nbytes_out` device->host
    concurrently (two streams, pinned buffers), all ranks at once - the traffic pattern of the e2e loop without any
    compute.  Returns seconds per (in + out) pair on this rank."""
    h_in = torch.empty(nbytes_in, dtype=torch.uint8).pin_memory()
    h_out = torch.empty(nbytes_out, dtype=torch.uint8).pin_memory()
    d_in = torch.empty(nbytes_in, dtype=torch.uint8, device=dev)
    d_out = torch.empty(nbytes_out, dtype=torch.uint8, device=dev)
    s1, s2 = torch.cuda.Stream(dev), torch.cuda.Stream(dev)

    def both():
        with torch.cuda.stream(s1):
            d_in.copy_(h_in, non_blocking=True)
        with torch.cuda.stream(s2):
            h_out.copy_(d_out, non_blocking=True)
    both()
    barrier()
    t0 = time.perf_counter()
    for _ in range(reps):
        both()
    torch.cuda.synchronize()
    dt = (time.perf_counter() - t0) / reps
    barrier()
    return dt


class ClockSampler(threading.Thread):
    """SM clock and throttle reasons during the timed region, read in-process through NVML
    (nvidia_ml_py) every 200 ms plus one explicit sample in the middle of the timed loop.  Clock queries
    were measured to stall GPU work by 50-100 ms now and then (one step of ten taking 108 ms instead of
    6.4, both with `nvidia-smi -lms 50` in a child process and with NVML polled every 25 ms), hence the
    low rate.  NVML is initialised before the warm-up; only samples taken between mark_begin() and
    mark_end() are summarised."""

    def sample_now(self):
        if self.ok:
            try:
                mhz = float(self.nv.nvmlDeviceGetClockInfo(self.h, self.nv.NVML_CLOCK_SM))
                self.samples.append((time.perf_counter(), mhz, self._reasons()))
            except Exception:
                pass

    def __init__(self, index):
        super().__init__(daemon=True)
        self.index, self.samples, self.stop_flag = index, [], False
        self.period = 0.2                 # the recipe's 200 ms; NVML queries can stall GPU work (see class doc)
        self.t0 = self.t1 = None
        self.ok = False
        try:
            import pynvml
            self.nv = pynvml
            pynvml.nvmlInit()
            # NVML enumerates physical devices; honour CUDA_VISIBLE_DEVICES when it is a plain index list
            vis = os.environ.get("CUDA_VISIBLE_DEVICES")
            phys = index
            if vis:
                try:
                    phys = int(vis.split(",")[index])
                except (ValueError, IndexError):
                    phys = index
            self.h = pynvml.nvmlDeviceGetHandleByIndex(phys)
            self.max_mhz = float(pynvml.nvmlDeviceGetMaxClockInfo(self.h, pynvml.NVML_CLOCK_SM))
            self.ok = True
        except Exception:
            self.ok = False

    def _reasons(self):
        nv = self.nv
        try:
            bits = nv.nvmlDeviceGetCurrentClocksEventReasons(self.h)
        except Exception:
            bits = nv.nvmlDeviceGetCurrentClocksThrottleReasons(self.h)
        names = []
        for name, attr in (("hw_slowdown", "nvmlClocksThrottleReasonHwSlowdown"),
                           ("hw_thermal_slowdown", "nvmlClocksThrottleReasonHwThermalSlowdown"),
                           ("sw_thermal_slowdown", "nvmlClocksThrottleReasonSwThermalSlowdown"),
                           ("sw_power_cap", "nvmlClocksThrottleReasonSwPowerCap")):
            if bits & getattr(nv, attr, 0):
                names.append(name)
        return names

    def run(self):
        if not self.ok:
            return
        while not self.stop_flag:
            try:
                mhz = float(self.nv.nvmlDeviceGetClockInfo(self.h, self.nv.NVML_CLOCK_SM))
                self.samples.append((time.perf_counter(), mhz, self._reasons()))
            except Exception:
                pass
            time.sleep(self.period)

    def mark_begin(self):
        self.t0 = time.perf_counter()

    def mark_end(self):
        self.t1 = time.perf_counter()

    def finish(self):
        self.stop_flag = True
        if self.is_alive():
            self.join(timeout=1.0)          # no stray sample may land in a later timed region
        inside = [s for s in self.samples if self.t0 is not None and self.t0 <= s[0] <= (self.t1 or s[0])]
        if not inside:      # region shorter than one polling period: take the nearest samples
            inside = self.samples[-2:]
        sm = [s[1] for s in inside]
        reasons = sorted({r for s in inside for r in s[2]})
        return {"sm_mhz": statistics.median(sm) if sm else None, "sm_max_mhz": self.max_mhz if self.ok else None,
                "reasons": reasons, "samples": len(sm), "source": "nvml" if self.ok else "unavailable"}


# ---------------------------------------------------------------------------------- reference arm
def oracle_modules(kind="combine1"):
    """The CPU arm's weights: shapes from the dump of the REFERENCE modules' own state_dict
    (tests/golden/state_dict_keys.json) - nothing of the product (modules, kernels, library) is on this path."""
    from oracle import cfp_oracle as O
    with open(os.path.join(os.path.dirname(os.path.abspath(__file__)), "tests", "golden", "state_dict_keys.json")) as fh:
        keys = json.load(fh)
    sds = {"hist_encoder": synth.synthetic_state_dict(keys["hist_encoder"], 0)}
    for lv, name in ((3, "cross_atten3"), (2, "cross_atten2"), (1, "cross_atten1")):
        sds[name] = synth.synthetic_state_dict(keys[f"fusion_{kind}_L{lv}"], lv)
    return O, sds


def time_cpu_frames(n_frames, steps, warmup, seed=1, geometry=GEOMETRY, layers=synth.COMBINE1_LAYERS):
    """Time the oracle port (fp32, all host threads) on `n_frames`-frame batches."""
    O, sds = oracle_modules("combine1" if "combine1" in layers else "baseline")
    torch.set_num_threads(os.cpu_count() or 1)
    inp = synth.make_inputs(geometry, n_frames, seed=seed)
    xs = [inp["x3"], inp["x2"], inp["x1"]]
    times = []
    with torch.no_grad():
        for i in range(warmup + steps):
            torch.manual_seed(2)
            t0 = time.perf_counter()
            O.fusion_path(sds, layers, xs, inp["hist_data"], inp["mask"], inp["patch_info"])
            dt = time.perf_counter() - t0
            if i >= warmup:
                times.append(dt)
    return times


def run_reference(a):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    cores = os.cpu_count() or 1
    probe = time_cpu_frames(1, 1, 1)[0]
    budget_s = 90.0
    n = max(1, min(64, int(budget_s / ((a.steps + a.warmup) * max(probe, 1e-3)))))
    times = time_cpu_frames(n, a.steps, a.warmup)
    total = sum(times)
    fps = n * a.steps / total
    sample = f"{n} frames/step x {a.steps} steps (+{a.warmup} warm-up), fp32, torch CPU ops, {cores} threads"
    line = {
        "impl": "reference", "metric": METRIC, "value": fps, "unit": "frames/s", "n_gpus": a.gpus,
        "steps": a.steps, "warmup": a.warmup, "ms_per_step": 1e3 * total / a.steps, "higher_is_better": True,
        "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": workload_config(a, per_gpu_batch=n),
        "cpu_baseline": {"value": fps, "unit": "frames/s", "cores": cores, "kind": "port", "sample": sample},
        "e2e": {"value": fps, "unit": "frames/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
    }
    print(json.dumps(line), flush=True)


def workload_config(a, per_gpu_batch):
    return {"workload": "CFPNet combine1 fusion path (hist encoder + cross_atten3/2/1), 416x544, 8x8 zones of 48 px, "
                        f"{per_gpu_batch} frames per GPU, batch-sharded (BASELINE.json configs[2])",
            "layers": list(synth.COMBINE1_LAYERS), "per_gpu_batch": per_gpu_batch, "global_batch": per_gpu_batch * a.gpus,
            "l2_policy": "inputs rotate over 3 distinct batches + workspace > 126 MB L2 between reuse",
            "launch_mode": "CUDA-graph replay per step (FusionPath.make_graphed; positional-encoding crops drawn per replay)"
                           if os.environ.get("CFP_GRAPH", "1") != "0" else "eager launches",
            "levels": "sequential (one stream)" if os.environ.get("CFP_SEQUENTIAL_LEVELS") else
                      "the three levels on three streams (valid for the synthetic harness, whose level inputs are independent; "
                      "inside the reference decoder the levels are serially dependent - see drop_in_sequential)",
            "micro_batches": os.environ.get("CFP_MICRO", "default")}


# ---------------------------------------------------------------------------------- product arm
def run_cfp(a):
    import torch.distributed as dist
    from cfpnet_b200 import FusionPath, _lib, shard
    from cfpnet_b200.build import build

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py --impl cfp needs a CUDA device: the fusion path has no CPU fallback")
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)
    build()
    dtype = {"bf16": torch.bfloat16, "f32": torch.float32}[a.dtype]
    B = a.batch
    host_binding = bind_host_to_gpu(local) if not os.environ.get("CFP_BENCH_NO_BIND") else "off (CFP_BENCH_NO_BIND)"

    path = FusionPath(synth.COMBINE1_LAYERS)
    path.hist_encoder.load_state_dict(synth.synthetic_state_dict(
        {k: v.shape for k, v in path.hist_encoder.state_dict().items()}, 0))
    for lv, name in ((3, "cross_atten3"), (2, "cross_atten2"), (1, "cross_atten1")):
        m = getattr(path, name)
        m.load_state_dict(synth.synthetic_state_dict({k: v.shape for k, v in m.state_dict().items()}, lv))
    path = path.to(dev).eval().set_dtype(dtype)

    # three distinct input batches per rank (rotated so consecutive steps never reuse L2 contents)
    NSETS = 3
    host_sets, dev_sets = [], []
    for s in range(NSETS):
        inp = synth.make_inputs(GEOMETRY, B, seed=100 + rank * NSETS + s)
        h = {"x3": inp["x3"].to(dtype).pin_memory(), "x2": inp["x2"].to(dtype).pin_memory(),
             "x1": inp["x1"].to(dtype).pin_memory(), "hist_data": inp["hist_data"].pin_memory(),
             "mask": inp["mask"].pin_memory()}
        host_sets.append(h)
        dev_sets.append({k: v.to(dev) for k, v in h.items()})
        patch_info = inp["patch_info"]
    h2d = sum(v.numel() * v.element_size() for v in host_sets[0].values())

    # CUDA-graph replay of the forward (one graph per rotating input set, the set's tensors are the captured inputs; the
    # positional-encoding crops are drawn per replay and read from device memory): CFP_GRAPH=0 runs eager launches
    use_graph = os.environ.get("CFP_GRAPH", "1") != "0"
    graphs = []
    if use_graph:
        with torch.no_grad():
            for d in dev_sets:
                graphs.append(path.make_graphed(d["x3"], d["x2"], d["x1"], d["hist_data"], d["mask"], patch_info, copy_inputs=False))
    launches_per_forward = [0]

    def step(i):
        d = dev_sets[i % NSETS]
        shard.seed_posenc(i)                # same positional-encoding crop on every rank
        if use_graph:
            return graphs[i % NSETS]()
        return path(d["x3"], d["x2"], d["x1"], d["hist_data"], d["mask"], patch_info)

    def barrier():
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
            torch.cuda.synchronize()

    def max_over_ranks(ms):
        if world == 1:
            return ms
        t = torch.tensor([ms], device=dev, dtype=torch.float64)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item())

    sampler = ClockSampler(local) if rank == 0 and not os.environ.get("CFP_BENCH_NO_SAMPLER") else None
    sampler_t = time.perf_counter()
    if sampler:
        sampler.start()
    with torch.no_grad():
        for i in range(a.warmup):
            outs = step(i)
        d2h = sum(o.numel() * o.element_size() for o in outs)
        barrier()
        if sampler:                         # first NVML samples in before timing (rank 0 only)
            while not sampler.samples and sampler.is_alive() and time.perf_counter() - sampler_t < 5.0:
                time.sleep(0.05)
        for i in range(2):                  # every rank: same sequence of steps and collectives
            step(i)
        barrier()
        # ---- device-resident throughput ("value")
        if sampler:
            sampler.mark_begin()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        marks = [torch.cuda.Event(enable_timing=True) for _ in range(a.steps)]
        attempts = []
        for attempt in range(2):
            n0 = _lib.launch_count()
            ms0 = torch.cuda.memory_stats(dev)
            e0.record()
            for i in range(a.steps):
                outs = step(i)
                marks[i].record()           # per-step marks (diagnostic)
                if sampler and i == a.steps // 2:
                    sampler.sample_now()    # one clock sample while the GPU is busy with the queued steps
            e1.record()
            barrier()
            step_ms = [(e0 if i == 0 else marks[i - 1]).elapsed_time(marks[i]) for i in range(a.steps)]
            launches = _lib.launch_count() - n0
            if use_graph:                   # replays do not pass through the library's launch counter: one eager forward does
                n1 = _lib.launch_count()
                path(dev_sets[0]["x3"], dev_sets[0]["x2"], dev_sets[0]["x1"], dev_sets[0]["hist_data"], dev_sets[0]["mask"], patch_info)
                torch.cuda.synchronize()
                launches = (_lib.launch_count() - n1) * a.steps
            ms_total = max_over_ranks(e0.elapsed_time(e1))
            attempts.append(ms_total)
            ms1 = torch.cuda.memory_stats(dev)
            alloc_delta = {k: ms1.get(k, 0) - ms0.get(k, 0) for k in ("num_device_alloc", "num_device_free", "num_alloc_retries", "num_sync_all_streams")}
            # a clock query occasionally stalls the GPU for 50-100 ms: if one step took > 1.6x the median on any
            # rank, the K steps are timed once more (both attempts are reported)
            perturbed = max_over_ranks(1.0 if max(step_ms) > 1.6 * statistics.median(step_ms) else 0.0)
            if not perturbed:
                break
        # the last timed step's result, copied before the replays below can overwrite a graph's output buffers
        last_outs = [o.clone() for o in outs] if a.dump_outputs and rank == 0 else None
        if sampler:
            sampler.mark_end()
        clocks = sampler.finish() if sampler else None

        # ---- the same K steps with the three levels on ONE stream: what a drop-in into the reference's decoder can use
        # (there x_d2 depends on the fused x_d3, decoder.py:109-121, so the levels cannot overlap)
        seq_ms = None
        if path.concurrent_levels:
            path.concurrent_levels = False
            seq_graphs = []
            if use_graph:
                for d in dev_sets:
                    seq_graphs.append(path.make_graphed(d["x3"], d["x2"], d["x1"], d["hist_data"], d["mask"], patch_info, copy_inputs=False))

            def seq_step(i):
                d = dev_sets[i % NSETS]
                shard.seed_posenc(i)
                return seq_graphs[i % NSETS]() if use_graph else path(d["x3"], d["x2"], d["x1"], d["hist_data"], d["mask"], patch_info)
            for i in range(3):
                seq_step(i)
            barrier()
            e0.record()
            for i in range(a.steps):
                seq_step(i)
            e1.record()
            barrier()
            seq_ms = max_over_ranks(e0.elapsed_time(e1))
            del seq_graphs
            path.concurrent_levels = True

        # ---- end-to-end through the public host-buffer API ("e2e"): pinned host inputs in, pinned host
        # outputs back, every step; FusionPath.stream_host overlaps the copies of neighbouring steps
        # with compute on separate streams (each step still pays its own H2D + D2H).
        def host_batches(n):
            for i in range(n):
                yield host_sets[i % NSETS]

        for _ in path.stream_host(host_batches(max(a.warmup, 3)), patch_info, dev, seeds=range(2, 2 + max(a.warmup, 3)), graph=use_graph):
            pass
        e2e_attempts = []
        for attempt in range(2):
            barrier()
            t_wall = time.perf_counter()
            e0.record()
            stamps = []
            for _idx, _outs in path.stream_host(host_batches(a.steps), patch_info, dev, seeds=range(2, 2 + a.steps), graph=use_graph):
                stamps.append(time.perf_counter())
            e1.record()
            barrier()
            t_wall = time.perf_counter() - t_wall
            assert len(stamps) == a.steps
            # the last D2H completes on a side stream: take the larger of the device-event and wall-clock spans
            ms_e2e = max_over_ranks(max(e0.elapsed_time(e1), t_wall * 1e3))
            e2e_attempts.append(ms_e2e)
            if os.environ.get("CFP_BENCH_DEBUG"):
                t_start = stamps[0] - (time.perf_counter() - t_wall) if False else None
                print("e2e debug: wall %.1f ms, event %.1f ms, gaps %s" % (
                    t_wall * 1e3, e0.elapsed_time(e1), [round((b - a_) * 1e3, 1) for a_, b in zip(stamps, stamps[1:])]),
                    file=sys.stderr, flush=True)
            gaps = [b - a_ for a_, b in zip(stamps, stamps[1:])]
            # same rule as above: a sporadic stall in the region (an outlier gap between results, or a start-up
            # hiccup of the first host->device copies that makes the span exceed (K+1) median gaps by > 12 %)
            # -> time the K steps once more; both attempts are reported
            med = statistics.median(gaps) if gaps else 0.0
            slow_start = len(gaps) >= 3 and t_wall > 1.12 * (a.steps + 1.0) * med
            perturbed = max_over_ranks(1.0 if len(gaps) >= 3 and (max(gaps) > 1.6 * med + 1e-3 or slow_start) else 0.0)
            if not perturbed:
                break

        # ---- what the host link gives this run: the e2e loop's copies alone (no compute), all ranks at once
        link_s = max_over_ranks(probe_host_link(dev, h2d, d2h, barrier) * 1e3) * 1e-3

        # ---- per-kernel breakdown with CUDA events on the launch stream (roofline)
        prof = None
        if rank == 0:
            torch.cuda.synchronize()
            path.concurrent_levels = False      # one stream: the gap between events is one kernel's time
            _lib.profile_start()
            for i in range(a.steps):            # eager launches (the profiler records an event per launch)
                d = dev_sets[i % NSETS]
                shard.seed_posenc(i)
                path(d["x3"], d["x2"], d["x1"], d["hist_data"], d["mask"], patch_info)
            prof = _lib.profile_stop()
            path.concurrent_levels = not bool(os.environ.get("CFP_SEQUENTIAL_LEVELS"))
    if world > 1:
        dist.barrier()

    if rank != 0:
        if world > 1:
            dist.destroy_process_group()
        return
    peaks = load_peaks()
    frames = B * world * a.steps
    value = frames / (ms_total * 1e-3)
    es = 2 if dtype == torch.bfloat16 else 4
    line = {
        "metric": METRIC, "value": value, "unit": "frames/s", "n_gpus": world, "steps": a.steps, "warmup": a.warmup,
        "ms_per_step": ms_total / a.steps, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
        "dtype": a.dtype, "data": "synthetic", "config": workload_config(a, B),
        "e2e": {"value": frames / (ms_e2e * 1e-3), "unit": "frames/s", "h2d_bytes_per_step": h2d,
                "d2h_bytes_per_step": d2h,
                # the copies of one step alone, every rank at once (slowest rank): the host link's ceiling for this metric
                "host_link": {"copy_only_ms_per_step": link_s * 1e3, "ceiling_frames_per_s": B * world / link_s,
                              "GBps_each_way_per_gpu": [h2d / link_s / 1e9, d2h / link_s / 1e9],
                              "e2e_frac_of_ceiling": (frames / (ms_e2e * 1e-3)) / (B * world / link_s),
                              "host_binding": host_binding}},
        "gpu_launches": int(launches), "clocks": clocks,
        "step_ms": {"min": min(step_ms), "median": statistics.median(step_ms), "max": max(step_ms)},
        "timed_attempts_ms": attempts, "e2e_attempts_ms": e2e_attempts, "allocator_in_timed_region": alloc_delta,
    }
    if seq_ms:
        line["drop_in_sequential"] = {"ms_per_step": seq_ms / a.steps, "value": frames / (seq_ms * 1e-3), "unit": "frames/s",
                                      "note": "levels L3, L2, L1 on one stream, as inside the reference decoder (decoder.py:109-121)"}
    # whole-path roofline view (algorithmic bytes / dense flops per frame x measured frames/s)
    per_gpu_fps = value / world
    line["path"] = {"algorithmic_GBps": ELEMS_PER_FRAME * es * per_gpu_fps / 1e9,
                    "dense_TFLOPs": DENSE_FLOP_PER_FRAME * per_gpu_fps / 1e12,
                    "hbm_peak_GBps": peaks["hbm_gbs"], "bf16_peak_TFLOPs": peaks["bf16_tflops_sustained"]}
    if prof:
        line["roofline"], line["kernels"] = roofline_from_profile(prof, a.steps, B, es, peaks)
    if not a.no_cpu and world == 1:          # the CPU baseline is reported at N = 1 only (rank 0's host cores)
        cores = os.cpu_count() or 1
        t = time_cpu_frames(1, 10, 3)
        med = statistics.median(t)
        line["cpu_baseline"] = {"value": 1.0 / med, "unit": "frames/s", "cores": cores, "kind": "port",
                                "sample": "1 frame/step, 3 warm-up + 10 timed, median, fp32 torch CPU ops on all host threads"}
    if last_outs:
        share = dump_outputs(a.dump_outputs, list(zip(("fused3", "fused2", "fused1"), last_outs)))
        print(f"--dump-outputs: step {a.steps - 1} written to {a.dump_outputs} ({share:.3f} of the elements)", file=sys.stderr)
    print(json.dumps(line), flush=True)
    if world > 1:
        dist.destroy_process_group()


# Algorithmic work per LAUNCH of each kernel at G416 (derivations: DESIGN.md §4, SURVEY.md §8d).
#   flops  = useful multiply-adds x 2 of the op as the reference defines it (no padding / Toeplitz zeros)
#   bytes  = compulsory HBM traffic: every activation the op reads + writes once, weights amortised
LEVEL = {  # C: (N tokens, k, zone patch side p, window ws, inside Ni)
    32: dict(N=14144, k=31, p=12, ws=12, Ni=9216, H=104, W=136),
    64: dict(N=3536, k=15, p=6, ws=9, Ni=2304, H=52, W=68),
    128: dict(N=884, k=7, p=3, ws=6, Ni=576, H=26, W=34),
}


def _decoder_work():
    """Per-frame, per-LAUNCH averages (useful flops, algorithmic bf16 bytes) of the decoder / head kernels at 416x544:
    every conv of decoder.py:70-80 + DepthRegression.conv3x3 grouped by its output width (= the kernel instantiation)."""
    px = {2: 208 * 272, 4: 104 * 136, 8: 52 * 68, 16: 26 * 34, 32: 13 * 17}
    convs = [  # (pixels, cin, cout, taps)
        (px[32], 232, 256, 1), (px[16], 392, 256, 9), (px[16], 256, 256, 9), (px[16], 256, 128, 1),
        (px[8], 312, 128, 9), (px[8], 128, 128, 9), (px[8], 128, 64, 1),
        (px[4], 168, 64, 9), (px[4], 64, 64, 9), (px[4], 64, 32, 1),
        (px[2], 80, 32, 9), (px[2], 32, 32, 9), (px[2], 32, 128, 9), (px[2], 128, 128, 9)]
    work = {}
    for cout in (256, 128, 64, 32):
        sel = [c for c in convs if c[2] == cout]
        work[f"conv_gen_tc<{cout}>"] = (sum(2.0 * p * ci * co * t for p, ci, co, t in sel) / len(sel),
                                        sum(2.0 * p * (ci + co) for p, ci, co, t in sel) / len(sel))
    ups = [(px[32], 232, 0), (px[16], 392, 256), (px[8], 312, 256), (px[4], 168, 128), (px[2], 80, 64)]
    work["upsample_concat"] = (0.0, sum(2.0 * p * c + 2.0 * (p // 4) * lo for p, c, lo in ups) / len(ups))
    work["head_expect_tc<256>"] = (2.0 * px[2] * 128 * 256, 2.0 * px[2] * 128 + 4.0 * px[2])
    work["channel_mean"] = (0.0, 2.0 * px[2] * 128)
    work["copy_channels"] = (0.0, sum(4.0 * p * c for p, c in ((px[16], 128), (px[8], 64), (px[4], 32))) / 3)
    work["posenc_tokens_nhwc"] = work["copy_channels"]
    return work


DECODER_WORK = _decoder_work()


def kernel_work(name, B, es):
    import re
    # kernels launched once per level under one name: average per launch over the levels that use them
    if name == "layout_kernel":          # pos-enc + NCHW -> tokens and tokens -> NCHW, each level: read + write the map
        return dict(flops=0.0, bytes=sum(2.0 * g["N"] * C * es * B for C, g in LEVEL.items()) / 3, bound="hbm")
    if name == "dw_plane_pack":          # levels with k >= 15: read the token map, write the planes (>= the same size)
        return dict(flops=0.0, bytes=sum(2.0 * LEVEL[C]["N"] * C * es * B for C in (32, 64)) / 2, bound="hbm")
    if name.startswith("hist_encoder"):  # 1024 samples per frame: 4 B in, (32+64+128) elements out; 109 MFLOP per frame
        return dict(flops=109e6 * B, bytes=1024.0 * B * (4 + 224 * es), bound="tensor" if name.endswith("_tc") else "fma")
    if name in DECODER_WORK:
        f, by = DECODER_WORK[name]
        return dict(flops=f * B, bytes=by * B * es / 2.0, bound="tensor" if f > 0 else "hbm")
    m = re.search(r"(\d+)>$", name)
    if not m:
        return None
    v = int(m.group(1))
    if name.startswith(("dwconv", "tr_dwconv_wgrad")):  # dwconv<k> / dwconv_tc<k> / weight gradient: v is the kernel size
        C = {31: 32, 15: 64, 7: 128}[v]
        g = LEVEL[C]
        return dict(flops=2.0 * g["N"] * C * v * v * B, bytes=2.0 * g["N"] * C * es * B, bound="tensor" if "_tc" in name else "fma")
    C = v
    g = LEVEL[C]
    N, Ni, p, ws = g["N"], g["Ni"], g["p"], g["ws"]
    No = N - Ni
    nwin = -(-g["H"] // ws) * -(-g["W"] // ws)
    Ns = (g["H"] // ws) * (g["W"] // ws)
    chain = 16.0 * C * C                                # q, merge, mlp0 (2Cx2C), mlp2 (2C->C): flops per query row
    rows = {"hist2image": 64 * p * p, "lsa": nwin * ws * ws, "gsa": N, "dapm": No}
    src = {"hist2image": 64 * 16, "lsa": nwin * ws * ws, "gsa": Ns, "dapm": Ni}
    heads = {"hist2image": 4, "lsa": 8, "gsa": 8, "dapm": 4}
    for kind in rows:
        if f"<{kind}," in name:
            dh = C // heads[kind]
            if name.startswith("loftr_query"):
                return dict(flops=(chain + 2.0 * C * dh) * rows[kind] * B, bytes=2.0 * rows[kind] * C * es * B, bound="tensor")
            if name.startswith("attn_query"):
                return dict(flops=(2.0 * C * C + 2.0 * C * dh) * rows[kind] * B, bytes=2.0 * rows[kind] * C * es * B, bound="tensor")
            if name.startswith("kv_state"):
                return dict(flops=(4.0 * C * C + 2.0 * C * dh) * src[kind] * B, bytes=src[kind] * C * es * B, bound="tensor")
    if name.startswith("lkpm_mlp"):
        return dict(flops=16.0 * N * C * C * B, bytes=3.0 * N * C * es * B, bound="tensor")
    if name.startswith("conv3x3"):
        cin = 2 * C if "2C->C" in name else C
        return dict(flops=2.0 * N * cin * 9 * C * B, bytes=(cin + C + (C if cin == C else 0)) * N * es * B, bound="tensor")
    if name.startswith("sr_conv"):
        return dict(flops=2.0 * Ns * ws * ws * C * C * B, bytes=N * C * es * B, bound="tensor")
    return None


# dram bytes (read + write) per launch from the committed ncu capture of this workload (tools/ncu_traffic.py ->
# profiles/ncu_traffic.json: {bench kernel name: bytes per launch}); null when the kernel was not captured
def load_ncu_traffic():
    try:
        with open(os.path.join(ROOT, "profiles", "ncu_traffic.json")) as fh:
            return {k: float(v) for k, v in json.load(fh).get("bytes_per_launch", {}).items()}
    except Exception:
        return {}


def roofline_of(name, avg_s, B, es, peaks):
    """Roofline of one kernel: the bound is whichever of (algorithmic bytes / HBM peak) and (useful flops / tensor
    peak) takes longer; `achieved` is the algorithmic quantity of that bound / measured launch time."""
    w = kernel_work(name, B, es)
    if not w:
        return dict(bound="hbm", achieved=None, peak=peaks["hbm_gbs"], unit="GB/s", frac=None)
    t_hbm = w["bytes"] / (peaks["hbm_gbs"] * 1e9)
    t_tc = w["flops"] / (peaks["bf16_tflops_sustained"] * 1e12) if w["bound"] == "tensor" else 0.0
    gbps, tflops = w["bytes"] / avg_s / 1e9, w["flops"] / avg_s / 1e12
    if t_tc >= t_hbm:
        return dict(bound="tensor", achieved=tflops, peak=peaks["bf16_tflops_sustained"], unit="TFLOP/s",
                    frac=tflops / peaks["bf16_tflops_sustained"],
                    note="useful flops of the op (no padding / Toeplitz zeros) / CUDA-event time; peak = sustained cuBLAS bf16",
                    other={"hbm_GBps": gbps, "hbm_frac": gbps / peaks["hbm_gbs"]})
    return dict(bound="hbm", achieved=gbps, peak=peaks["hbm_gbs"], unit="GB/s", frac=gbps / peaks["hbm_gbs"],
                note="algorithmic bytes (activations read + written once) / CUDA-event time; peak = measured copy bandwidth",
                other={"TFLOPs": tflops, "tensor_frac": tflops / peaks["bf16_tflops_sustained"]} if w["bound"] == "tensor" else
                      {"fp32_TFLOPs": tflops})


def roofline_from_profile(prof, steps, B, es, peaks):
    total_ms = sum(v[1] for v in prof.values())
    traffic = load_ncu_traffic()
    kernels = {}
    for k, v in sorted(prof.items(), key=lambda kv: -kv[1][1]):
        rec = {"launches_per_step": v[0] / steps, "ms_per_step": v[1] / steps, "share": v[1] / total_ms if total_ms else None}
        w = kernel_work(k, B, es)
        if w:
            avg_s = v[1] / v[0] * 1e-3
            r = roofline_of(k, avg_s, B, es, peaks)
            rec["TFLOPs"] = w["flops"] / avg_s / 1e12
            rec["GBps"] = w["bytes"] / avg_s / 1e9
            rec["bound"], rec["roofline_frac"] = r["bound"], r["frac"]
        kernels[k] = rec
    name, (count, ms) = max(prof.items(), key=lambda kv: kv[1][1])
    avg_s = ms / count * 1e-3
    roof = {"kernel": name, "avg_launch_ms": avg_s * 1e3, "peak_source": peaks["source"], "traffic": traffic.get(name)}
    roof.update(roofline_of(name, avg_s, B, es, peaks))
    return roof, kernels


# ---------------------------------------------------------------------------------- other BASELINE.json configs
def run_aux(a):
    """The two single-GPU side configurations of BASELINE.json (not the headline line; SURVEY.md 8d):
      --workload baseline_b16   configs[1]: DELTAR-style layer list (hist2image image x2, no cross-zone propagation),
                                batch 16, 416x544 - frames/s, device-resident, K timed steps;
      --workload latency_480    configs[3]: combine1, ZJUL5-shaped 480x640 (8x8 zones of 56 px: the bilinear-resize
                                branch at 1/16), batch 1, evaluate_time.py's protocol (evaluate_time.py:56-82): 100
                                warm-up forwards, 500 timed ones each bracketed by a device synchronise, trimmed mean
                                sum(sorted(dt)[1:-2]) / (n - 3) in ms."""
    from cfpnet_b200 import FusionPath, shard
    from cfpnet_b200.build import build
    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA device: the fusion path has no CPU fallback")
    torch.cuda.set_device(0)
    dev = torch.device("cuda", 0)
    build()
    dtype = {"bf16": torch.bfloat16, "f32": torch.float32}[a.dtype]
    latency = a.workload == "latency_480"
    layers = synth.COMBINE1_LAYERS if latency else ("hist2image", "image", "hist2image", "image")
    geom, B = ("G480", 1) if latency else ("G416", 16)
    path = FusionPath(layers)
    path.hist_encoder.load_state_dict(synth.synthetic_state_dict({k: v.shape for k, v in path.hist_encoder.state_dict().items()}, 0))
    for lv, name in ((3, "cross_atten3"), (2, "cross_atten2"), (1, "cross_atten1")):
        m = getattr(path, name)
        m.load_state_dict(synth.synthetic_state_dict({k: v.shape for k, v in m.state_dict().items()}, lv))
    path = path.to(dev).eval().set_dtype(dtype)
    sets = []
    for s_ in range(3):
        inp = synth.make_inputs(geom, B, seed=100 + s_)
        sets.append({k: (inp[k].to(dtype) if k.startswith("x") else inp[k]).to(dev) for k in ("x3", "x2", "x1", "hist_data", "mask")})
    patch_info = inp["patch_info"]

    def step(i):
        d = sets[i % 3]
        shard.seed_posenc(i)
        return path(d["x3"], d["x2"], d["x1"], d["hist_data"], d["mask"], patch_info)

    with torch.no_grad():
        if latency:
            for i in range(100):
                step(i)
            dts = []
            for i in range(500):
                torch.cuda.synchronize()
                t0 = time.perf_counter()
                step(i)
                torch.cuda.synchronize()
                dts.append(time.perf_counter() - t0)
            ms_eager = 1e3 * sum(sorted(dts)[1:-2]) / (len(dts) - 3)
            # the same protocol through a CUDA-graph replay of the forward (the maps fill the positional-encoding tables
            # at 480x640, so nothing random is frozen): removes the ~95 host-side launches per forward
            d0 = sets[0]
            run = path.make_graphed(d0["x3"], d0["x2"], d0["x1"], d0["hist_data"], d0["mask"], patch_info)
            for i in range(100):
                d = sets[i % 3]
                run(d["x3"], d["x2"], d["x1"], d["hist_data"], d["mask"])
            dts = []
            for i in range(500):
                d = sets[i % 3]
                torch.cuda.synchronize()
                t0 = time.perf_counter()
                run(d["x3"], d["x2"], d["x1"], d["hist_data"], d["mask"])
                torch.cuda.synchronize()
                dts.append(time.perf_counter() - t0)
            ms = 1e3 * sum(sorted(dts)[1:-2]) / (len(dts) - 3)
            line = {"metric": "CFP fusion path latency @480x640, 8x8 zones, batch 1 (evaluate_time.py protocol)", "value": ms,
                    "unit": "ms", "higher_is_better": False, "n_gpus": 1, "steps": 500, "warmup": 100, "ms_per_step": ms,
                    "dtype": a.dtype, "data": "synthetic", "vs_baseline": None,
                    "config": {"workload": "CFPNet combine1 fusion path, ZJUL5-shaped 480x640, 8x8 zones of 56 px, batch 1 "
                                           "(BASELINE.json configs[3]); hot path only (hist encoder + three TransformerFusion calls)",
                               "layers": list(layers), "median_ms": 1e3 * statistics.median(dts), "min_ms": 1e3 * min(dts),
                               "mode": "CUDA-graph replay (FusionPath.make_graphed)", "eager_ms": ms_eager}}
        else:
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)

            def timed(fn):
                for i in range(max(a.warmup, 3)):
                    fn(i)
                torch.cuda.synchronize()
                e0.record()
                for i in range(a.steps):
                    fn(i)
                e1.record()
                torch.cuda.synchronize()
                return e0.elapsed_time(e1) / a.steps

            ms_eager = timed(step)            # ~90 host-side launches per step: bound by the launching thread, +-20 % run to run
            d0 = sets[0]
            run = path.make_graphed(d0["x3"], d0["x2"], d0["x1"], d0["hist_data"], d0["mask"], patch_info)

            def replay(i):                    # positional-encoding crops drawn per replay, read from device memory
                d = sets[i % 3]
                shard.seed_posenc(i)
                return run(d["x3"], d["x2"], d["x1"], d["hist_data"], d["mask"])

            ms = timed(replay)
            line = {"metric": "DELTAR-style fusion (no cross-zone propagation) frames/s @416x544, 8x8 zones, batch 16", "value": B * 1e3 / ms,
                    "unit": "frames/s", "higher_is_better": True, "n_gpus": 1, "steps": a.steps, "warmup": max(a.warmup, 3),
                    "ms_per_step": ms, "dtype": a.dtype, "data": "synthetic", "vs_baseline": None,
                    "config": {"workload": "DELTAR-style baseline layer list (..._10x config), 416x544, batch 16, 1 GPU "
                                           "(BASELINE.json configs[1])", "layers": list(layers), "per_gpu_batch": B,
                               "mode": "CUDA-graph replay (FusionPath.make_graphed)", "eager_ms": ms_eager}}
        # per-kernel breakdown (CUDA events on the launch stream, levels on one stream, eager launches) and its roofline
        from cfpnet_b200 import _lib
        n_prof = 20 if latency else a.steps
        torch.cuda.synchronize()
        path.concurrent_levels = False
        _lib.profile_start()
        for i in range(n_prof):
            step(i)
        prof = _lib.profile_stop()
    peaks = load_peaks()
    es = 2 if dtype == torch.bfloat16 else 4
    roof, kernels = roofline_from_profile(prof, n_prof, B, es, peaks)
    if latency:
        # kernel_work() holds the algorithmic bytes / flops of the 416x544 shapes: at 480x640 only the time shares are reported
        roof = {"kernel": roof["kernel"], "avg_launch_ms": roof["avg_launch_ms"], "bound": roof["bound"], "achieved": None,
                "peak": roof["peak"], "unit": roof["unit"], "frac": None, "traffic": None,
                "note": "batch-1 launches are latency-bound single waves; per-kernel time shares in `kernels`"}
        kernels = {k: {kk: vv for kk, vv in v.items() if kk in ("launches_per_step", "ms_per_step", "share")} for k, v in kernels.items()}
    line["roofline"], line["kernels"] = roof, kernels
    if not a.no_cpu:
        cores = os.cpu_count() or 1
        t = time_cpu_frames(1, 6, 2, geometry=geom, layers=tuple(layers))
        med = statistics.median(t)
        line["cpu_baseline"] = ({"value": med * 1e3, "unit": "ms"} if latency else {"value": 1.0 / med, "unit": "frames/s"})
        line["cpu_baseline"].update({"cores": cores, "kind": "port",
                                     "sample": "1 frame/step, 2 warm-up + 6 timed, median, fp32 torch CPU ops on all host threads"})
    print(json.dumps(line), flush=True)


# ---------------------------------------------------------------------------------- training step (BASELINE.json configs[4])
def run_train(a):
    """--workload train_b32: the training step of the path (BASELINE.json configs[4]; reference train.py:96-135) - the
    histogram encoder and the three TransformerFusion calls (hist2image, DAPM, LKPM, LSA, GSA; the encoder's outputs feed
    the fusion calls, so the backward runs through both) in .train() mode, 32 frames per GPU, fp32 as the reference trains:

        zero_grad -> forward (BatchNorm on per-replica batch statistics) -> backward -> NCCL all-reduce of the flat
        gradient bucket -> clip_grad_norm_(0.1) -> AdamW

    Every op of the forward and of the backward is a libcfp kernel (cfp_tr_*; cfpnet_b200/train.py sequences them).
    `value` = frames/s of that step with inputs resident in HBM; `e2e` = the same with the step's inputs copied from
    pinned host memory and the gradient norm read back.  `collective` reports the all-reduce inside the step (bytes,
    CUDA-event time, share of the step, bus bandwidth)."""
    import torch.distributed as dist
    import cfpnet_b200
    from cfpnet_b200 import _lib
    from cfpnet_b200.build import build
    from cfpnet_b200.config import args as cfg
    from cfpnet_b200.train import FlatTrainer

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA device: the path has no CPU fallback")
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)
    build()
    B = a.batch
    enc = cfpnet_b200.HistogramEncoder()
    enc.load_state_dict(synth.synthetic_state_dict({k: v.shape for k, v in enc.state_dict().items()}, 0))
    fusion = {}
    saved_layers = list(cfg.attention_layer)
    cfg.attention_layer = list(synth.COMBINE1_LAYERS)
    try:
        for lv in (3, 2, 1):
            C, _, max_res, k = synth.LEVELS[lv]
            m = cfpnet_b200.TransformerFusion(C, list(max_res), large_kernel=k, patch_size=640 // max_res[1])
            m.load_state_dict(synth.synthetic_state_dict({kk: v.shape for kk, v in m.state_dict().items()}, lv))
            fusion[lv] = m
    finally:
        cfg.attention_layer = saved_layers
    mods = [enc.to(dev).train()] + [fusion[lv].to(dev).train() for lv in (3, 2, 1)]
    trainer = FlatTrainer(mods, lr=1e-4, weight_decay=0.1, max_norm=0.1)

    NSETS = 3
    host_sets, dev_sets = [], []
    for s_ in range(NSETS):
        inp = synth.make_inputs(GEOMETRY, B, seed=300 + rank * NSETS + s_)
        h = {"hist": inp["hist_data"].unsqueeze(-1).contiguous().pin_memory(), "mask": inp["mask"].to(torch.uint8).contiguous().pin_memory()}
        for lv in (3, 2, 1):
            h[f"x{lv}"] = inp[f"x{lv}"].float().contiguous().pin_memory()
        host_sets.append(h)
        dev_sets.append({k: v.to(dev) for k, v in h.items()})
        patch_info, rect_data = inp["patch_info"], inp["rect_data"]      # the same zone layout in every set
    h2d = sum(v.numel() * v.element_size() for v in host_sets[0].values())
    g = torch.Generator().manual_seed(11 + rank)
    # cotangents of the three fused maps (what the decoder behind them would send back), scaled like a mean loss
    cts = {}
    for lv in (3, 2, 1):
        x = host_sets[0][f"x{lv}"]
        cts[f"x{lv}"] = (torch.randn(x.shape, generator=g) / x.numel()).to(dev)

    ev_a = [torch.cuda.Event(enable_timing=True) for _ in range(2)]

    def step(d, timed_exchange=False):
        trainer.zero_grad()
        feats = dict(zip((32, 64, 128), enc(d["hist"])))   # differentiable: the fusion calls' feat1 gradients flow back into the encoder
        outs, grads = [], []
        for lv in (3, 2, 1):
            x = d[f"x{lv}"].requires_grad_(True)            # the image branch upstream needs dx: the full backward runs
            x.grad = None
            outs.append(fusion[lv](x, feats[synth.LEVELS[lv][0]], mask=d["mask"], patch_info=patch_info, rect_data=rect_data, rgb=None))
            grads.append(cts[f"x{lv}"])
        torch.autograd.backward(outs, grads)
        if trainer.flat_g is None:
            trainer.adopt()
        if timed_exchange:
            ev_a[0].record()
        trainer.exchange()
        if timed_exchange:
            ev_a[1].record()
        trainer.update()

    def barrier():
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
            torch.cuda.synchronize()

    def max_over_ranks(ms):
        if world == 1:
            return ms
        t = torch.tensor([ms], device=dev, dtype=torch.float64)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item())

    sampler = ClockSampler(local) if rank == 0 and not os.environ.get("CFP_BENCH_NO_SAMPLER") else None
    if sampler:
        sampler.start()
    for i in range(max(a.warmup, 3)):
        step(dev_sets[i % NSETS])
    barrier()
    if sampler:
        t_s = time.perf_counter()
        while not sampler.samples and sampler.is_alive() and time.perf_counter() - t_s < 5.0:
            time.sleep(0.05)
        sampler.mark_begin()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    n0 = _lib.launch_count()
    e0.record()
    for i in range(a.steps):
        step(dev_sets[i % NSETS])
        if sampler and i == a.steps // 2:
            sampler.sample_now()
    e1.record()
    barrier()
    launches = _lib.launch_count() - n0
    ms_total = max_over_ranks(e0.elapsed_time(e1))
    if sampler:
        sampler.mark_end()
    clocks = sampler.finish() if sampler else None

    # all-reduce inside the step, CUDA events on the launch stream (separate instrumented pass)
    ar_ms = []
    for i in range(a.steps):
        step(dev_sets[i % NSETS], timed_exchange=True)
        torch.cuda.synchronize()
        ar_ms.append(ev_a[0].elapsed_time(ev_a[1]))
    ar_med = max_over_ranks(statistics.median(ar_ms))
    # the same collective on a bucket of the complete path's gradient size (6.65 M parameters)
    full_ms = None
    if world > 1:
        big = torch.zeros(6_650_000, device=dev, dtype=torch.float32)
        for _ in range(5):
            dist.all_reduce(big)
        torch.cuda.synchronize()
        t_ = []
        for _ in range(20):
            ev_a[0].record()
            dist.all_reduce(big)
            ev_a[1].record()
            torch.cuda.synchronize()
            t_.append(ev_a[0].elapsed_time(ev_a[1]))
        full_ms = max_over_ranks(statistics.median(t_))

    # end to end: inputs from pinned host memory every step, the gradient norm read back
    side = torch.cuda.Stream(device=dev)
    norm_host = torch.zeros(1).pin_memory()

    def e2e_run(n):
        cur = torch.cuda.current_stream()
        staged = None
        for i in range(n + 1):
            nxt = None
            if i < n:
                with torch.cuda.stream(side):
                    nxt = {k: v.to(dev, non_blocking=True) for k, v in host_sets[i % NSETS].items()}
                    ev = torch.cuda.Event()
                    ev.record(side)
            if staged is not None:
                cur.wait_event(staged[1])
                step(staged[0])
                norm_host.copy_(trainer.sumsq[:1], non_blocking=True)
                for t in staged[0].values():
                    t.record_stream(cur)
            staged = (nxt, ev) if nxt is not None else None
        torch.cuda.synchronize()

    e2e_run(3)
    barrier()
    t_wall = time.perf_counter()
    e0.record()
    e2e_run(a.steps)
    e1.record()
    barrier()
    t_wall = time.perf_counter() - t_wall
    ms_e2e = max_over_ranks(max(e0.elapsed_time(e1), t_wall * 1e3))

    prof = None
    torch.cuda.synchronize()
    if rank == 0:
        _lib.profile_start()
    for i in range(a.steps):                # every rank: the step contains a collective
        step(dev_sets[i % NSETS])
    if rank == 0:
        prof = _lib.profile_stop()
    barrier()
    if rank != 0:
        if world > 1:
            dist.destroy_process_group()
        return
    peaks = load_peaks()
    frames = B * world * a.steps
    nparams = int(trainer.flat_g.numel())
    bus = lambda nbytes, ms: (2.0 * (world - 1) / world * nbytes / (ms * 1e-3) / 1e9) if world > 1 and ms else None   # noqa: E731
    line = {
        "metric": "CFP path training step (hist encoder + three TransformerFusion calls) frames/s @416x544, 8x8 zones", "value": frames / (ms_total * 1e-3),
        "unit": "frames/s", "n_gpus": world, "steps": a.steps, "warmup": max(a.warmup, 3), "ms_per_step": ms_total / a.steps,
        "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": {"workload": "training step of the path: HistogramEncoder + cross_atten3/2/1 (combine1 layer list) in .train() mode, "
                               f"forward + backward + all-reduce + clip + AdamW, fp32, {B} frames per GPU, 416x544 (BASELINE.json configs[4])",
                   "per_gpu_batch": B, "global_batch": B * world, "optimizer": "clip_grad_norm_(0.1) + AdamW on the flat bucket",
                   "l2_policy": "inputs rotate over 3 distinct batches; activations of a step (> 1 GB) exceed the 126 MB L2"},
        "e2e": {"value": frames / (ms_e2e * 1e-3), "unit": "frames/s", "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": 4},
        "gpu_launches": int(launches), "clocks": clocks,
        "collective": {"op": "NCCL all-reduce (sum) of one flat fp32 gradient bucket", "parameters": nparams, "bytes": nparams * 4,
                       "ms": ar_med, "share_of_step": ar_med / (ms_total / a.steps) if world > 1 else 0.0,
                       "busbw_GBps": bus(nparams * 4, ar_med),
                       "full_path_bucket": {"bytes": 6_650_000 * 4, "ms": full_ms, "busbw_GBps": bus(6_650_000 * 4, full_ms)}},
    }
    if prof:
        line["roofline"], line["kernels"] = roofline_from_profile(prof, a.steps, B, 4, peaks)
    print(json.dumps(line), flush=True)
    if world > 1:
        dist.destroy_process_group()



# ---------------------------------------------------------------------------------- decoder + fusion + head (SURVEY 8 f1 / f2)
def run_tail(a):
    """--workload tail_b16: everything of the reference model below the third-party image encoder - histogram encoder,
    Decoder (UpSampleBN blocks, 1x1 convs, the three TransformerFusion calls in their true serial order) and the
    adaptive-bins head - as libcfp kernels, bf16, channels-last: five encoder feature maps + zone histograms in, depth out.
    `value`: frames/s with the inputs resident in HBM; `e2e`: inputs from pinned host memory, depth maps read back."""
    import cfpnet_b200
    from cfpnet_b200 import _lib, decoder as D, shard
    from cfpnet_b200.build import build
    from cfpnet_b200.config import args as cargs
    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA device: the path has no CPU fallback")
    torch.cuda.set_device(0)
    dev = torch.device("cuda", 0)
    build()
    B = a.batch
    cargs.attention_layer = list(synth.COMBINE1_LAYERS)
    with open(os.path.join(ROOT, "tests", "golden", "depth_tail_keys.json")) as fh:
        sd = synth.synthetic_state_dict(json.load(fh), seed=11)
    dec = D.Decoder(num_classes=128)
    dec.load_state_dict({k[len("decoder."):]: v for k, v in sd.items() if k.startswith("decoder.")}, strict=True)
    dec = dec.to(dev).eval()
    for m in (dec.cross_atten1, dec.cross_atten2, dec.cross_atten3):
        m.to(torch.bfloat16)
    head = D.DepthHead(n_bins=256, min_val=1e-3, max_val=10.0)
    head.load_state_dict({k: v for k, v in sd.items() if k.startswith(("depth_head.", "conv_out."))}, strict=True)
    head = head.to(dev).eval()
    enc = cfpnet_b200.HistogramEncoder()
    enc.load_state_dict({k[len("hist_encoder."):]: v for k, v in sd.items() if k.startswith("hist_encoder.")}, strict=True)
    enc = enc.to(dev).eval()
    enc.out_dtype = torch.bfloat16
    NSETS = 3
    host_sets, dev_sets = [], []
    for s_ in range(NSETS):
        inp = synth.make_inputs(GEOMETRY, B, seed=200 + s_, levels=())
        h = {f"f{i}": t.contiguous().pin_memory() for i, t in enumerate(synth.encoder_features(GEOMETRY, B, seed=200 + s_))}
        h["hist_data"] = inp["hist_data"].pin_memory()
        h["mask"] = inp["mask"].pin_memory()
        host_sets.append(h)
        dev_sets.append({k: v.to(dev) for k, v in h.items()})
    patch_info = inp["patch_info"]
    h2d = sum(v.numel() * v.element_size() for v in host_sets[0].values())

    def step(d, i):
        shard.seed_posenc(i)
        hist = enc(d["hist_data"].unsqueeze(-1))
        unet, H, W = dec.forward_nhwc([d[f"f{j}"] for j in range(5)], hist, rect_data=None, mask=d["mask"], patch_info=patch_info, rgb=None)
        return head.forward_nhwc(unet, H, W)

    sampler = ClockSampler(0) if not os.environ.get("CFP_BENCH_NO_SAMPLER") else None
    if sampler:
        sampler.start()
    with torch.no_grad():
        for i in range(max(a.warmup, 3)):
            edges, pred = step(dev_sets[i % NSETS], i)
        torch.cuda.synchronize()
        d2h = pred.numel() * pred.element_size() + edges.numel() * edges.element_size()
        if sampler:
            t_s = time.perf_counter()
            while not sampler.samples and sampler.is_alive() and time.perf_counter() - t_s < 5.0:
                time.sleep(0.05)
            sampler.mark_begin()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        n0 = _lib.launch_count()
        e0.record()
        for i in range(a.steps):
            step(dev_sets[i % NSETS], i)
            if sampler and i == a.steps // 2:
                sampler.sample_now()
        e1.record()
        torch.cuda.synchronize()
        launches = _lib.launch_count() - n0
        ms_total = e0.elapsed_time(e1)
        if sampler:
            sampler.mark_end()
        clocks = sampler.finish() if sampler else None
        # end to end: inputs copied from pinned host memory on a side stream one step ahead, depth read back
        side = torch.cuda.Stream(dev)
        pred_host = torch.empty(pred.shape, dtype=pred.dtype).pin_memory()
        edges_host = torch.empty(edges.shape, dtype=edges.dtype).pin_memory()

        def e2e_run(n):
            cur = torch.cuda.current_stream()
            staged = None
            for i in range(n + 1):
                nxt = None
                if i < n:
                    with torch.cuda.stream(side):
                        nxt = {k: v.to(dev, non_blocking=True) for k, v in host_sets[i % NSETS].items()}
                        ev = torch.cuda.Event()
                        ev.record(side)
                if staged is not None:
                    cur.wait_event(staged[1])
                    ed, pr = step(staged[0], i)
                    pred_host.copy_(pr, non_blocking=True)
                    edges_host.copy_(ed, non_blocking=True)
                    for t in staged[0].values():
                        t.record_stream(cur)
                staged = (nxt, ev) if nxt is not None else None
            torch.cuda.synchronize()

        e2e_run(3)
        t_wall = time.perf_counter()
        e0.record()
        e2e_run(a.steps)
        e1.record()
        torch.cuda.synchronize()
        ms_e2e = max(e0.elapsed_time(e1), (time.perf_counter() - t_wall) * 1e3)
        _lib.profile_start()
        for i in range(a.steps):
            step(dev_sets[i % NSETS], i)
        prof = _lib.profile_stop()
    peaks = load_peaks()
    frames = B * a.steps
    line = {"metric": "CFPNet below the image encoder (hist encoder + decoder + fusion + adaptive-bins head) frames/s @416x544, 8x8 zones",
            "value": frames / (ms_total * 1e-3), "unit": "frames/s", "n_gpus": 1, "steps": a.steps, "warmup": max(a.warmup, 3),
            "ms_per_step": ms_total / a.steps, "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "bf16",
            "data": "synthetic",
            "config": {"workload": "histogram encoder + Decoder (UpSampleBN x4, 1x1 convs, cross_atten3/2/1 in their serial order) + "
                                   f"DepthRegression / conv_out head, combine1 layer list, 416x544, {B} frames, 1 GPU (SURVEY.md 8 f1 / f2 "
                                   "around the hot path); the image encoder's five feature maps are synthetic inputs",
                       "per_gpu_batch": B, "l2_policy": "inputs rotate over 3 distinct batches; a step's activations exceed the 126 MB L2"},
            "e2e": {"value": frames / (ms_e2e * 1e-3), "unit": "frames/s", "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": d2h},
            "gpu_launches": int(launches), "clocks": clocks}
    line["roofline"], line["kernels"] = roofline_from_profile(prof, a.steps, B, 2, peaks)
    print(json.dumps(line), flush=True)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="cfp", choices=["cfp", "reference"])
    ap.add_argument("--batch", type=int, default=None, help="frames per GPU per step (default 64; train_b32: 32)")
    ap.add_argument("--dtype", default="bf16", choices=["bf16", "f32"])
    ap.add_argument("--no-cpu", action="store_true", help="skip the cpu_baseline leg")
    ap.add_argument("--workload", default="combine1_b64", choices=["combine1_b64", "baseline_b16", "latency_480", "train_b32", "tail_b16"],
                    help="combine1_b64 = the headline (BASELINE.json configs[2]); the other two are side configurations")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write the last timed step's fused maps to DIR/<name>.npy (float32, a seeded sample above 64 MB)")
    a = ap.parse_args()
    if a.steps < 1:
        ap.error("--steps must be at least 1")
    if a.dump_outputs and (a.impl != "cfp" or a.workload != "combine1_b64"):
        ap.error("--dump-outputs serves the headline workload of --impl cfp")
    if a.batch is None:
        a.batch = {"train_b32": 32, "tail_b16": 16}.get(a.workload, 64)
    if a.workload == "tail_b16":
        if a.impl == "reference":
            print(json.dumps({"impl": "reference", "unavailable": "--impl reference serves the headline workload"}))
            return None
        return run_tail(a)
    if a.workload == "train_b32":
        if a.impl == "reference":
            print(json.dumps({"impl": "reference", "unavailable": "the training-step workload has no CPU arm; --impl reference "
                              "serves the headline workload"}))
            return None
        return run_train(a)
    if a.workload != "combine1_b64":
        return run_aux(a)
    a.warmup = max(a.warmup, 3) if a.impl == "cfp" else a.warmup
    if a.impl == "reference":
        run_reference(a)
    else:
        run_cfp(a)


if __name__ == "__main__":
    main()
