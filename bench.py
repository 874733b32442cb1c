#!/usr/bin/env python
"""bench.py — RepSurf-U fwd+bwd(+SGD step) throughput on synthetic clouds, one process per GPU.

  python bench.py [--gpus N] [--steps K] [--warmup W] [--workload seg|cls] [--impl reference] [--dump-outputs DIR]

Prints ONE JSON line (rank 0).  Contract: see the task statement / DESIGN.md "Measurement".
  value         clouds/sec, whole job, inputs already resident in HBM
  e2e           same metric through the public module API with HOST (pinned) inputs: H2D of the step's
                inputs and D2H of the loss inside the timed region
  roofline      the dominant repsurf_b200 kernel, timed with CUDA events inside the timed region
  cpu_baseline  the oracle port (oracle/model_ref.py + oracle C) on the host cores, bounded sample
  --impl reference   times that CPU port alone (the reference has no CPU path for segmentation; see DESIGN.md)
  --dump-outputs DIR after the timed steps (rank 0), what the last timed step of each workload returned to its caller:
                     DIR/<workload>_loss.npy, and the gradients and updated parameters, flattened in parameters() order,
                     as DIR/<workload>_grads.npy / DIR/<workload>_params.npy (float32).  Model, optimizer and random
                     state are reset to their seeded initial values before the last timed step, so that the dumped step
                     does not depend on the steps before it (how many warm-up steps ran, float atomics in their backward):
                     two builds given the same arguments compute the same step.
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

import numpy as np
import torch
import torch.nn as nn

# -------------------------------------------------------------------------------------------- workloads
WORKLOADS = {
    # BASELINE.json configs[2]/[3]: RepSurf-U S3DIS seg, B=8 clouds x N=40960 per GPU, training mode
    "seg": dict(name="RepSurf-U S3DIS seg (repsurf_umb_ssg), B=8 x N=40960 per GPU, fwd+bwd+SGD", clouds=8, n=40960),
    # BASELINE.json configs[1]: RepSurf-U ScanObjectNN cls, B=32, N=1024
    "cls": dict(name="RepSurf-U ScanObjectNN cls (repsurf_ssg_umb), B=32 x N=1024 per GPU, fwd+bwd+SGD", clouds=32, n=1024),
}


def make_inputs(workload, clouds, n, seed, pin):
    """Synthetic data of SURVEY.md §8(d): seg coord=rand*[8,8,3] mean-centred per cloud, feat=randn, 13 classes;
    cls points=rand*2-1, 15 classes.  Host tensors (pinned when asked)."""
    g = torch.Generator().manual_seed(seed)
    if workload == "seg":
        coord = torch.rand(clouds * n, 3, generator=g) * torch.tensor([8.0, 8.0, 3.0])
        coord = (coord.view(clouds, n, 3) - coord.view(clouds, n, 3).mean(1, keepdim=True)).reshape(-1, 3).contiguous()
        feat = torch.randn(clouds * n, 3, generator=g)
        target = torch.randint(0, 13, (clouds * n,), generator=g)
        offset = (torch.arange(1, clouds + 1) * n).int()
        ts = [coord, feat, offset, target]
    else:
        pts = torch.rand(clouds, 3, n, generator=g) * 2 - 1
        target = torch.randint(0, 15, (clouds,), generator=g)
        ts = [pts, target]
    if pin:
        ts = [t.pin_memory() for t in ts]
    return ts


# -------------------------------------------------------------------------------------------- clocks
class ClockSampler:
    """SM clock / throttle reasons sampled DURING the timed region (B200_PROFILING.md).  Uses NVML in-process
    (nvidia_ml_py) from a background thread: an external `nvidia-smi -lms` loop measurably slows the step."""

    def __init__(self, gpu_index):
        self.idx, self.rows, self.stop_flag, self.thread, self.ok = gpu_index, [], False, None, False

    def start(self):
        try:
            import pynvml
            pynvml.nvmlInit()
            # torch's device index follows CUDA_VISIBLE_DEVICES; map through the PCI bus id
            bus = torch.cuda.get_device_properties(self.idx).pci_bus_id if hasattr(torch.cuda.get_device_properties(self.idx), "pci_bus_id") else None
            h = None
            if bus is not None:
                for i in range(pynvml.nvmlDeviceGetCount()):
                    hi = pynvml.nvmlDeviceGetHandleByIndex(i)
                    if int(pynvml.nvmlDeviceGetPciInfo(hi).bus) == int(bus):
                        h = hi
            if h is None:
                h = pynvml.nvmlDeviceGetHandleByIndex(self.idx)
            self.nv, self.h, self.ok = pynvml, h, True
            self.max_mhz = float(pynvml.nvmlDeviceGetMaxClockInfo(h, pynvml.NVML_CLOCK_SM))
        except Exception:
            self.ok = False
            return

        def loop():
            nv = self.nv
            while not self.stop_flag:
                try:
                    sm = nv.nvmlDeviceGetClockInfo(self.h, nv.NVML_CLOCK_SM)
                    rs = nv.nvmlDeviceGetCurrentClocksEventReasons(self.h) if hasattr(nv, "nvmlDeviceGetCurrentClocksEventReasons") \
                        else nv.nvmlDeviceGetCurrentClocksThrottleReasons(self.h)
                    self.rows.append((float(sm), int(rs)))
                except Exception:
                    pass
                time.sleep(0.02)      # ~10 samples over a 10-step region; in-process NVML queries cost ~0.1 ms each
        self.thread = threading.Thread(target=loop, daemon=True)
        self.thread.start()

    def stop(self):
        if not self.ok:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvml unavailable"]}
        self.stop_flag = True
        self.thread.join(timeout=1.0)
        nv = self.nv
        names = {"hw_slowdown": getattr(nv, "nvmlClocksThrottleReasonHwSlowdown", 0x8),
                 "hw_thermal_slowdown": getattr(nv, "nvmlClocksThrottleReasonHwThermalSlowdown", 0x40),
                 "sw_thermal_slowdown": getattr(nv, "nvmlClocksThrottleReasonSwThermalSlowdown", 0x20),
                 "sw_power_cap": getattr(nv, "nvmlClocksThrottleReasonSwPowerCap", 0x4)}
        reasons = sorted({k for _sm, rs in self.rows for k, bit in names.items() if rs & bit})
        sm = [r[0] for r in self.rows]
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_min_mhz": float(min(sm)) if sm else None,
                "sm_max_mhz": self.max_mhz, "reasons": reasons, "samples": len(sm)}


# -------------------------------------------------------------------------------------------- per-entry timing
class _OpndInfo:
    def __init__(self, o):
        self.K, self.ku, self.kind = int(o.K), int(o.ku), int(o.kind)


def _lite(x):
    if isinstance(x, (int, float)) or x is None:
        return x
    if hasattr(x, "kind") and hasattr(x, "ku"):
        return _OpndInfo(x)
    return None


class EntryTimer:
    """CUDA-event timing of every C-ABI call made through repsurf_b200._native.call (torch's current stream)."""

    def __init__(self, native, only=None):
        self.native, self.orig, self.ev, self.only = native, native.call, [], only

    def __enter__(self):
        def timed(name, *args):
            if self.only is not None and name not in self.only:
                return self.orig(name, *args)
            a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            a.record()
            self.orig(name, *args)
            b.record()
            # keep only plain numbers: holding tensors / descriptors here would pin every activation of the step
            self.ev.append((name, tuple(_lite(x) for x in args[:8]), a, b))
        self.native.call = timed
        return self

    def __exit__(self, *exc):
        self.native.call = self.orig
        return False

    def summary(self):
        torch.cuda.synchronize()
        out = {}
        for name, args, a, b in self.ev:
            d = out.setdefault(name, {"ms": 0.0, "calls": 0, "each": []})
            t = a.elapsed_time(b)
            d["ms"] += t
            d["calls"] += 1
            d["each"].append((args, t))
        return out


# -------------------------------------------------------------------------------------------- algorithmic work
def fps_algorithmic_bytes(n, m):
    """SURVEY.md §8(d) streaming model: (m-1) * n * 20 B (12 B xyz + 4 B read + 4 B write of the running
    minimum) + 4 m B of indices, per segment."""
    return (m - 1) * n * 20 + 4 * m


def peaks():
    """(HBM GB/s, bf16 TFLOP/s, where from): the driver-written MEASURED_PEAKS.json; if that file is absent (it is git-ignored and
    did not survive a re-created build container in round 2) the measured values as an earlier run of this bench recorded them
    from it (profiles/r02_bench_seg.json); else the fallback of B200_PROFILING.md."""
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        d = json.load(open(p))
        return d["hbm_gbs"], d.get("bf16_tflops", 1590.0), "measured (MEASURED_PEAKS.json)"
    rec = os.path.join(ROOT, "profiles", "r02_bench_seg.json")
    try:
        r = json.load(open(rec))["roofline"]
        if str(r.get("peak_source", "")).startswith("measured") and r.get("unit") == "GB/s":
            return float(r["peak"]), 1719.0, "measured (MEASURED_PEAKS.json is absent: its hbm_gbs as recorded in profiles/r02_bench_seg.json)"
    except Exception:
        pass
    return 6650.0, 1590.0, "fallback (B200_PROFILING.md)"


# -------------------------------------------------------------------------------------------- CPU arm
CPU_SAMPLE = {"seg": (2, 40960), "cls": (32, 1024)}


def cpu_port_inner(workload, steps, warmup, threads):
    """Runs INSIDE the child process started by cpu_arm (one thread pool of `threads`, passive OpenMP waiting): fwd+bwd of
    the oracle port (oracle/model_ref.py over the OpenMP C oracle) on the bounded sample; prints seconds per step."""
    from oracle import model_ref as MR
    torch.set_num_threads(threads)
    torch.manual_seed(0)
    np.random.seed(0)
    clouds, n = CPU_SAMPLE[workload]
    if workload == "seg":
        model = MR.SegNet().train()
        coord, feat, offset, target = make_inputs("seg", clouds, n, 0, False)
        crit = nn.CrossEntropyLoss()

        def step():
            model.zero_grad(set_to_none=True)
            crit(model([coord, feat, offset]), target).backward()
    else:
        from repsurf_b200.models import SmoothClsLoss
        model = MR.ClsNet().train()
        pts, target = make_inputs("cls", clouds, n, 0, False)
        crit = SmoothClsLoss()

        def step():
            model.zero_grad(set_to_none=True)
            crit(model(pts), target).backward()
    for _ in range(warmup):
        step()
    ts = []
    for _ in range(steps):
        t0 = time.perf_counter()
        step()
        ts.append(time.perf_counter() - t0)
    print("CPU_PORT_RESULT " + json.dumps({"threads": threads, "sec": ts}), flush=True)


def cpu_arm(workload, steps):
    """The reference's CPU path for this workload = the oracle port (DESIGN.md section 6), timed on the host cores.
    Each candidate thread count runs in its OWN process with ONE pool of that size (OMP_NUM_THREADS = torch threads,
    OMP_WAIT_POLICY=passive): round 1 ran torch's 128 intra-op threads and 128 spinning OpenMP threads in one process and
    was 37x slower than the same code with one thread.  Result: best step over all candidates (best-of-k), with the
    thread count that achieved it."""
    cores = os.cpu_count() or 1
    cands = sorted({min(cores, 8), min(cores, 32), cores})
    clouds, n = CPU_SAMPLE[workload]
    tried, best = {}, None
    for t in cands:
        env = dict(os.environ)
        env.update({"OMP_NUM_THREADS": str(t), "MKL_NUM_THREADS": str(t), "OMP_WAIT_POLICY": "passive", "GOMP_SPINCOUNT": "0",
                    "OMP_PROC_BIND": "false", "CUDA_VISIBLE_DEVICES": ""})
        for k in ("RANK", "LOCAL_RANK", "WORLD_SIZE", "MASTER_ADDR", "MASTER_PORT", "TORCHELASTIC_RUN_ID"):
            env.pop(k, None)
        cmd = [sys.executable, os.path.abspath(__file__), "--impl", "reference-inner", "--workload", workload,
               "--steps", str(steps), "--warmup", "1", "--threads", str(t)]
        try:
            out = subprocess.run(cmd, env=env, capture_output=True, text=True, timeout=600).stdout
            line = [l for l in out.splitlines() if l.startswith("CPU_PORT_RESULT ")][-1]
            sec = json.loads(line[len("CPU_PORT_RESULT "):])["sec"]
        except Exception:
            continue
        tried[str(t)] = round(clouds / min(sec), 4)
        if best is None or min(sec) < best[0]:
            best = (min(sec), t)
    if best is None:
        raise RuntimeError("the CPU port did not run")
    dt, threads = best
    desc = (f"{clouds} cloud(s) x N={n} of the same workload, fwd+bwd, best of {steps} step(s) after 1 warm-up, "
            f"one pool of {threads} threads (of {cores} cores; clouds/s by thread count: {tried})")
    return {"value": clouds / dt, "unit": "clouds/s", "cores": threads, "kind": "port", "sample": desc,
            "sec_per_step": dt, "host_cores": cores, "tried": tried}


# -------------------------------------------------------------------------------------------- our arm
TIMED_ENTRIES = {"rsb_furthestsampling_packed", "rsb_furthestsampling_packed_bounded", "rsb_furthestsampling_dense",
                 "rsb_knnquery_packed", "rsb_knnquery_dense", "rsb_knnquery_grid", "rsb_gemm_wgrad", "rsb_gemm_rows",
                 "rsb_ballquery"}


def opnd_bytes(o, rows):
    # gathered operand (kind 5): the row index + the gathered table row (SURVEY 8d: fused gather m*ns*(4 + 4C) bytes)
    per_row = {0: o.K, 1: o.K, 2: 2 * o.K, 3: o.K + min(o.K, o.ku), 4: o.K, 5: o.K + 1}[o.kind]
    return rows * per_row * 4


def gemm_alg_bytes(name, a):
    """algorithmic HBM bytes of one GEMM launch: every operand tensor read once, the result written once"""
    if name == "rsb_gemm_wgrad":
        return opnd_bytes(a[1], a[0]) + opnd_bytes(a[2], a[0]) + a[1].K * a[2].K * 4
    return opnd_bytes(a[2], a[0]) + a[0] * a[1] * 4


def gemm_desc(name, a):
    if name == "rsb_gemm_wgrad":
        return f"wgrad rows={a[0]} dW[{a[1].K}x{a[2].K}], operand kinds {a[1].kind}/{a[2].kind}"
    return f"rows={a[0]} K={a[2].K} N={a[1]}, operand kind {a[2].kind}"


DUMP_LIMIT_BYTES = 64 << 20


def run_ours(workload, args, rank, local_rank, world, dev, full):
    """Times `workload` (value: inputs resident; e2e: pinned host inputs + loss read-back).  full: also the per-entry
    rooflines, launch count and clocks (primary workload only).  With --dump-outputs, res["outputs"] holds what the last
    timed step returned (loss, gradients, updated parameters)."""
    import torch.distributed as dist
    from repsurf_b200 import _native
    from repsurf_b200.models import RepSurfCls, RepSurfSeg, SmoothClsLoss
    from repsurf_b200.seg import pointops as PS
    from repsurf_b200.dist import FlatGrads, broadcast_module

    wl = WORKLOADS[workload]
    torch.manual_seed(rank)
    np.random.seed(rank)
    model = (RepSurfSeg() if workload == "seg" else RepSurfCls()).to(dev).train()
    if workload == "seg":
        from repsurf_b200.seg.loss import CrossEntropyLoss      # the step's criterion (nn.CrossEntropyLoss semantics), one kernel
        crit = CrossEntropyLoss()
    else:
        crit = SmoothClsLoss()
    params = [p for p in model.parameters()]
    broadcast_module(model)
    initial_state = {k: v.detach().clone() for k, v in model.state_dict().items()} if args.dump_outputs else None
    # gradients are packed into one flat buffer after backward: ONE all-reduce per step (3.9 MB seg / 5.9 MB cls)
    fg = FlatGrads(params)
    opt = torch.optim.SGD(params, lr=1e-3, momentum=0.9, weight_decay=1e-4)

    host = make_inputs(workload, wl["clouds"], wl["n"], 100 + rank, pin=True)
    devin = [t.to(dev) for t in host]
    if workload == "seg":
        PS.register_offsets(devin[2], host[2].tolist())
    h2d_bytes = sum(t.numel() * t.element_size() for t in host)

    def fwd_bwd(inp):
        fg.zero()
        if workload == "seg":
            loss = crit(model([inp[0], inp[1], inp[2]]), inp[3])
        else:
            loss = crit(model(inp[0]), inp[1])
        loss.backward()
        fg.allreduce_mean()
        opt.step()
        return loss

    # Both steps have static shapes here (fixed B x N; fixed offsets) and are captured once in a CUDA graph and replayed
    # (repsurf_b200/graph.py): issued eagerly the classification step is host-bound (~300 launches of a few us), and the
    # segmentation step (~370 launches, 19.6 ms of GPU work) becomes host-bound on a box with a slow host (measured 25.3 ms).
    # One process: forward + backward + SGD in the graph.  N > 1 (segmentation): forward + backward in the graph, then the
    # gradient all-reduce and the optimizer step eagerly; classification keeps its eager step with the overlapped all-reduce.
    # RSB_CLS_EAGER=1 / RSB_SEG_EAGER=1 force the eager step; a capture that fails falls back to it and says so (graph_error).
    gstep, graph_error = None, None
    if workload == "cls" and world == 1 and not os.environ.get("RSB_CLS_EAGER"):
        from repsurf_b200.graph import GraphedTrainStep
        gstep = GraphedTrainStep(model, crit, opt, [devin[0]], devin[1])
    elif workload == "seg" and not os.environ.get("RSB_SEG_EAGER"):
        from repsurf_b200.graph import graphed_seg_step
        try:
            gstep = graphed_seg_step(model, crit, opt, devin[0], devin[1], devin[2], devin[3], optimizer_in_graph=(world == 1),
                                     after_backward=(fg.allreduce_mean if world > 1 else None),
                                     capture_error_mode="global" if world == 1 else "thread_local")
        except Exception as e:                                # noqa: BLE001 - any capture failure: the eager step still runs
            graph_error = f"{type(e).__name__}: {e}"[:300]
            gstep = None
            torch.cuda.synchronize()
            opt.zero_grad(set_to_none=True)
    if workload == "seg" and world > 1 and not os.environ.get("RSB_SEG_EAGER"):
        # every rank must take the same path (the graphed step reduces the packed buffer once, the eager step in two runs from
        # hooks): if the capture failed anywhere, everybody steps eagerly
        ok = torch.tensor([1 if gstep is not None else 0], device=dev)
        dist.all_reduce(ok, op=dist.ReduceOp.MIN)
        if int(ok) == 0 and gstep is not None:
            gstep, graph_error = None, "capture failed on another rank"
    if gstep is not None and workload == "seg":
        h2d_bytes -= host[2].numel() * host[2].element_size()     # the offsets are fixed by the capture, not copied per step

    def step_eager():
        return fwd_bwd(devin)

    last = {}

    def step_resident():
        if gstep is not None:
            loss = gstep(gstep.static_in, gstep.static_tgt)
        else:
            loss = fwd_bwd(devin)
        last["loss"] = loss
        return loss

    def step_e2e():
        if gstep is not None:                                # pinned host -> the graph's static buffers -> replay -> loss read
            if workload == "seg":
                return float(gstep([host[0], host[1], gstep.static_in[2]], host[3]).detach())
            return float(gstep([host[0]], host[1]).detach())
        inp = [t.to(dev, non_blocking=True) for t in host]
        if workload == "seg":
            PS.register_offsets(inp[2], host[2].tolist())   # the host already holds the offsets it uploads
        loss = fwd_bwd(inp)
        return float(loss.detach())                          # D2H read of the step's result

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    host_issue = {}

    def timed(fn, steps, on_start=None, before_last=None):
        # the host needs ~12 of a step's ~20 ms to issue it: a full (generation-2) pass of Python's cyclic garbage collector
        # inside the 10-step region (tens of ms over the autograd graphs of a step) makes those steps host-bound - seen twice
        # as a 22 / 33 ms first pass.  Collect before, keep the collector off while timing (reference counting still frees).
        import gc
        gc.collect()
        gc.disable()
        # three more untimed steps back to back with the timed ones: the GPU has just idled through the collector / NVML set-up
        # above (tens to hundreds of ms on a freshly booted box), and the first pass after such a gap was sporadically 15-90 %
        # slower than every later pass of the same process at unchanged reported clocks (host issue time unchanged, so the
        # slowdown is on the device: memory / power state ramp).  Timing starts from a busy device.
        for _ in range(3):
            fn()
        barrier()
        if on_start is not None:
            on_start()                                       # e.g. drop the per-entry events of the pre-roll steps
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        t0 = time.perf_counter()
        e0.record()
        marks = []
        for i in range(steps):
            if before_last is not None and i == steps - 1:
                before_last()
            fn()
            if os.environ.get("RSB_STEP_MARKS"):
                m = torch.cuda.Event(enable_timing=True)
                m.record()
                marks.append(m)
        e1.record()
        host_issue[fn.__name__] = (time.perf_counter() - t0) * 1e3 / steps     # host time to ISSUE a step (diagnostic)
        if marks:
            torch.cuda.synchronize()
            ts = [e0.elapsed_time(m) for m in marks]
            host_issue[fn.__name__ + "_marks"] = [round(b - a, 2) for a, b in zip([0.0] + ts[:-1], ts)]
        gc.enable()
        barrier()
        ms = torch.tensor([e0.elapsed_time(e1)], device=dev)
        if world > 1:
            dist.all_reduce(ms, op=dist.ReduceOp.MAX)
        return float(ms) / steps

    for _ in range(max(args.warmup, 3)):
        step_resident()
    # still warm-up, never timed: keep stepping until the caching allocator has stopped growing.  The geometry plan allocates
    # on side streams (blocks return to their pool only after the consumer stream's recorded use), so the steady-state set of
    # blocks can take a few more steps than W to appear; a cudaMalloc of a GB-sized block inside the timed region costs tens
    # of milliseconds (seen once: 33 ms/step in the first pass against 20 ms in every later pass of the same process).
    if workload == "seg":
        from repsurf_b200.seg.modules import reserve_allocator_headroom
        reserve_allocator_headroom(dev)          # one big cached block per stream: later requests split it instead of cudaMalloc
    reserved = -1
    for _ in range(12):
        torch.cuda.synchronize()
        now = torch.cuda.memory_reserved(dev)
        if now == reserved:
            break
        reserved = now
        step_resident()
        step_resident()

    def restore_initial_state():
        # in place and in stream order: a captured graph keeps reading / writing these same tensors
        for k, v in model.state_dict().items():
            v.copy_(initial_state[k])
        for st in opt.state.values():
            if st.get("momentum_buffer") is not None:
                st["momentum_buffer"].zero_()       # SGD's first step with a zero buffer is its step without one
        torch.manual_seed(rank)
        np.random.seed(rank)

    clocks = ClockSampler(local_rank)
    if full and rank == 0 and not os.environ.get("RSB_NO_CLOCKS"):
        clocks.start()
    _native.reset_launch_count()
    mallocs0 = torch.cuda.memory_stats(dev).get("num_device_alloc", 0)
    ms_step = timed(step_resident, args.steps, before_last=restore_initial_state if initial_state is not None else None)
    outputs = None
    if args.dump_outputs:
        flat = lambda ts: torch.cat([t.detach().reshape(-1) for t in ts]).float().cpu().numpy()
        outputs = {"loss": last["loss"].detach().float().cpu().numpy(),
                   "grads": flat([p.grad if p.grad is not None else torch.zeros_like(p) for p in params]),
                   "params": flat(params)}
    device_allocs = torch.cuda.memory_stats(dev).get("num_device_alloc", 0) - mallocs0      # cudaMalloc calls inside (diagnostic)
    launches = _native.launch_count() if gstep is None else gstep.launches_per_step * args.steps   # replays bypass the counter
    clk = clocks.stop() if (full and rank == 0) else None
    # per-entry kernel times for the rooflines: a SEPARATE pass of the same steps with the side streams of the geometry plan
    # switched off, so that every launch is timed alone on one stream (CUDA events around each C-ABI call); in the throughput
    # pass above FPS / kNN run concurrently with the GEMMs and event times of one stream would include that interference
    per_entry, ms_serial = {}, None
    if full:
        from repsurf_b200.seg import modules as seg_modules
        timed_entries = None if os.environ.get("RSB_TIME_ALL_ENTRIES") else TIMED_ENTRIES
        seg_modules.USE_SIDE_STREAMS = False
        step_eager()
        with EntryTimer(_native, timed_entries) as et:
            ms_serial = timed(step_eager, args.steps, on_start=et.ev.clear)     # exactly `steps` steps of events
        per_entry = et.summary()
        seg_modules.USE_SIDE_STREAMS = True
        step_eager()
    for _ in range(2):
        step_e2e()
    ms_e2e = timed(step_e2e, args.steps)
    # work counters of the grid kNN: ONE extra untimed step (the counting adds an atomic per query)
    knn_work = None
    if full and workload == "seg":
        ctr = torch.zeros(3, dtype=torch.int64, device=dev)
        _native.lib().rsb_knn_grid_set_counters(ctr.data_ptr())
        step_eager()                                         # eager: a graph replay carries the launch arguments of its capture
        torch.cuda.synchronize()
        _native.lib().rsb_knn_grid_set_counters(None)
        knn_work = [int(v) for v in ctr.tolist()]

    clouds_total = wl["clouds"] * world
    res = {"key": workload, "workload": wl["name"], "value": clouds_total / (ms_step * 1e-3), "ms_per_step": ms_step,
           "e2e": {"value": clouds_total / (ms_e2e * 1e-3), "unit": "clouds/s", "ms_per_step": ms_e2e,
                   "h2d_bytes_per_step": h2d_bytes, "d2h_bytes_per_step": 4},
           "gpu_launches": int(launches), "clocks": clk, "per_entry": per_entry, "knn_work": knn_work, "ms_serial": ms_serial,
           "host_issue_ms": {k: (v if isinstance(v, list) else round(v, 3)) for k, v in host_issue.items()},
           "device_allocs": int(device_allocs), "cuda_graph": gstep is not None, "graph_error": graph_error, "outputs": outputs}
    del model, opt, fg, devin, gstep
    torch.cuda.empty_cache()
    return res


def build_rooflines(per_entry, knn_work, ms_step, steps, workload):
    wl = WORKLOADS[workload]
    hbm_peak, tf_peak, peak_src = peaks()
    entry_share = {k: round(v["ms"] / (ms_step * steps), 4) for k, v in per_entry.items()}
    rooflines = {}

    def biggest(v):
        big = max(t for _a, t in v["each"])
        sel = [(a, t) for a, t in v["each"] if t > 0.6 * big]
        return sel[0][0], float(np.mean([t for _a, t in sel]))

    # ---- GEMMs: per shape (launches of one shape averaged), then the heaviest shape per entry, the time-weighted total of
    # ALL launches of both entries, and the worst shape among those that matter (>= 2 % of the GEMM time)
    shapes = {}
    for name in ("rsb_gemm_rows", "rsb_gemm_wgrad"):
        for a, t in per_entry.get(name, {"each": []})["each"]:
            key = (name, gemm_desc(name, a))
            d = shapes.setdefault(key, {"bytes": gemm_alg_bytes(name, a), "ms": 0.0, "n": 0,
                                        "flops": 2.0 * a[0] * (a[1].K * a[2].K if name == "rsb_gemm_wgrad" else a[1] * a[2].K)})
            d["ms"] += t
            d["n"] += 1
    gemm_ms = sum(d["ms"] for d in shapes.values())
    for name, kern in (("rsb_gemm_rows", "gemm_rows2_kernel (TMA-fed tcgen05 3xTF32)"), ("rsb_gemm_wgrad", "gemm_wgrad2_kernel (TMA-fed tcgen05 3xTF32)")):
        mine = {k: d for k, d in shapes.items() if k[0] == name}
        if not mine:
            continue
        k, d = max(mine.items(), key=lambda kd: kd[1]["bytes"])
        t_ms = d["ms"] / d["n"]
        ach = d["bytes"] / (t_ms * 1e-3) / 1e9
        if name == "rsb_gemm_wgrad" and "dW[" in k[1]:
            mn = k[1].split("dW[")[1].split("]")[0].split("x")
            if int(mn[0]) <= 32 and int(mn[1]) <= 32:
                kern = "wgrad_narrow_kernel (fp32 pipe, register-blocked; the 32 x 32 class does not go to the tensor core)"
        rooflines[name] = {"kernel": kern, "bound": "hbm", "achieved": ach, "peak": hbm_peak, "unit": "GB/s", "frac": ach / hbm_peak,
                           "launch_ms": t_ms, "launch": k[1] + " (the shape that moves the most bytes)",
                           "algorithmic_bytes_per_launch": d["bytes"], "algorithmic_tflops": d["flops"] / (t_ms * 1e-3) / 1e12}
    if shapes:
        tot_b = sum(d["bytes"] * d["n"] for d in shapes.values())
        ach = tot_b / (gemm_ms * 1e-3) / 1e9
        rooflines["gemm_total"] = {"kernel": "all gemm_rows + gemm_wgrad launches of the timed steps", "bound": "hbm", "achieved": ach,
                                   "peak": hbm_peak, "unit": "GB/s", "frac": ach / hbm_peak, "launch_ms": gemm_ms / steps,
                                   "launch": f"{sum(d['n'] for d in shapes.values()) // steps} launches per step, time-weighted",
                                   "algorithmic_bytes_per_launch": tot_b / steps,
                                   "algorithmic_tflops": sum(d["flops"] * d["n"] for d in shapes.values()) / (gemm_ms * 1e-3) / 1e12}
        heavy = {k: d for k, d in shapes.items() if d["ms"] >= 0.02 * gemm_ms}
        k, d = min(heavy.items(), key=lambda kd: kd[1]["bytes"] * kd[1]["n"] / kd[1]["ms"])
        t_ms = d["ms"] / d["n"]
        ach = d["bytes"] / (t_ms * 1e-3) / 1e9
        rooflines["gemm_worst"] = {"kernel": k[0], "bound": "hbm", "achieved": ach, "peak": hbm_peak, "unit": "GB/s", "frac": ach / hbm_peak,
                                   "launch_ms": t_ms, "launch": k[1] + f" (lowest fraction among shapes with >= 2 % of the GEMM time; "
                                   f"{round(100 * d['ms'] / gemm_ms, 1)} % of it)", "algorithmic_bytes_per_launch": d["bytes"]}

    if shapes:
        top = sorted(shapes.items(), key=lambda kd: -kd[1]["ms"])[:12]
        rooflines["gemm_total"]["shapes_by_time"] = [
            {"launch": k[1], "entry": k[0], "launches_per_step": d["n"] / steps, "ms_per_step": round(d["ms"] / steps, 4),
             "frac": round(d["bytes"] * d["n"] / (d["ms"] * 1e-3) / 1e9 / hbm_peak, 3)} for k, d in top]
    for name, v in per_entry.items():
        if name.startswith("rsb_furthestsampling"):
            a, t_ms = biggest(v)
            if name.endswith("dense"):
                nseg, n_seg, m_seg = a[0], a[1], a[2]
            elif name.endswith("bounded"):          # sectorized FPS: nseg sectors of ~n/4 points
                nseg = a[0]
                n_seg, m_seg = wl["n"] * wl["clouds"] // nseg, wl["n"] // 4 * wl["clouds"] // nseg
            else:
                nseg, n_seg = a[0], a[1]
                m_seg = n_seg // 4
            alg = nseg * fps_algorithmic_bytes(n_seg, m_seg)
            ach = alg / (t_ms * 1e-3) / 1e9
            rooflines[name] = {"kernel": "fps2_kernel (cluster, st.async exchange)" if nseg * 0 == 0 else "", "bound": "hbm",
                               "achieved": ach, "peak": hbm_peak, "unit": "GB/s", "frac": ach / hbm_peak, "launch_ms": t_ms,
                               "launch": f"{nseg} segments of ~{n_seg} points -> {m_seg} samples (streaming model of SURVEY 8d; the "
                                         "kernel is register-resident and latency-bound, see us_per_sample)",
                               "algorithmic_bytes_per_launch": alg, "us_per_sample": 1e3 * t_ms / max(m_seg, 1),
                               "busy_sms_note": "one cluster of CTAs per segment: nseg x cluster size of 148 SMs"}
        elif name == "rsb_knnquery_grid" and knn_work:
            # all grid launches of a step together: the counters are per step
            t_ms = v["ms"] / steps
            cand, ranges, replays = knn_work
            queries = sum(a[6] for a, _t in v["each"]) / steps
            fp32_peak = 148 * 128 * 2 * 1.965e9 / 1e12     # B200: 148 SMs x 128 FFMA lanes x 2 x 1.965 GHz
            ach = cand * 9 / (t_ms * 1e-3) / 1e12
            rooflines[name] = {"kernel": "knn_grid_kernel (+ grid build)", "bound": "fp32 (candidates actually evaluated x 9 flop)",
                               "achieved": ach, "peak": fp32_peak, "unit": "TFLOP/s", "frac": ach / fp32_peak, "launch_ms": t_ms,
                               "launch": f"{v['calls'] // steps} searches per step, {int(queries)} queries",
                               "candidates_per_step": cand, "candidates_per_query": cand / max(queries, 1),
                               "cell_ranges_per_query": ranges / max(queries, 1), "tie_replays_per_step": replays,
                               "candidate_gbs": cand * 16 / (t_ms * 1e-3) / 1e9,
                               "all_pairs_equivalent_gpairs_per_s": sum(a[6] * (a[5] / max(a[2], 1)) for a, _t in v["each"]) / steps / (t_ms * 1e-3) / 1e9}
    # measured DRAM traffic per launch from the committed ncu --set full capture of the same kernels
    traffic = {}
    for cand_path in ("r02_ncu_full_seg_traffic.json", "r01_ncu_full_seg_v2_traffic.json"):
        tpath = os.path.join(ROOT, "profiles", cand_path)
        if os.path.exists(tpath) and workload == "seg":
            traffic = json.load(open(tpath))
            break
    fam = {"rsb_gemm_wgrad": ("gemm_wgrad2_kernel", "gemm_wgrad_kernel"), "rsb_gemm_rows": ("gemm_rows2_kernel", "gemm_rows_kernel"),
           "rsb_knnquery_grid": ("knn_grid_kernel",), "rsb_furthestsampling_packed": ("fps2_kernel", "fps_kernel"),
           "rsb_furthestsampling_packed_bounded": ("fps2_kernel", "fps_kernel"), "rsb_furthestsampling_dense": ("fps2_kernel", "fps_kernel")}
    shape_traffic = {}
    sp = os.path.join(ROOT, "profiles", "r02_ncu_gemm_traffic.json")
    if os.path.exists(sp):
        shape_traffic = json.load(open(sp))["by_shape"]
    for name, r in rooflines.items():
        if name.startswith("rsb_gemm") or name.startswith("gemm_"):
            # GEMM launches run at many shapes: DRAM traffic only where the ncu capture holds the SAME launch shape
            r["traffic"] = next((v for k, v in shape_traffic.items() if r["launch"].startswith(k)), None)
        else:
            t = next((traffic[f] for f in fam.get(name, ()) if f in traffic), None)
            r["traffic"] = t["dram_bytes"] if t else None
        r["peak_source"] = peak_src
    return rooflines, entry_share


# -------------------------------------------------------------------------------------------- main
def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--workload", default=os.environ.get("RSB_WORKLOAD", "seg"), choices=list(WORKLOADS) + ["micro"])
    ap.add_argument("--impl", default="ours", choices=["ours", "reference", "reference-inner"])
    ap.add_argument("--threads", type=int, default=1)
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-secondary", action="store_true")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None)
    args = ap.parse_args()

    rank = int(os.environ.get("RANK", 0))
    local_rank = int(os.environ.get("LOCAL_RANK", 0))
    world = int(os.environ.get("WORLD_SIZE", 1))
    metric = "clouds/sec fwd+bwd RepSurf-U"

    if args.impl == "reference-inner":
        cpu_port_inner(args.workload, args.steps, args.warmup, args.threads)
        return
    if args.workload == "micro":
        from scripts.microbench import main as micro_main
        micro_main()
        return
    wl = WORKLOADS[args.workload]

    # ---------------- reference arm: the CPU port on the host cores (rank 0 only) ----------------
    if args.impl == "reference":
        if rank != 0:
            return
        steps = max(1, min(args.steps, 3))
        cb = cpu_arm(args.workload, steps)
        print(json.dumps({
            "impl": "reference", "metric": metric, "value": cb["value"], "unit": "clouds/s", "n_gpus": args.gpus, "steps": steps,
            "warmup": 1, "ms_per_step": cb["sec_per_step"] * 1e3, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
            "dtype": "f32", "data": "synthetic", "config": {"workload": wl["name"], "sample": cb["sample"]},
            "cpu_baseline": cb,
            "e2e": {"value": cb["value"], "unit": "clouds/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}))
        return

    # ---------------- our arm ---------------------------------------------------------------------
    import torch.distributed as dist
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)
    torch.backends.cudnn.allow_tf32 = False          # fp32-faithful MLP (north star: 1e-5 rel)
    torch.backends.cuda.matmul.allow_tf32 = False

    r = run_ours(args.workload, args, rank, local_rank, world, dev, full=True)
    second = None
    if not args.no_secondary:
        other = "cls" if args.workload == "seg" else "seg"
        second = run_ours(other, args, rank, local_rank, world, dev, full=False)
    if rank != 0:
        if world > 1:
            dist.destroy_process_group()
        return
    if args.dump_outputs:
        arrays = {f"{res['key']}_{name}": a for res in (r, second) if res is not None for name, a in res["outputs"].items()}
        total = sum(a.nbytes for a in arrays.values())
        if total > DUMP_LIMIT_BYTES:
            raise RuntimeError(f"--dump-outputs: {total} bytes exceed the {DUMP_LIMIT_BYTES} byte limit")
        os.makedirs(args.dump_outputs, exist_ok=True)
        for name, a in arrays.items():
            np.save(os.path.join(args.dump_outputs, name + ".npy"), a)

    rooflines, entry_share = build_rooflines(r["per_entry"], r["knn_work"], r["ms_serial"] or r["ms_per_step"], args.steps, args.workload)
    dom = max(r["per_entry"].items(), key=lambda kv: kv[1]["ms"]) if r["per_entry"] else None
    roof = dict(rooflines[dom[0]]) if dom and dom[0] in rooflines else None
    out = {
        "metric": metric, "value": r["value"], "unit": "clouds/s", "n_gpus": world, "steps": args.steps, "warmup": max(args.warmup, 3),
        "ms_per_step": r["ms_per_step"], "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32",
        "data": "synthetic",
        "config": {"workload": wl["name"], "clouds_per_gpu": wl["clouds"], "points_per_cloud": wl["n"], "parallelism": f"dp{world}",
                   "optimizer_step": "SGD momentum inside the timed region", "tf32": False, "cuda_graph": r["cuda_graph"],
                   "cuda_graph_error": r["graph_error"],
                   "l2": "per-step working set (activations > 126 MB) exceeds L2; no explicit flush"},
        "e2e": r["e2e"], "gpu_launches": r["gpu_launches"], "roofline": roof, "rooflines": rooflines,
        "entry_time_share": entry_share, "dominant_entry": dom[0] if dom else None, "clocks": r["clocks"],
        "host_issue_ms_per_step": r["host_issue_ms"], "cudaMalloc_calls_in_timed_region": r["device_allocs"],
        "roofline_pass": {"note": "rooflines / entry_time_share come from a second pass of the same steps with the geometry plan's side "
                                  "streams off (every kernel timed alone, CUDA events around each C-ABI call); value / e2e are the "
                                  "overlapped production path", "ms_per_step_serialized": r["ms_serial"]},
    }
    if second is not None:
        # BASELINE.json's other single-GPU configuration, same run, same timing rules (no per-entry breakdown)
        out["secondary"] = {"metric": metric, "config": {"workload": second["workload"], "cuda_graph": second["cuda_graph"]}, "value": second["value"], "unit": "clouds/s",
                            "ms_per_step": second["ms_per_step"], "e2e": second["e2e"], "gpu_launches": second["gpu_launches"],
                            "n_gpus": world, "steps": args.steps}
    if not args.no_cpu_baseline:
        out["cpu_baseline"] = cpu_arm(args.workload, 2)
    print(json.dumps(out))
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
