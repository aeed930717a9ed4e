#!/usr/bin/env python
"""bench.py -- ray-cell updates/s of the post-flight mapping path (BASELINE.json metric).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--workload c3|c4] [--configs all|none|c1,c4,..]
                    [--dump-outputs DIR]

One "step" = one pass of the hot path (P0 pose integration -> ray set-up -> grid replay) over one batch of
synthetic logs.  Headline workload: BASELINE config 3 AS WRITTEN -- the 4096-flight optical-flow drift ensemble
(3000 frames x 32 beams each, one 400x400 int8 grid per flight) sharded across the N GPUs (strong scaling:
4096 flights in total at every N, contiguous blocks per rank from uqs_flight_shard, one process per GPU, no
data-path collective).  `--workload c4` makes config 4 (one 16384^2 grid in owned row bands, one NCCL all-gather
inside the C library) the headline instead.

Printed JSON line (rank 0):
  value        whole-job ray-cell updates/s, inputs already resident in HBM, CUDA-event timed, max over ranks
  e2e          same metric through the C ABI with HOST (pinned) buffers: H2D of the logs and D2H of the grids
               inside the timed region; e2e.copy_floor_ms = the same call with its kernels switched off
  hash / hash_n1   64-bit digest of all result grids reduced over the ranks, and the digest of the same job
               replayed on rank 0's GPU alone in the same run: equal means the N-GPU result is the 1-GPU result
  roofline     replay kernel: algorithmic bytes per launch / its event-timed duration vs the measured HBM copy
               bandwidth (MEASURED_PEAKS.json); plus the measured on-chip RMW ceiling
  cpu_baseline the reference's own mapping code (oracle/_ref) on the box's host cores, bounded sample (N=1 only)
  configs      one record per BASELINE configuration c1..c5 at this N (value, e2e, hash[, hash_n1]); c3_weak is
               round 1's N x 4096-flight variant, kept for continuity
  --impl reference   times the reference CPU implementation as the main line (rank 0 only)

--dump-outputs DIR writes, after the timed steps, what the headline's last timed step computed as DIR/<name>.npy
(float32), so that two builds can be compared output for output on the same seeded logs:
  c3   grids [k, 400, 400] and poses x, y [k, 3000] of k = 64 flights drawn with a fixed seed from the ensemble (42 MB)
  c4   grid_rows [512, 16384]: 512 rows of the one grid drawn with a fixed seed (34 MB)
"""
from __future__ import annotations

import argparse
import importlib
import json
import multiprocessing as mp
import os
import statistics
import subprocess
import sys
import threading
import time
import traceback

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)
sys.dont_write_bytecode = True          # a run leaves the tree as it found it (it may be read-only)

METRIC = "ray_cell_updates_per_s"
DATA = "synthetic (seeded logs, SURVEY.md 8(d); ranges on the ToF sensor's 1 mm lattice like a real scan log)"
LOG_KEYS = ("t_ms", "of_rate_x", "of_rate_y", "h_m", "yaw_deg", "of_q", "ranges")
M64 = (1 << 64) - 1
DUMP_SEED = 20240607    # fixed: the sample --dump-outputs writes is the same in every run and at every N
DUMP_FLIGHTS = 64
DUMP_ROWS = 512


def describe(w, n_gpus, flights_total=None, scaling="strong"):
    F = flights_total if flights_total is not None else w.n_flights
    return {
        "workload": f"BASELINE config {w.config_id if w.config_id < 1000 else 5}: {w.name}",
        "flights_total": F, "flights_per_gpu": -(-F // n_gpus), "frames_per_flight": w.n_frames, "beams_per_frame": 32,
        "grid": f"{w.W}x{w.W}", "res_m": float(w.res),
        "parallelism": (f"{F} flights in contiguous blocks over {n_gpus} GPU(s) (uqs_flight_shard), no collective" if F > 1 else
                        "one grid"),
        "scaling": scaling,
        "l2_policy": "inputs (logs + ray records, >1.7 GB at full size) exceed the 126 MB L2; no flush needed",
    }


# ------------------------------------------------------------------------------------------------
# digests
# ------------------------------------------------------------------------------------------------
def _mix64(z: int) -> int:
    z = (z + 0x9E3779B97F4A7C15) & M64
    z = ((z ^ (z >> 30)) * 0xBF58476D1CE4E5B9) & M64
    z = ((z ^ (z >> 27)) * 0x94D049BB133111EB) & M64
    return z ^ (z >> 31)


def combine_hashes(per_grid: np.ndarray, first_id: int) -> int:
    """Order-independent digest of a set of grids: sum of mix(grid digest ^ mix(global id)) mod 2^64."""
    h = 0
    for i, g in enumerate(per_grid.tolist()):
        h = (h + _mix64(int(g) ^ _mix64(first_id + i))) & M64
    return h


def dump_sample(n: int, k: int) -> np.ndarray:
    """k of the indices [0, n), drawn with DUMP_SEED, ascending."""
    return np.sort(np.random.default_rng(DUMP_SEED).choice(n, size=min(k, n), replace=False))


def write_outputs(cx, out_dir, part):
    """Gather every rank's piece of the sample on rank 0 (shards are contiguous and in rank order, so the
    concatenation is in sample order) and write one float32 .npy per array."""
    parts = [part]
    if cx.world > 1:
        parts = [None] * cx.world if cx.rank == 0 else None
        cx.dist.gather_object(part, parts, dst=0)
    if cx.rank != 0:
        return
    os.makedirs(out_dir, exist_ok=True)
    for name in sorted({k for q in parts for k in q}):
        a = np.concatenate([q[name] for q in parts if name in q], axis=0).astype(np.float32, copy=False)
        np.save(os.path.join(out_dir, name + ".npy"), a)


# ------------------------------------------------------------------------------------------------
# CPU arm: the reference's own mapping code, one forked worker per host core
# ------------------------------------------------------------------------------------------------
_CPU_JOB = {}          # inherited by forked workers (no pickling of the logs)


def _cpu_worker(c, cores, barrier, ret):
    J = _CPU_JOB
    from oracle import orc
    o = orc.Oracle()
    W, res = J["W"], J["res"]
    ref = orc.Reference(W, W, res) if J["kind"] == "reference" else None
    p = importlib.import_module("micro-quad-slam_b200").make_params(W, W, float(res))
    t_ms, rx, ry, h, yaw, q, ranges = (J[k] for k in LOG_KEYS)
    barrier.wait()
    t0 = time.perf_counter()
    for f in range(c, J["n"], cores):
        px, py = o.pose_integrate(t_ms[f], rx[f], ry[f], h[f], yaw[f], q[f])      # P0 (builder-defined), CPU statement
        if ref is not None:
            ref.reset(0.0, 0.0)
            ref.L.ref_replay(px.size, px.ctypes.data, py.ctypes.data, yaw[f].ctypes.data, ranges[f].ctypes.data, 0)
        else:
            o.replay(p, px, py, yaw[f], ranges[f])
    ret[c] = time.perf_counter() - t0


def cpu_replay_rate(w, d, updates_per_flight, cores, flights_per_core):
    """Replay cores*flights_per_core flights of workload w, one forked process per core (the reference's
    static grid forbids threads).  Returns (updates/s, frames/s, kind, flights, processes, wall seconds)."""
    from oracle import orc
    kind = "reference" if os.path.exists(orc.ref_lib_path(w.W, w.W, w.res)) else "port"
    n = min(w.n_flights, cores * flights_per_core)
    cores = min(cores, n)
    _CPU_JOB.clear()
    _CPU_JOB.update({k: d[k] for k in LOG_KEYS})
    _CPU_JOB.update(W=w.W, res=w.res, kind=kind, n=n)
    ctx = mp.get_context("fork")
    barrier = ctx.Barrier(cores)
    ret = ctx.Array("d", cores)
    procs = [ctx.Process(target=_cpu_worker, args=(c, cores, barrier, ret)) for c in range(cores)]
    for pr in procs:
        pr.start()
    for pr in procs:
        pr.join()
    if any(pr.exitcode != 0 for pr in procs):
        raise RuntimeError("CPU baseline worker failed")
    wall = max(ret[:])
    return updates_per_flight * n / wall, n * w.n_frames / wall, kind, n, cores, wall


# ------------------------------------------------------------------------------------------------
# clocks during the timed region
# ------------------------------------------------------------------------------------------------
class ClockSampler:
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index):
        self.idx, self.proc, self.lines = gpu_index, None, []

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits", "-lms", "100",
                                          "-i", str(self.idx)], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.t = threading.Thread(target=lambda: self.lines.extend(self.proc.stdout), daemon=True)
            self.t.start()
        except OSError:
            self.proc = None

    def stop(self):
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.15)
        self.proc.terminate()
        self.t.join(timeout=2)
        sm, mx, reasons = [], [], set()
        for ln in self.lines:
            f = [x.strip() for x in ln.split(",")]
            if len(f) < 9:
                continue
            try:
                sm.append(float(f[1])); mx.append(float(f[2]))
            except ValueError:
                continue
            for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), f[5:9]):
                if v.lower().startswith("active"):
                    reasons.add(name)
        return {"sm_mhz": statistics.median(sm) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": sorted(reasons), "samples": len(sm)}


def bind_to_gpu_numa_node(gpu_index):
    """Run this rank (and its pinned allocations, by first touch) on the CPUs local to its GPU; on multi-socket
    boxes this keeps H2D/D2H traffic of the e2e path off the inter-socket link.  Best effort."""
    try:
        import pynvml
        pynvml.nvmlInit()
        h = pynvml.nvmlDeviceGetHandleByIndex(gpu_index)
        n_words = (os.cpu_count() + 63) // 64
        mask = pynvml.nvmlDeviceGetCpuAffinity(h, n_words)
        cpus = {64 * i + b for i, w in enumerate(mask) for b in range(64) if (w >> b) & 1}
        cpus &= os.sched_getaffinity(0)
        if cpus:
            os.sched_setaffinity(0, cpus)
            return len(cpus)
    except Exception:
        pass
    return None


def measured_hbm_peak():
    try:
        with open(os.path.join(ROOT, "MEASURED_PEAKS.json")) as f:
            return float(json.load(f)["hbm_gbs"]), "measured (MEASURED_PEAKS.json)"
    except Exception:
        return 6650.0, "fallback (B200_PROFILING.md)"


def recorded_capture(w, flights):
    """Figures of the committed ncu --set full capture of the replay kernel, when it is for this workload."""
    try:
        with open(os.path.join(ROOT, "profiles", "traffic.json")) as f:
            t = json.load(f)
        if t.get("workload") == w.name and t.get("flights") == flights and t.get("frames") == w.n_frames:
            return t
    except Exception:
        pass
    return {}


# ------------------------------------------------------------------------------------------------
def run_reference_arm(args, synth, out_fd):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    w = synth.on_mm_lattice(synth.CONFIGS["c3"])
    cores = os.cpu_count() or 1
    fpc = max(1, min(args.cpu_flights_per_core, max(1, w.n_flights // cores)))
    n = min(w.n_flights, cores * fpc)
    ws = synth.scaled(w, n_flights=n)
    d = synth.generate(ws)
    from oracle import orc
    o = orc.Oracle()
    # per-flight update counts differ slightly (drift); count them all once with the port (untimed)
    U = 0
    for f in range(n):
        px, py = o.pose_integrate(d["t_ms"][f], d["of_rate_x"][f], d["of_rate_y"][f], d["h_m"][f], d["yaw_deg"][f], d["of_q"][f])
        U += o.replay(ws.params(), px, py, d["frame_yaw_deg"][f], d["ranges"][f])[1]
    upf = U / n
    times, kind, used = [], "port", cores
    for i in range(args.warmup + args.steps):
        ups, fps, kind, nn, used, wall = cpu_replay_rate(ws, d, upf, cores, fpc)
        if i >= args.warmup:
            times.append(wall)
    wall = sum(times) / len(times)
    value = U / wall
    sample = f"{n} of {w.n_flights} flights per step ({fpc} per worker process), P0 + mapping, logs in RAM"
    cfg = describe(w, args.gpus)
    cfg["flights_replayed_per_step"] = n            # the CPU arm replays a bounded sample of the 4096 (the rate is what compares)
    cfg["parallelism"] = f"{used} forked worker processes on the host cores (the reference's static grid forbids threads)"
    out_fd.emit(json.dumps({
        "impl": "reference", "metric": METRIC, "value": value, "unit": "updates/s", "n_gpus": args.gpus, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": wall * 1e3, "higher_is_better": True, "scaling": "strong", "vs_baseline": None,
        "dtype": "i8", "data": DATA, "config": cfg, "frames_per_s": n * w.n_frames / wall,
        "cpu_baseline": {"value": value, "unit": "updates/s", "cores": used, "kind": kind, "sample": sample},
        "e2e": {"value": value, "unit": "updates/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
    }))


class OneLineStdout:
    """Everything any library prints to fd 1 (NCCL's version banner, ...) goes to stderr; only emit() writes to the
    real stdout -- the driver reads ONE JSON line from it."""

    def __init__(self):
        sys.stdout.flush()
        self.real = os.dup(1)
        os.dup2(2, 1)

    def emit(self, line: str):
        sys.stdout.flush()
        os.write(self.real, (line + "\n").encode())


# ------------------------------------------------------------------------------------------------
# the GPU arm
# ------------------------------------------------------------------------------------------------
class Ctx:
    """What every configuration's runner needs: the library, torch plumbing, rank geometry, timing helpers."""

    def __init__(self, args, m, synth):
        import torch
        import torch.distributed as dist
        self.args, self.m, self.synth, self.torch, self.dist = args, m, synth, torch, dist
        self.world = int(os.environ.get("WORLD_SIZE", "1"))
        self.rank = int(os.environ.get("RANK", "0"))
        self.local = int(os.environ.get("LOCAL_RANK", "0"))
        if args.gpus != self.world:
            raise SystemExit(f"--gpus {args.gpus} but WORLD_SIZE={self.world}: launch with python -m torch.distributed.run "
                             f"--nnodes=1 --nproc-per-node {args.gpus} --master-addr 127.0.0.1 bench.py --gpus {args.gpus}")
        torch.cuda.set_device(self.local)
        self.dev = torch.device("cuda", self.local)
        self.local_cpus = bind_to_gpu_numa_node(self.local) if self.world > 1 else None
        if self.world > 1:
            import datetime
            # a rank that dies inside one configuration must not leave the others waiting for ever
            dist.init_process_group("nccl", device_id=self.dev, timeout=datetime.timedelta(seconds=240))
        m.init(self.local)                                   # fails loudly if the CUDA library cannot run
        m.set_stream(torch.cuda.current_stream().cuda_stream)
        m.set_engine(args.engine, args.flight_warps)
        self.e0, self.e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        self.comm_ready = False

    def barrier(self):
        if self.world > 1:
            self.dist.barrier()
        self.torch.cuda.synchronize()

    def max_over_ranks(self, v: float) -> float:
        if self.world == 1:
            return float(v)
        t = self.torch.tensor([float(v)], dtype=self.torch.float64, device=self.dev)
        self.dist.all_reduce(t, op=self.dist.ReduceOp.MAX)
        return float(t.item())

    def sum_over_ranks(self, v: float) -> float:
        if self.world == 1:
            return float(v)
        t = self.torch.tensor([float(v)], dtype=self.torch.float64, device=self.dev)
        self.dist.all_reduce(t)
        return float(t.item())

    def sum_hash(self, h: int) -> int:
        """sum mod 2^64 of one digest per rank (exact: four 16-bit limbs through an int64 all-reduce)."""
        if self.world == 1:
            return h & M64
        t = self.torch.tensor([(h >> (16 * i)) & 0xFFFF for i in range(4)], dtype=self.torch.int64, device=self.dev)
        self.dist.all_reduce(t)
        limbs = t.tolist()
        return sum(int(v) << (16 * i) for i, v in enumerate(limbs)) & M64

    def all_equal(self, h: int) -> bool:
        if self.world == 1:
            return True
        t = self.torch.tensor([(h >> 32) & 0xFFFFFFFF, h & 0xFFFFFFFF], dtype=self.torch.int64, device=self.dev)
        lo, hi = t.clone(), t.clone()
        self.dist.all_reduce(lo, op=self.dist.ReduceOp.MIN)
        self.dist.all_reduce(hi, op=self.dist.ReduceOp.MAX)
        return bool(self.torch.equal(lo, hi))

    def all_true(self, ok: bool) -> bool:
        if self.world == 1:
            return bool(ok)
        t = self.torch.tensor([1 if ok else 0], dtype=self.torch.int64, device=self.dev)
        self.dist.all_reduce(t, op=self.dist.ReduceOp.MIN)
        return bool(t.item())

    def free_host_cache(self):
        """torch keeps freed pinned blocks; the configurations use different sizes, so give them back in between."""
        try:
            self.torch.cuda.empty_cache()
            self.torch._C._host_emptyCache()
        except Exception:
            pass

    def timed(self, fn, steps, warmup):
        """ms per step on the device (CUDA events on the launching stream), max over ranks."""
        for _ in range(warmup):
            fn()
        self.barrier()
        self.e0.record()
        for _ in range(steps):
            fn()
        self.e1.record()
        self.barrier()
        return self.max_over_ranks(self.e0.elapsed_time(self.e1)) / steps

    def timed_host(self, fn, steps, warmup):
        """ms per step of a synchronous host-buffer call: max(device events, host wall clock), max over ranks."""
        for _ in range(warmup):
            fn()
        self.barrier()
        t0 = time.perf_counter()
        self.e0.record()
        for _ in range(steps):
            fn()
        self.e1.record()
        self.barrier()
        return self.max_over_ranks(max(self.e0.elapsed_time(self.e1), (time.perf_counter() - t0) * 1e3)) / steps

    def pinned(self, shape, dt):
        return self.torch.empty(shape, dtype=dt, pin_memory=True)

    def ensure_comm(self):
        """The library's own NCCL communicator (uqs_comm_init_rank); the 128-byte id travels over torch.distributed."""
        if self.comm_ready or self.world == 1:
            return
        t = self.torch.zeros(self.m.COMM_ID_BYTES, dtype=self.torch.uint8, device=self.dev)
        if self.rank == 0:
            t.copy_(self.torch.frombuffer(bytearray(self.m.comm_unique_id()), dtype=self.torch.uint8))
        self.dist.broadcast(t, 0)
        self.m.comm_init_rank(t.cpu().numpy().tobytes(), self.world, self.rank)
        self.comm_ready = True


def host_logs(cx, F, N, NF):
    t = cx.torch
    host = {"t_ms": cx.pinned((F, N), t.int32), "of_rate_x": cx.pinned((F, N), t.float32), "of_rate_y": cx.pinned((F, N), t.float32),
            "h_m": cx.pinned((F, N), t.float32), "yaw_deg": cx.pinned((F, N), t.float32), "of_q": cx.pinned((F, N), t.uint8),
            "ranges": cx.pinned((F, NF, 32), t.float32), "x_true": cx.pinned((F, N), t.float32), "y_true": cx.pinned((F, N), t.float32)}
    views = {k: v.numpy() for k, v in host.items()}
    views["t_ms"] = views["t_ms"].view(np.uint32)
    return host, views


def run_flights(cx, w, first, cnt, total, label, verify_n1, headline=False, variants=False):
    """A flow-driven many-flight workload (configs 3 and 1/2 with total == 1): this rank replays flights
    [first, first+cnt) of `total`.  Returns the record; the headline call also returns roofline / launch details."""
    m, synth, torch, args = cx.m, cx.synth, cx.torch, cx.args
    p = w.params()
    F, N, NF = cnt, w.n_samples, w.n_frames
    rec = {"workload": f"BASELINE config {w.config_id}: {w.name}", "flights_total": total, "flights_this_rank": F,
           "frames_per_flight": NF, "grid": f"{p.W}x{p.H}", "label": label}
    active = F > 0
    U = 0
    steps, warmup = (args.steps, args.warmup) if headline else (max(2, min(args.steps, 3)), 2)
    if active:
        host, d = host_logs(cx, F, N, NF)
        d = synth.generate(synth.scaled(w, n_flights=F), flight_id0=first, n_flights=F, out=dict(d))
        h_grids = cx.pinned((F, p.H, p.W), torch.int8)
        dv = {k: host[k].to(cx.dev, non_blocking=True) for k in LOG_KEYS}
        d_x = torch.empty((F, N), dtype=torch.float32, device=cx.dev)
        d_y = torch.empty((F, N), dtype=torch.float32, device=cx.dev)
        d_grids = torch.empty((F, p.H, p.W), dtype=torch.int8, device=cx.dev)
        torch.cuda.synchronize()

        def step_device(want_stats=False, mode=0):
            m.pose_integrate_dev(F, N, dv["t_ms"].data_ptr(), dv["of_rate_x"].data_ptr(), dv["of_rate_y"].data_ptr(), dv["h_m"].data_ptr(),
                                 dv["yaw_deg"].data_ptr(), dv["of_q"].data_ptr(), d_x.data_ptr(), d_y.data_ptr(), mode)
            return m.replay_dev(p, F, NF, d_x.data_ptr(), d_y.data_ptr(), dv["yaw_deg"].data_ptr(), dv["ranges"].data_ptr(),
                                d_grids.data_ptr(), want_stats=want_stats)

        def step_e2e():
            m.replay_flow(p, d["t_ms"], d["of_rate_x"], d["of_rate_y"], d["h_m"], d["yaw_deg"], d["of_q"], d["ranges"],
                          want_poses=False, out=h_grids.numpy())
        U = step_device(want_stats=True)["ray_cell_updates"]
    else:
        def step_device(want_stats=False, mode=0):
            return None

        def step_e2e():
            return None
    total_U = cx.sum_over_ranks(U)

    clocks = ClockSampler(cx.local) if (headline and cx.rank == 0) else None
    if clocks:
        clocks.start()
    if active:
        for _ in range(max(warmup - 1, 0)):
            step_device()
        m.set_profiling(True)
        m.profile_collect()
    l0 = m.kernel_launches()
    ms = cx.timed(step_device, steps, 0)
    launches = m.kernel_launches() - l0
    outputs = {}
    if headline and args.dump_outputs and active:
        # what the last timed step left on the device, for the flights of the fixed sample that this rank holds
        ids = dump_sample(total, DUMP_FLIGHTS)
        mine = torch.as_tensor(ids[(ids >= first) & (ids < first + F)] - first, dtype=torch.long, device=cx.dev)
        outputs = {"grids": d_grids[mine].float().cpu().numpy(), "x": d_x[mine].cpu().numpy(), "y": d_y[mine].cpu().numpy()}
    kms = [0.0, 0.0, 0.0]
    if active:
        kms, _ = m.profile_collect()
        m.set_profiling(False)
    rec.update(value=total_U / (ms * 1e-3), unit="updates/s", ms_per_step=ms, updates=total_U,
               frames_per_s=total * NF / (ms * 1e-3), steps=steps, warmup=warmup,
               kernel_ms={"pose": kms[0] / steps, "ray_setup": kms[1] / steps, "replay": kms[2] / steps},
               what="P0 + ray set-up + replay, logs resident in HBM")

    # digests of the device-resident result
    h = combine_hashes(m.grid_hashes_dev(d_grids.data_ptr(), F, p.W * p.H), first) if active else 0
    rec["hash"] = f"{cx.sum_hash(h):016x}"

    # ---- e2e: the C-ABI call with host buffers, H2D + D2H inside the timed region ---------------------------------
    if not args.no_e2e:
        e_ms = cx.timed_host(step_e2e, steps, 1)
        h2d = sum(d[k].nbytes for k in LOG_KEYS) if active else 0
        rec["e2e"] = {"value": total_U / (e_ms * 1e-3), "unit": "updates/s", "ms_per_step": e_ms,
                      "h2d_bytes_per_step": int(cx.sum_over_ranks(h2d)), "d2h_bytes_per_step": int(cx.sum_over_ranks(F * p.W * p.H)),
                      "api": "uqs_replay_flow (host pointers, pinned), every rank on its shard"}
        # the grids the host-buffer call returned must be the device-resident ones (recorded, and agreed on by all ranks)
        rec["e2e"]["matches_device_result"] = cx.all_true(not active or bool(torch.equal(h_grids, d_grids.cpu())))
        # the same call with its kernels switched off: what the copies alone cost on this box at this N
        if active:
            m.set_copy_only(True)
        try:
            rec["e2e"]["copy_floor_ms"] = cx.timed_host(step_e2e, steps, 1)
        finally:
            if active:
                m.set_copy_only(False)
        if variants:
            # other forms of the same call: ranges as the sensor's u16 millimetres (half the H2D bytes), and boxed output
            # (only each flight's touched box comes back).  Same logs, same grids.
            if active:
                mm = cx.pinned((F, NF, 32), torch.int16)
                mm_np = mm.numpy().view(np.uint16)
                synth.ranges_to_mm(d["ranges"], out=mm_np)
                boxes = cx.pinned((F, 4), torch.int32)
                offs = cx.pinned((F,), torch.int64)
                packed = cx.pinned((max(F * p.W * p.H // 2, 1 << 20),), torch.int8)
                flow = (d["t_ms"], d["of_rate_x"], d["of_rate_y"], d["h_m"], d["yaw_deg"], d["of_q"])

                def step_mm():
                    m.replay_flow_mm(p, *flow, mm_np, want_poses=False, out=h_grids.numpy())

                def step_mm_boxed():
                    return m.replay_flow_boxed(p, *flow, ranges_mm=mm_np, packed=packed.numpy(), boxes=boxes.numpy(),
                                               offsets=offs.numpy().view(np.uint64))
            else:
                step_mm = step_mm_boxed = lambda: None
            h_grids.zero_() if active else None
            mm_ms = cx.timed_host(step_mm, steps, 1)
            ok_mm = not active or bool(torch.equal(h_grids, d_grids.cpu()))
            box_ms = cx.timed_host(step_mm_boxed, steps, 1)
            used = 0
            ok_box = True
            if active:
                _, _, _, used, _ = step_mm_boxed()
                dense = m.unpack_boxed(p, boxes.numpy(), offs.numpy().view(np.uint64), packed.numpy(), out=h_grids.numpy())
                ok_box = bool(torch.equal(torch.from_numpy(dense), d_grids.cpu()))
            h2d_mm = (sum(d[k].nbytes for k in LOG_KEYS[:-1]) + mm.numel() * 2) if active else 0
            rec["e2e_variants"] = {
                "mm": {"value": total_U / (mm_ms * 1e-3), "ms_per_step": mm_ms, "h2d_bytes_per_step": int(cx.sum_over_ranks(h2d_mm)),
                       "d2h_bytes_per_step": int(cx.sum_over_ranks(F * p.W * p.H)), "matches_device_result": cx.all_true(ok_mm),
                       "api": "uqs_replay_flow_mm: ranges as u16 millimetres (uav_local_nav.c:1328 on the device), dense grids out"},
                "mm_boxed": {"value": total_U / (box_ms * 1e-3), "ms_per_step": box_ms, "h2d_bytes_per_step": int(cx.sum_over_ranks(h2d_mm)),
                             "d2h_bytes_per_step": int(cx.sum_over_ranks(used + F * 24)), "matches_device_result": cx.all_true(ok_box),
                             "api": "uqs_replay_flow_boxed: u16 millimetres in, each flight's touched box out (expanded and compared outside the timed region)"}}
    clk = clocks.stop() if clocks else None

    # ---- the same job on ONE GPU (rank 0 alone), for the cross-N identity of the result -----------------------------
    if verify_n1 and cx.world > 1:
        h1 = 0
        if cx.rank == 0:
            blk = 1024
            for f0 in range(0, total, blk):
                nf = min(blk, total - f0)
                db = synth.generate(synth.scaled(w, n_flights=nf), flight_id0=f0, n_flights=nf)
                tv = {k: torch.from_numpy(db[k].view(np.int32) if k == "t_ms" else db[k]).to(cx.dev) for k in LOG_KEYS}
                bx = torch.empty((nf, N), dtype=torch.float32, device=cx.dev)
                by = torch.empty_like(bx)
                bg = torch.empty((nf, p.H, p.W), dtype=torch.int8, device=cx.dev)
                m.pose_integrate_dev(nf, N, tv["t_ms"].data_ptr(), tv["of_rate_x"].data_ptr(), tv["of_rate_y"].data_ptr(), tv["h_m"].data_ptr(),
                                     tv["yaw_deg"].data_ptr(), tv["of_q"].data_ptr(), bx.data_ptr(), by.data_ptr(), 0)
                m.replay_dev(p, nf, NF, bx.data_ptr(), by.data_ptr(), tv["yaw_deg"].data_ptr(), tv["ranges"].data_ptr(), bg.data_ptr())
                h1 = (h1 + combine_hashes(m.grid_hashes_dev(bg.data_ptr(), nf, p.W * p.H), f0)) & M64
        cx.barrier()
        rec["hash_n1"] = f"{cx.sum_hash(h1):016x}"
        rec["hash_matches_n1"] = rec["hash_n1"] == rec["hash"]
    extra = {"U_rank": U, "kms": kms, "launches": int(launches), "clocks": clk, "steps": steps,
             "d_pinned": d if (active and headline) else None, "F": F, "outputs": outputs}
    return rec, extra


def run_p0_variants(cx, w):
    """P0 alone on one long log: the exact-order chain (mode 0, what every grid above is computed from) and the
    look-back scan (mode 1).  Rank 0."""
    m, synth, torch = cx.m, cx.synth, cx.torch
    d = synth.generate(w)
    tv = {k: torch.from_numpy(d[k].view(np.int32) if k == "t_ms" else d[k]).to(cx.dev) for k in LOG_KEYS[:-1]}
    F, N = w.n_flights, w.n_samples
    bx = torch.empty((F, N), dtype=torch.float32, device=cx.dev)
    by = torch.empty_like(bx)
    out = {}
    for mode, name in ((0, "chain_exact_order_ms"), (1, "lookback_scan_ms")):
        def go():
            m.pose_integrate_dev(F, N, tv["t_ms"].data_ptr(), tv["of_rate_x"].data_ptr(), tv["of_rate_y"].data_ptr(), tv["h_m"].data_ptr(),
                                 tv["yaw_deg"].data_ptr(), tv["of_q"].data_ptr(), bx.data_ptr(), by.data_ptr(), mode)
        for _ in range(3):
            go()
        torch.cuda.synchronize()
        cx.e0.record()
        for _ in range(5):
            go()
        cx.e1.record()
        torch.cuda.synchronize()
        out[name] = cx.e0.elapsed_time(cx.e1) / 5
    out["samples"] = N
    return out


def run_c4(cx, verify_n1, headline=False):
    """Config 4: ONE 16384^2 grid; every rank owns a band of rows (uqs_row_band), replays the whole log into it,
    one ncclAllGather inside the library assembles the grid on every rank."""
    m, synth, torch, args = cx.m, cx.synth, cx.torch, cx.args
    w = synth.on_mm_lattice(synth.CONFIGS["c4"] if not args.c4_samples else synth.scaled(synth.CONFIGS["c4"], n_samples=args.c4_samples))
    p = w.params()
    d = synth.generate(w)                                  # every rank holds the whole log (it reads the same file)
    x, y = synth.frame_poses(d, d["x_true"], d["y_true"])
    NF = w.n_frames
    cx.ensure_comm()
    hp = {k: cx.pinned((NF,) + ((32,) if k == "ranges" else ()), torch.float32) for k in ("x", "y", "yaw", "ranges")}
    hp["x"].numpy()[:] = x[0]; hp["y"].numpy()[:] = y[0]; hp["yaw"].numpy()[:] = d["frame_yaw_deg"][0]; hp["ranges"].numpy()[:] = d["ranges"][0]
    dv = {k: v.to(cx.dev, non_blocking=True) for k, v in hp.items()}
    grid = torch.empty((p.H, p.W), dtype=torch.int8, device=cx.dev)
    h_grid = cx.pinned((p.H, p.W), torch.int8) if cx.rank == 0 else None
    torch.cuda.synchronize()
    steps, warmup = (args.steps, args.warmup) if headline else (max(2, min(args.steps, 3)), 2)

    def step_device(want_stats=False, gather=True):
        return m.replay_banded_dev(p, NF, dv["x"].data_ptr(), dv["y"].data_ptr(), dv["yaw"].data_ptr(), dv["ranges"].data_ptr(),
                                   grid.data_ptr(), gather=gather, want_stats=want_stats)

    def step_e2e():
        m.replay_banded(p, hp["x"].numpy(), hp["y"].numpy(), hp["yaw"].numpy(), hp["ranges"].numpy(),
                        out=h_grid.numpy() if h_grid is not None else None, want_grid=h_grid is not None)

    st = step_device(want_stats=True)
    U = st["ray_cell_updates"]
    for _ in range(warmup - 1):
        step_device()
    m.set_profiling(True)
    m.profile_collect()
    l0 = m.kernel_launches()
    ms = cx.timed(step_device, steps, 0)
    launches = m.kernel_launches() - l0
    outputs = {}
    if headline and args.dump_outputs and cx.rank == 0:
        # every rank holds the whole grid after the gather; rank 0 writes the fixed sample of its rows
        rows = torch.as_tensor(dump_sample(p.H, DUMP_ROWS), dtype=torch.long, device=cx.dev)
        outputs = {"grid_rows": grid[rows].float().cpu().numpy()}
    kms, _ = m.profile_collect()
    m.set_profiling(False)
    # the same step without the exchange (what the NCCL gather of the bands costs), and every rank's own kernel time
    ms_nogather = cx.timed(lambda: step_device(gather=False), steps, 0) if cx.world > 1 else ms
    per_rank = [0.0] * cx.world
    per_rank[cx.rank] = (kms[1] + kms[2]) / steps
    if cx.world > 1:
        tr = torch.tensor(per_rank, dtype=torch.float64, device=cx.dev)
        cx.dist.all_reduce(tr)
        per_rank = tr.tolist()
    edges = m.band_edges()
    hh = int(m.grid_hashes_dev(grid.data_ptr(), 1, p.W * p.H)[0])
    rec = {"workload": f"BASELINE config 4: {w.name}", "samples": w.n_samples, "frames": NF, "beams_per_sample": 64,
           "grid": f"{p.W}x{p.H}", "value": U / (ms * 1e-3), "unit": "updates/s", "ms_per_step": ms, "updates": U,
           "frames_per_s": NF / (ms * 1e-3), "steps": steps, "warmup": warmup,
           "kernel_ms_rank0": {"ray_setup": kms[1] / steps, "replay": kms[2] / steps},
           "kernel_ms_per_rank": [round(v, 3) for v in per_rank], "ms_per_step_without_gather": ms_nogather,
           "partition": f"{cx.world} owned row bands cut at rows {edges} (equal shares of the log: origin-row histogram widened by the "
                        "sensor's reach, computed on the device every call)", "exchange": "one ncclAllGather of the bands inside libuqs_mapping, in the timed region",
           "comm_nranks_seen": [m.comm_nranks()], "nccl_version": m.nccl_version() if cx.world > 1 else None,
           "what": "ray set-up + band replay + band all-gather, log resident in HBM on every rank",
           "hash": f"{hh:016x}", "hash_identical_on_every_rank": cx.all_equal(hh), "gpu_launches": int(launches)}
    if not args.no_e2e:
        e_ms = cx.timed_host(step_e2e, steps, 1)
        log_bytes = sum(v.numel() * 4 for v in hp.values())
        rec["e2e"] = {"value": U / (e_ms * 1e-3), "unit": "updates/s", "ms_per_step": e_ms, "h2d_bytes_per_step": int(log_bytes),
                      "d2h_bytes_per_step": int(p.W * p.H),
                      "api": "uqs_replay_banded (host pointers, pinned): each rank uploads 1/N of the log, log all-gather over NVLink, "
                             "band replay, band all-gather, whole grid D2H on rank 0"}
        rec["e2e"]["matches_device_result"] = cx.all_true(cx.rank != 0 or m.grid_hash(h_grid.numpy()) == hh)
    if verify_n1 and cx.world > 1:
        h1 = 0
        if cx.rank == 0:
            g1 = torch.empty_like(grid)
            m.replay_dev(p, 1, NF, dv["x"].data_ptr(), dv["y"].data_ptr(), dv["yaw"].data_ptr(), dv["ranges"].data_ptr(), g1.data_ptr())
            h1 = int(m.grid_hashes_dev(g1.data_ptr(), 1, p.W * p.H)[0])
        cx.barrier()
        rec["hash_n1"] = f"{cx.sum_hash(h1):016x}"
        rec["hash_matches_n1"] = rec["hash_n1"] == rec["hash"]
    extra = {"U_rank": U, "kms": kms, "launches": int(launches), "steps": steps, "n_rays": NF * 32, "n_frames": NF, "cells": p.W * p.H,
             "outputs": outputs}
    return rec, extra


def run_c5(cx, verify_n1):
    """Config 5: 16 resolutions x 16 range-noise levels x 64 flights = 16384 flights, one grid per flight.  The 1024
    flights of a resolution share the grid geometry and are one call; every rank takes a contiguous block of each
    resolution's 1024 (uqs_flight_shard), so all ranks see the same mix of cheap and expensive geometries."""
    m, synth, torch, args = cx.m, cx.synth, cx.torch, cx.args
    steps = 2
    tot_ms = tot_e_ms = 0.0
    tot_U = 0
    h_all = h1_all = 0
    h2d = d2h = 0
    per_res = []
    n_res = len(synth.C5_RES) if not args.c5_resolutions else args.c5_resolutions

    def gen_block(ir, a, n):
        """flights [a, a+n) of resolution ir's 1024 (global index = sigma*64 + seed)."""
        parts, g = [], a
        while g < a + n:
            isg, f0 = divmod(g, 64)
            k = min(64 - f0, a + n - g)
            wc = synth.on_mm_lattice(synth.c5_workload(ir, isg, n_flights=k))
            parts.append(synth.generate(wc, flight_id0=f0, n_flights=k))
            g += k
        cat = lambda key: np.ascontiguousarray(np.concatenate([q[key] for q in parts], axis=0))
        return {k: cat(k) for k in ("x_true", "y_true", "frame_yaw_deg", "ranges")}

    first, cnt = m.flight_shard(1024, cx.rank, cx.world)
    w_max = max(synth.c5_width(r) for r in synth.C5_RES[:n_res])
    if cnt:             # one pinned set for all resolutions (only the grid size changes)
        hp = {"x_true": cx.pinned((cnt, 3000), torch.float32), "y_true": cx.pinned((cnt, 3000), torch.float32),
              "frame_yaw_deg": cx.pinned((cnt, 3000), torch.float32), "ranges": cx.pinned((cnt, 3000, 32), torch.float32)}
        hg_all = cx.pinned((cnt * w_max * w_max,), torch.int8)
    for ir in range(n_res):
        w0 = synth.c5_workload(ir, 0)
        p = w0.params()
        NF = w0.n_frames
        ms_r = e_r = 0.0
        U = 0
        if cnt:
            db = gen_block(ir, first, cnt)
            for k in db:
                hp[k].numpy()[:] = db[k]
            tv = {k: v.to(cx.dev, non_blocking=True) for k, v in hp.items()}
            g = torch.empty((cnt, p.H, p.W), dtype=torch.int8, device=cx.dev)
            hg = hg_all[:cnt * p.H * p.W].view(cnt, p.H, p.W)

            def go(want_stats=False):
                return m.replay_dev(p, cnt, NF, tv["x_true"].data_ptr(), tv["y_true"].data_ptr(), tv["frame_yaw_deg"].data_ptr(),
                                    tv["ranges"].data_ptr(), g.data_ptr(), want_stats=want_stats)
            U = go(want_stats=True)["ray_cell_updates"]
            go()
            torch.cuda.synchronize()
            cx.e0.record()
            for _ in range(steps):
                go()
            cx.e1.record()
            torch.cuda.synchronize()
            ms_r = cx.e0.elapsed_time(cx.e1) / steps
            h_all = (h_all + combine_hashes(m.grid_hashes_dev(g.data_ptr(), cnt, p.W * p.H), ir * 1024 + first)) & M64
            if not args.no_e2e:
                def e2e():
                    m.replay(p, hp["x_true"].numpy(), hp["y_true"].numpy(), hp["frame_yaw_deg"].numpy(), hp["ranges"].numpy(), out=hg.numpy())
                e2e()
                t0 = time.perf_counter()
                for _ in range(steps):
                    e2e()
                e_r = (time.perf_counter() - t0) * 1e3 / steps
                h2d += sum(v.numel() * 4 for v in hp.values())
                d2h += hg.numel()
            del tv, g
        tot_ms += ms_r
        tot_e_ms += e_r
        tot_U += U
        per_res.append({"res_m": float(w0.res), "grid": p.W, "ms_this_rank": round(ms_r, 3)})
        if verify_n1 and cx.world > 1 and cx.rank == 0:
            db = gen_block(ir, 0, 1024)
            tv = {k: torch.from_numpy(db[k]).to(cx.dev) for k in db}
            g = torch.empty((1024, p.H, p.W), dtype=torch.int8, device=cx.dev)
            m.replay_dev(p, 1024, NF, tv["x_true"].data_ptr(), tv["y_true"].data_ptr(), tv["frame_yaw_deg"].data_ptr(), tv["ranges"].data_ptr(), g.data_ptr())
            h1_all = (h1_all + combine_hashes(m.grid_hashes_dev(g.data_ptr(), 1024, p.W * p.H), ir * 1024)) & M64
            del tv, g
    cx.barrier()
    ms = cx.max_over_ranks(tot_ms)
    U_all = cx.sum_over_ranks(tot_U)
    rec = {"workload": "BASELINE config 5: 16 resolutions x 16 range-noise levels x 64 flights, one grid per (config, flight)",
           "flights_total": 1024 * n_res, "resolutions": n_res, "frames_per_flight": 3000, "value": U_all / (ms * 1e-3), "unit": "updates/s",
           "ms_per_step": ms, "updates": U_all, "frames_per_s": 1024 * n_res * 3000 / (ms * 1e-3), "steps": steps, "warmup": 2,
           "partition": "every rank takes a contiguous block of each resolution's 1024 flights (uqs_flight_shard); no collective",
           "what": "ray set-up + replay from poses resident in HBM, one call per resolution; time = sum over the 16 calls, max over ranks",
           "per_resolution_rank0": per_res, "hash": f"{cx.sum_hash(h_all):016x}"}
    if not args.no_e2e:
        e_ms = cx.max_over_ranks(tot_e_ms)
        rec["e2e"] = {"value": U_all / (e_ms * 1e-3), "unit": "updates/s", "ms_per_step": e_ms, "h2d_bytes_per_step": int(cx.sum_over_ranks(h2d)),
                      "d2h_bytes_per_step": int(cx.sum_over_ranks(d2h)), "api": "uqs_replay (host pointers, pinned), one call per resolution"}
    if verify_n1 and cx.world > 1:
        rec["hash_n1"] = f"{cx.sum_hash(h1_all):016x}"
        rec["hash_matches_n1"] = rec["hash_n1"] == rec["hash"]
    return rec


def guarded(cx, name, fn):
    """A secondary configuration must never cost the headline line: failures are recorded, not raised.  (Parity checks
    do not raise -- they are recorded booleans agreed on by all ranks -- so what lands here is an infrastructure
    error; if it hits one rank only, the process-group timeout ends the run instead of a hang.)"""
    try:
        return fn()
    except Exception as e:                          # noqa: BLE001
        traceback.print_exc()
        return {"error": f"{type(e).__name__}: {e}"}
    finally:
        cx.free_host_cache()


def main():
    out_fd = OneLineStdout()
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--workload", default="c3", choices=["c3", "c4"], help="the headline configuration")
    ap.add_argument("--configs", default="all", help="secondary records: all, none or a comma list of c1,c2,c3_weak,c4,c5")
    ap.add_argument("--flights", type=int, default=0, help="total flights of the config-3 ensemble (default 4096)")
    ap.add_argument("--c4-samples", type=int, default=0, help="config-4 log length (default 1 048 576 samples)")
    ap.add_argument("--c5-resolutions", type=int, default=0, help="config 5: only the first k resolutions (default all 16)")
    ap.add_argument("--cpu-flights-per-core", type=int, default=48)
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--no-verify-n1", action="store_true", help="skip replaying every job on rank 0 alone for hash_n1")
    ap.add_argument("--engine", type=int, default=0, help="0 auto, 1 sub-tiles, 2 resident (tuning experiments)")
    ap.add_argument("--flight-warps", type=int, default=0, help="warps per resident CTA (0 = library default)")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write a fixed sample of what the headline's last timed step computed to DIR/<name>.npy")
    args = ap.parse_args()
    args.warmup = max(args.warmup, 3) if args.impl == "ours" else args.warmup

    m = importlib.import_module("micro-quad-slam_b200")
    synth = importlib.import_module("micro-quad-slam_b200.synth")
    if args.impl == "reference":
        run_reference_arm(args, synth, out_fd)
        return

    cx = Ctx(args, m, synth)
    world, rank = cx.world, cx.rank
    verify = not args.no_verify_n1
    want = {"c1", "c2", "c3_weak", "c4", "c5"} if args.configs == "all" else (set() if args.configs == "none" else set(args.configs.split(",")))
    # every bench log carries its ranges on the sensor's millimetre lattice (float and u16 forms are then the same log)
    w3 = synth.on_mm_lattice(synth.CONFIGS["c3"] if not args.flights else synth.scaled(synth.CONFIGS["c3"], n_flights=args.flights))
    configs = {}

    # ---- headline ---------------------------------------------------------------------------------------------------------
    if args.workload == "c3":
        first, cnt = m.flight_shard(w3.n_flights, rank, world)
        head, ex = run_flights(cx, w3, first, cnt, w3.n_flights, "c3 strong: the ensemble sharded over the ranks", verify, headline=True,
                               variants=True)
        configs["c3"] = head
        cfg = describe(w3, world)
        F_rank, NF = ex["F"], w3.n_frames
        n_rays, n_frames_r, cells = F_rank * NF * 32, F_rank * NF, w3.W * w3.W * F_rank
        kernel_name = "k_replay_flights (resident engine)"
    else:
        head, ex = run_c4(cx, verify, headline=True)
        configs["c4"] = head
        w4 = synth.CONFIGS["c4"]
        cfg = {"workload": head["workload"], "samples": head["samples"], "frames": head["frames"], "beams_per_sample": 64,
               "grid": head["grid"], "res_m": float(w4.res), "parallelism": head["partition"] + "; " + head["exchange"],
               "scaling": "strong", "l2_policy": "log + ray records (>800 MB) exceed the 126 MB L2; no flush needed"}
        n_rays, n_frames_r, cells = ex["n_rays"], ex["n_frames"], ex["cells"] // world
        kernel_name = "k_replay_tiles (sub-tile engine, owned row band)"

    if args.dump_outputs:
        write_outputs(cx, args.dump_outputs, ex["outputs"])
    ex["outputs"] = None

    # ---- roofline of the dominant kernel (replay), rank 0's share of the job -----------------------------------------------
    roofline = cpu = None
    if rank == 0:
        peak, peak_src = measured_hbm_peak()
        U_r = ex["U_rank"]
        b_alg = 2 * U_r + 8 * n_rays + 16 * n_frames_r + cells             # per replay launch(es) of one step, this rank
        replay_ms = ex["kms"][2] / max(ex["steps"], 1)
        achieved = b_alg / (replay_ms * 1e-3) / 1e9 if replay_ms > 0 else 0.0
        rmw_peak = m.measure_rmw_peak()
        atoms_peak = m.measure_atoms_peak()
        cap = recorded_capture(w3, ex.get("F")) if args.workload == "c3" else {}
        roofline = {"bound": "hbm", "kernel": kernel_name, "achieved": achieved, "peak": peak, "unit": "GB/s",
                    "frac": achieved / peak, "peak_source": peak_src, "traffic": cap.get("dram_bytes_per_launch"),
                    "algorithmic_bytes_per_step": int(b_alg), "kernel_ms_per_step": replay_ms,
                    "kernel_share_of_step": replay_ms / head["ms_per_step"],
                    "setup_kernel_ms_per_step": ex["kms"][1] / ex["steps"], "pose_kernels_ms_per_step": ex["kms"][0] / ex["steps"],
                    "smem_pipe_recorded": {"pct_of_peak": cap.get("smem_pipe_pct_of_peak"), "issue_slots_pct": cap.get("issue_slots_pct_of_peak"),
                                           "l2_gbs": cap.get("l2_gbs"), "capture": cap.get("capture"),
                                           "note": "shared-memory wavefronts of the replay kernel in the committed ncu --set full capture: "
                                                   "the pipe this kernel is bound by"},
                    "onchip_rmw": {"achieved_updates_per_s": U_r / (replay_ms * 1e-3) if replay_ms > 0 else 0.0, "peak_updates_per_s": rmw_peak,
                                   "frac": (U_r / (replay_ms * 1e-3) / rmw_peak) if replay_ms > 0 else 0.0,
                                   "atomics_updates_per_s": atoms_peak,
                                   "note": "peak = conflict-free shared-memory byte load/clamp/store microbenchmark on this GPU; "
                                           "atomics_updates_per_s = the same pattern with one ATOMS.ADD per update (the rejected design)"}}

        if not args.no_cpu_baseline and world == 1 and args.workload == "c3":
            d = ex["d_pinned"]
            cores = os.cpu_count() or 1
            F = ex["F"]
            fpc = max(1, min(args.cpu_flights_per_core, max(1, F // cores)))
            ns = min(F, cores * fpc)
            # pageable copies of the sample: CUDA-pinned pages are not inherited by forked workers
            ds = {k: np.array(d[k][:ns]) for k in LOG_KEYS}
            ups, fps, kind, n, used, wall = cpu_replay_rate(synth.scaled(w3, n_flights=ns), ds, U_r / F, cores, fpc)
            cpu = {"value": ups, "unit": "updates/s", "cores": used, "kind": kind, "frames_per_s": fps,
                   "sample": f"{n} of {F} flights ({fpc} per worker process), P0 + mapping, logs in RAM, {wall:.2f} s wall"}
    ex["d_pinned"] = None
    cx.free_host_cache()

    # ---- the other BASELINE configurations at this N ---------------------------------------------------------------------------
    if args.workload == "c3" and "c3_weak" in want and world > 1:
        configs["c3_weak"] = guarded(cx, "c3_weak", lambda: run_flights(
            cx, w3, rank * w3.n_flights, w3.n_flights, world * w3.n_flights, "round 1's weak-scaling variant: 4096 flights PER GPU", False)[0])
    for name in ("c1", "c2"):
        if name in want:
            # one small / medium grid: replicas only (DESIGN.md section 8) -- rank 0 runs it, the others take part in the barriers
            wn = synth.on_mm_lattice(synth.CONFIGS[name])
            configs[name] = guarded(cx, name, lambda: run_flights(cx, wn, 0, 1 if rank == 0 else 0, 1,
                                                                  f"{name}: one flight, P0 included; replicas only (rank 0)", False)[0])
            if name == "c2" and rank == 0 and "error" not in configs[name]:
                configs[name]["p0"] = guarded(cx, "p0", lambda: run_p0_variants(cx, wn))
    if "c4" in want and args.workload != "c4":
        configs["c4"] = guarded(cx, "c4", lambda: run_c4(cx, verify)[0])
    if "c5" in want:
        configs["c5"] = guarded(cx, "c5", lambda: run_c5(cx, verify))

    if rank == 0:
        out = {"metric": METRIC, "value": head["value"], "unit": "updates/s", "n_gpus": world, "steps": head["steps"], "warmup": args.warmup,
               "ms_per_step": head["ms_per_step"], "higher_is_better": True, "scaling": "strong", "vs_baseline": None, "dtype": "i8",
               "data": DATA, "config": cfg, "frames_per_s": head["frames_per_s"],
               "ray_cell_updates_per_step": head["updates"], "hash": head.get("hash"), "hash_n1": head.get("hash_n1"),
               "roofline": roofline, "cpu_baseline": cpu, "e2e": head.get("e2e"), "e2e_variants": head.get("e2e_variants"),
               "gpu_launches": ex["launches"], "clocks": ex.get("clocks"), "host": {"cpus": os.cpu_count(), "rank_local_cpus": cx.local_cpus},
               "configs": configs}
        out_fd.emit(json.dumps(out))
    if world > 1:
        if cx.comm_ready:
            m.comm_destroy()
        cx.dist.destroy_process_group()


if __name__ == "__main__":
    main()
