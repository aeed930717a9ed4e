"""A/B of the device replay's schedule (uqs_set_setup_overlap): ray set-up of each chunk beside the previous chunk's
replay (n waves per chunk) against set-up then replay (0).  Config 3 at full size as bench.py steps it (P0 + ray
set-up + replay, logs resident in HBM), then the config-5 resolutions whose grids are 400^2 to 800^2 (1024 flights
each, the replay alone).  Variants alternate inside one process, each run is a CUDA-event time over a few steps, and
every variant must leave the same grid digest and stats.  Ends with one timeline of a config-3 step under the
overlapped schedule (uqs_profile_timeline: kind, start, end in ms per kernel span).

    python tools/setup_overlap_ab.py [runs] [waves ...]        (default: 7 runs, waves 0 2 3)
"""
import importlib, os, statistics, subprocess, sys
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import numpy as np, torch
m = importlib.import_module("micro-quad-slam_b200"); syn = importlib.import_module("micro-quad-slam_b200.synth")
m.init(0); dev = torch.device("cuda:0"); m.set_stream(torch.cuda.current_stream().cuda_stream)
RUNS = int(sys.argv[1]) if len(sys.argv) > 1 else 7
WAVES = [int(a) for a in sys.argv[2:]] or [0, 2, 3]
KIND = {0: "pose", 1: "set-up", 2: "replay"}
try:
    print(subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                         capture_output=True, text=True).stdout.strip(), flush=True)
except OSError:
    pass


def timed(fn, steps):
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record()
    for _ in range(steps):
        fn()
    b.record(); b.synchronize()
    return a.elapsed_time(b) / steps


def ab(label, step, digest, steps):
    """Alternate the variants RUNS times; print median and spread of each, check digests and stats."""
    ref, t = None, {v: [] for v in WAVES}
    for v in WAVES:                                          # warm every variant (and check it) first
        m.set_setup_overlap(v)
        st = step(True)
        key = (digest(), tuple(sorted(st.items())))
        ref = ref or key
        assert key == ref, f"{label}: waves={v} changes the result"
    chunks = {}
    for _ in range(RUNS):
        for v in WAVES:
            m.set_setup_overlap(v)
            t[v].append(timed(step, steps))
            chunks[v] = m.setup_overlap_chunks()
    base = statistics.median(t[WAVES[0]])
    for v in WAVES:
        med = statistics.median(t[v])
        print(f"{label:34s} waves={v}: median {med:8.3f} ms  min {min(t[v]):8.3f}  max {max(t[v]):8.3f}  "
              f"({100 * (med / base - 1):+5.1f} %)  chunks beside a replay: {chunks[v]}", flush=True)
    m.set_setup_overlap(-1)


def device_log(w):
    d = syn.generate(w)
    return d, [torch.from_numpy(np.ascontiguousarray(d[k])).to(dev) for k in ("t_ms", "of_rate_x", "of_rate_y", "h_m", "yaw_deg", "of_q", "ranges")]


# ---- config 3 at full size: P0 + set-up + replay per step, as bench.py's device step ----
w = syn.CONFIGS["c3"]
p = w.params()
d, (t_ms, rx, ry, h, yaw, q, rng) = device_log(w)
F, N = w.n_flights, w.n_samples
dx, dy = torch.empty((F, N), dtype=torch.float32, device=dev), torch.empty((F, N), dtype=torch.float32, device=dev)
g = torch.empty((F, p.H, p.W), dtype=torch.int8, device=dev)
assert N == w.n_frames, "config 3 has one frame per sample"


def c3_step(want_stats=False):
    m.pose_integrate_dev(F, N, t_ms.data_ptr(), rx.data_ptr(), ry.data_ptr(), h.data_ptr(), yaw.data_ptr(), q.data_ptr(),
                         dx.data_ptr(), dy.data_ptr(), 0)
    return m.replay_dev(p, F, N, dx.data_ptr(), dy.data_ptr(), yaw.data_ptr(), rng.data_ptr(), g.data_ptr(), want_stats=want_stats)


def c3_digest():
    return int(m.grid_hashes_dev(g.data_ptr(), F, p.W * p.H).sum(dtype=np.uint64))


ab(f"c3 {F} flights x {N} frames", c3_step, c3_digest, 3)

# one step's timeline under the overlapped schedule
m.set_setup_overlap(-1)
c3_step()
m.set_profiling(True); m.profile_collect()
c3_step()
spans = m.profile_timeline()
m.profile_collect(); m.set_profiling(False)
print("timeline of one config-3 step (default schedule), ms from the first span:")
for k, a, b in spans:
    print(f"  {KIND.get(k, k):7s} {a:8.3f} .. {b:8.3f}  ({b - a:7.3f} ms)")
del g, dx, dy, t_ms, rx, ry, h, yaw, q, rng
torch.cuda.empty_cache()

# ---- config 5: resolutions whose grids are 400^2 .. 800^2, 1024 flights each (the replay alone) ----
for ir in range(len(syn.C5_RES)):
    w = syn.c5_workload(ir, 5, n_flights=1024)
    if not 400 <= w.W <= 800:
        continue
    d = syn.generate(w); p = w.params()
    tt = [torch.from_numpy(np.ascontiguousarray(a)).to(dev) for a in (d["x_true"], d["y_true"], d["frame_yaw_deg"], d["ranges"])]
    g = torch.empty((w.n_flights, p.H, p.W), dtype=torch.int8, device=dev)
    step = lambda want_stats=False: m.replay_dev(p, w.n_flights, w.n_frames, *(a.data_ptr() for a in tt), g.data_ptr(),
                                                 want_stats=want_stats)
    ab(f"c5 res {w.res} m, {w.W}^2, 1024 flights", step,
       lambda: int(m.grid_hashes_dev(g.data_ptr(), w.n_flights, p.W * p.H).sum(dtype=np.uint64)), 2)
    del tt, g
    torch.cuda.empty_cache()
