"""What recentering costs in the batch replay: uqs_replay_recentering_dev on a config-3-shaped fleet (4096 flights x
3000 frames x 32 beams, 400x400 at 5 cm) with wandering poses, through the sub-tile route (engine 0) and the segment
route (engine 3), against uqs_replay_dev on the same logs at a fixed origin; and one long log through
uqs_replay_recentering of this library and, with --old-lib, of another build (e.g. the parent commit's), alternated
call by call in one process.  Device-resident inputs, CUDA events, medians of the repetitions.  Checks that both
routes give identical bytes and that a sample of flights equals the oracle.  Prints one JSON line.

    python tools/recentering_batch.py [--reps 5] [--old-lib PATH]
"""
import argparse
import ctypes
import importlib
import json
import os
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import numpy as np  # noqa: E402
import torch  # noqa: E402

from oracle import orc  # noqa: E402

m = importlib.import_module("micro-quad-slam_b200")
syn = importlib.import_module("micro-quad-slam_b200.synth")


def timed(fn, reps):
    out = []
    for _ in range(reps):
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        torch.cuda.synchronize()
        a.record()
        fn()
        b.record()
        b.synchronize()
        out.append(a.elapsed_time(b))
    return out


def wandering(F, N, seed):
    w = syn.scaled(syn.CONFIGS["c3"], n_flights=F, n_samples=N)
    d = syn.generate(w)
    rng = np.random.default_rng(seed)
    t = (np.arange(w.n_frames, dtype=np.float32) / np.float32(50.0))[None]
    sp = rng.uniform(0.5, 3.0, (F, 1)).astype(np.float32)
    hd = rng.uniform(-np.pi, np.pi, (F, 1)).astype(np.float32)
    x = (d["x_true"] + sp * np.cos(hd) * t).astype(np.float32)
    y = (d["y_true"] + sp * np.sin(hd) * t).astype(np.float32)
    return w, x, y, d["frame_yaw_deg"], d["ranges"]


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--old-lib", default=None)
    a = ap.parse_args()
    m.init(0)
    dev = torch.device("cuda:0")
    res = {"card": torch.cuda.get_device_name(0)}
    try:
        res["power_limit"] = subprocess.check_output(["nvidia-smi", "--query-gpu=power.limit", "--format=csv,noheader"],
                                                     text=True).strip()
    except Exception:
        res["power_limit"] = None
    # ---- the fleet ------------------------------------------------------------------------
    w, x, y, yaw, r = wandering(4096, 3000, 1)
    p = w.params()
    F, N = x.shape
    t = [torch.from_numpy(np.ascontiguousarray(v)).to(dev) for v in (x, y, yaw, r)]
    ptrs = [v.data_ptr() for v in t]
    grids = {k: torch.empty((F, p.H, p.W), dtype=torch.int8, device=dev) for k in ("A", "B", "plain")}
    origins = torch.empty((F, 2), dtype=torch.float32, device=dev)
    n_ev = torch.empty(F, dtype=torch.int32, device=dev)

    def rec(k):
        m.replay_recentering_dev(p, F, N, *ptrs, grids[k].data_ptr(), origins.data_ptr(), n_ev.data_ptr())

    def route(k):
        def go():
            m.set_engine(0 if k == "A" else 3, 0)
            rec(k)
        return go

    def plain():
        m.set_engine(0, 0)
        m.replay_dev(p, F, N, *ptrs, grids["plain"].data_ptr())

    fa, fb = route("A"), route("B")
    for f in (fa, fb, plain):
        f()
    torch.cuda.synchronize()
    ta, tb, tp = [], [], []
    for _ in range(a.reps):                                     # alternated
        ta += timed(fa, 1)
        tp += timed(plain, 1)
    tb = timed(fb, max(1, a.reps // 2))
    m.set_engine(0, 0)
    same = bool(torch.equal(grids["A"], grids["B"]))
    o = orc.Oracle()
    ga = grids["A"].cpu().numpy()
    ok = all(np.array_equal(ga[f], o.replay_recentering(p, x[f], y[f], yaw[f], r[f])[0]) for f in range(0, F, 512))
    ev = n_ev.cpu().numpy()
    res["fleet"] = {"flights": F, "frames": N, "grid": [p.W, p.H], "events_mean": float(ev.mean()),
                    "route_a_ms": float(np.median(ta)), "route_b_ms": float(np.median(tb)),
                    "replay_dev_fixed_origin_ms": float(np.median(tp)), "spread_a": [min(ta), max(ta)],
                    "spread_plain": [min(tp), max(tp)], "routes_identical": same, "sample_matches_oracle": ok}
    del grids, t
    torch.cuda.empty_cache()
    # ---- one long log: old and new uqs_replay_recentering (host buffers, wall clock) -------------------------------
    w1 = syn.Workload("wander", 3, 1, 60000, 400, "0.05", 20.0, 50.0)
    d1 = syn.generate(w1)
    p1 = w1.params()
    tt = np.arange(60000, dtype=np.float32) / np.float32(50.0)
    lx = (d1["x_true"][0] + np.float32(1.3) * tt * np.cos(tt / np.float32(90.0))).astype(np.float32)
    ly = (d1["y_true"][0] + np.float32(1.1) * tt * np.sin(tt / np.float32(70.0))).astype(np.float32)
    lyaw, lr = d1["yaw_deg"][0], d1["ranges"][0]
    libs = {"new": m.lib()}
    if a.old_lib:
        L = ctypes.CDLL(a.old_lib)
        L.uqs_replay_recentering.argtypes = m.lib().uqs_replay_recentering.argtypes
        if L.uqs_init(0) != 0:
            raise SystemExit("old library: uqs_init failed")
        libs["old"] = L
    outs, times = {}, {k: [] for k in libs}
    for _ in range(a.reps):
        for k, L in libs.items():
            g = np.empty((p1.H, p1.W), np.int8)
            org = np.zeros(2, np.float32)
            n = ctypes.c_int(0)
            t0 = time.perf_counter()
            rc = L.uqs_replay_recentering(ctypes.byref(p1), 60000, *(v.ctypes.data for v in (lx, ly, lyaw, lr, g, org)),
                                          ctypes.byref(n), None, 0, None)
            times[k].append((time.perf_counter() - t0) * 1e3)
            outs[k] = (rc, g, n.value)
    want = o.replay_recentering(p1, lx, ly, lyaw, lr)
    res["long_log"] = {"frames": 60000, "grid": [400, 400], "events": want[2],
                       **{f"{k}_ms": float(np.median(v)) for k, v in times.items()},
                       **{f"{k}_rc": outs[k][0] for k in outs},
                       **{f"{k}_matches_oracle": bool(outs[k][0] == 0 and np.array_equal(outs[k][1], want[0])) for k in outs}}
    print(json.dumps(res))


if __name__ == "__main__":
    main()
