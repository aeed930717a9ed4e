"""What frontier queries cost inside the batch replay with recentering: uqs_replay_recentering_frontier_dev against
uqs_replay_recentering_dev on the wandering config-3-shaped fleet of tools/recentering_batch.py (4096 flights x 3000
frames, 400x400 at 5 cm, the sub-tile route) with 0, 10 and 100 queries per flight at random frames, and on that tool's
one long log (60000 frames, the segment route) with one query per second.  Calls alternated, CUDA events around each,
medians of the repetitions; device-resident inputs.  Checks that the grids equal those of uqs_replay_recentering_dev
and that a sample of scores equals the oracle's frame-by-frame statement (tests/test_recentering_frontier_cpu.py).  Prints one JSON line.

    python tools/recentering_frontier.py [--reps 7]
"""
import argparse
import importlib
import json
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tools"))
sys.path.insert(0, os.path.join(ROOT, "tests"))
import numpy as np  # noqa: E402
import torch  # noqa: E402

from oracle import orc  # noqa: E402
from recentering_batch import timed, wandering  # noqa: E402
from test_recentering_frontier_cpu import recentering_walk  # noqa: E402

m = importlib.import_module("micro-quad-slam_b200")
syn = importlib.import_module("micro-quad-slam_b200.synth")
OFFSETS = np.array([-90.0, 0.0, 90.0], np.float32)


def case(p, x, y, yaw, r, q, reps, oracle, sample_flights):
    """median ms of both calls (alternated), identical grids/origins/events, sampled scores against the oracle"""
    dev = torch.device("cuda:0")
    F, N = x.shape
    t = [torch.from_numpy(np.ascontiguousarray(v)).to(dev) for v in (x, y, yaw, r)]
    ptrs = [v.data_ptr() for v in t]
    outs = {k: (torch.empty((F, p.H, p.W), dtype=torch.int8, device=dev), torch.empty((F, 2), dtype=torch.float32, device=dev),
                torch.empty(F, dtype=torch.int32, device=dev), torch.zeros((F, 4, 3), dtype=torch.int32, device=dev))
            for k in ("plain", "queries")}
    tq = torch.from_numpy(q.view(np.uint8)).to(dev) if q.size else None
    ts = torch.empty(max(q.size, 1), dtype=torch.int32, device=dev)

    def plain():
        m.replay_recentering_dev(p, F, N, *ptrs, *(o.data_ptr() for o in outs["plain"]), 4)

    def with_queries():
        m.replay_recentering_frontier_dev(p, F, N, *ptrs, *(o.data_ptr() for o in outs["queries"]), 4, q.size,
                                          tq.data_ptr() if q.size else 0, ts.data_ptr() if q.size else 0)

    plain()
    with_queries()
    tp, tw = [], []
    for _ in range(reps):
        tp += timed(plain, 1)
        tw += timed(with_queries, 1)
    torch.cuda.synchronize()
    same = all(bool(torch.equal(a, b)) for a, b in zip(outs["plain"], outs["queries"]))
    scores = ts.cpu().numpy()[:q.size]
    checked = bad = 0
    for f in sample_flights:
        mine = np.flatnonzero(q["flight"] == f)
        if mine.size:
            want = recentering_walk(oracle, p, x[f], y[f], yaw[f], r[f], q[mine])[4]
            checked += mine.size
            bad += int((scores[mine] != want).sum())
    del outs, t
    torch.cuda.empty_cache()
    return {"queries": int(q.size), "recentering_dev_ms": float(np.median(tp)), "with_queries_ms": float(np.median(tw)),
            "cost_ms": float(np.median(tw) - np.median(tp)), "spread_plain": [min(tp), max(tp)], "spread_queries": [min(tw), max(tw)],
            "outputs_identical": same, "scores_checked": checked, "scores_differing": bad}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=7)
    a = ap.parse_args()
    m.init(0)
    m.set_stream(torch.cuda.current_stream().cuda_stream)       # the library's kernels between the timing events
    res = {"card": torch.cuda.get_device_name(0)}
    try:
        res["power_limit"] = subprocess.check_output(["nvidia-smi", "--query-gpu=power.limit", "--format=csv,noheader"],
                                                     text=True).strip()
    except Exception:
        res["power_limit"] = None
    oracle = orc.Oracle()
    # ---- the fleet (route A) ---------------------------------------------------------------------------------------
    w, x, y, yaw, r = wandering(4096, 3000, 1)
    p = w.params()
    F, N = x.shape
    rng = np.random.default_rng(5)
    res["fleet"] = {"flights": F, "frames": N, "grid": [p.W, p.H]}
    for per in (0, 10, 100):
        fl = np.repeat(np.arange(F, dtype=np.int32), per)
        fr = rng.integers(0, N, fl.size).astype(np.int32)
        q = m.make_queries(fl, fr, x[fl, fr], y[fl, fr], yaw[fl, fr], rng.choice(OFFSETS, fl.size))
        q = q[rng.permutation(q.size)]
        res["fleet"][f"{per}_per_flight"] = case(p, x, y, yaw, r, q, a.reps, oracle, range(0, F, 512))
    del x, y, yaw, r
    # ---- the long log (route B, time-sliced segments) --------------------------------------------------------------
    w1 = syn.Workload("wander", 3, 1, 60000, 400, "0.05", 20.0, 50.0)
    d1 = syn.generate(w1)
    p1 = w1.params()
    tt = np.arange(60000, dtype=np.float32) / np.float32(50.0)
    lx = (d1["x_true"][0] + np.float32(1.3) * tt * np.cos(tt / np.float32(90.0))).astype(np.float32)[None]
    ly = (d1["y_true"][0] + np.float32(1.1) * tt * np.sin(tt / np.float32(70.0))).astype(np.float32)[None]
    lyaw, lr = d1["yaw_deg"][:1], np.ascontiguousarray(d1["ranges"][:1])
    fr = np.arange(49, 60000, 50, dtype=np.int32)
    q = m.make_queries(0, fr, lx[0, fr], ly[0, fr], lyaw[0, fr], rng.choice(OFFSETS, fr.size))
    res["long_log"] = {"frames": 60000, "grid": [400, 400], "events": int(oracle.replay_recentering(p1, lx, ly, lyaw, lr)[2]),
                       **case(p1, lx, ly, lyaw, lr, q, a.reps, oracle, [0])}
    print(json.dumps(res))


if __name__ == "__main__":
    main()
