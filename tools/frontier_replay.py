"""What frontier queries cost inside the batch replay: uqs_replay_frontier_dev against uqs_replay_dev on the same
device-resident inputs, alternated in one process, timed with CUDA events (median of the repetitions).  Also checks
that the grids are identical and that a sample of the scores equals the oracle's statement (each flight replayed by
the CPU restatement up to the query's frame, then frontier_score_dir).

Cases: config 3 at full size with 0 / 10 / 100 / 1000 queries per flight at random frames (offsets -90 / 0 / +90 deg,
the flight's own pose at that frame); config 2's one-hour log with one query per second (time slices active); one
config-5 resolution with 1000 x 1000 grids (sub-tile engine).  Prints one JSON line.

    python tools/frontier_replay.py [reps]
"""
import importlib
import json
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import numpy as np  # noqa: E402
import torch  # noqa: E402

from oracle import orc  # noqa: E402

m = importlib.import_module("micro-quad-slam_b200")
syn = importlib.import_module("micro-quad-slam_b200.synth")


def oracle_scores(o, p, x, y, yaw, r, q):
    out = np.zeros(q.size, np.int32)
    for f in np.unique(q["flight"]):
        grid = np.zeros((p.H, p.W), np.int8)
        mine = np.flatnonzero(q["flight"] == f)
        mine = mine[np.argsort(q["frame"][mine], kind="stable")]
        done = 0
        for i in mine:
            upto = int(q["frame"][i]) + 1
            if upto > done:
                o.replay(p, x[f, done:upto], y[f, done:upto], yaw[f, done:upto], r[f, done:upto], grid=grid)
                done = upto
            out[i] = o.frontier_score(p, grid, q["x"][i], q["y"][i], q["yaw_deg"][i], q["offset_deg"][i])
    return out


def queries_at(rng, x, y, yaw, flights, frames):
    off = rng.choice(np.array([-90.0, 0.0, 90.0], np.float32), flights.size)
    q = m.make_queries(flights, frames, x[flights, frames], y[flights, frames], yaw[flights, frames], off)
    return q[rng.permutation(q.size)]


def run_case(name, w, d, q, reps, o, n_check):
    dev = torch.device("cuda:0")
    p = w.params()
    F, N = w.n_flights, w.n_frames
    x, y, yaw, r = d["x_true"], d["y_true"], d["frame_yaw_deg"], d["ranges"]
    t = [torch.from_numpy(np.ascontiguousarray(a)).to(dev) for a in (x, y, yaw, r)]
    g0 = torch.empty((F, p.H, p.W), dtype=torch.int8, device=dev)
    g1 = torch.empty_like(g0)
    tq = torch.from_numpy(np.ascontiguousarray(q).view(np.uint8)).to(dev)
    ts = torch.empty(max(q.size, 1), dtype=torch.int32, device=dev)
    plain = lambda: m.replay_dev(p, F, N, *(a.data_ptr() for a in t), g0.data_ptr())
    query = lambda: m.replay_frontier_dev(p, F, N, *(a.data_ptr() for a in t), g1.data_ptr(), q.size, tq.data_ptr(), ts.data_ptr())
    plain(); query(); torch.cuda.synchronize()                      # warm-up: modules, scratch, CUB
    times = {"plain": [], "query": []}
    for _ in range(reps):
        for k, fn in (("plain", plain), ("query", query)):
            a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            a.record(); fn(); b.record(); b.synchronize()
            times[k].append(a.elapsed_time(b))
    same = bool(torch.equal(g0, g1))
    scores = ts[:q.size].cpu().numpy()
    ok = None
    if q.size:
        pick = np.random.default_rng(7).choice(q.size, min(n_check, q.size), replace=False)
        want = oracle_scores(o, p, x, y, yaw, r, q[pick])
        ok = bool(np.array_equal(scores[pick], want))
    tp, tqm = float(np.median(times["plain"])), float(np.median(times["query"]))
    res = {"case": name, "flights": F, "frames": N, "grid": [p.W, p.H], "queries": int(q.size), "replay_ms": round(tp, 3),
           "replay_frontier_ms": round(tqm, 3), "queries_cost_ms": round(tqm - tp, 3),
           "spread_ms": [round(float(np.min(times["plain"])), 3), round(float(np.max(times["plain"])), 3),
                         round(float(np.min(times["query"])), 3), round(float(np.max(times["query"])), 3)],
           "grids_identical": same, "scores_checked": min(n_check, int(q.size)), "scores_match_oracle": ok}
    print(json.dumps(res), file=sys.stderr, flush=True)
    del t, g0, g1, tq, ts
    torch.cuda.empty_cache()
    return res


def main():
    reps = int(sys.argv[1]) if len(sys.argv) > 1 else 7
    m.init(0)
    m.set_stream(torch.cuda.current_stream().cuda_stream)
    o = orc.Oracle()
    try:
        power = subprocess.check_output(["nvidia-smi", "--query-gpu=power.limit", "--format=csv,noheader", "-i", "0"],
                                        text=True).strip()
    except (OSError, subprocess.CalledProcessError):
        power = "unknown"
    out = {"card": torch.cuda.get_device_name(0), "power_limit": power, "reps": reps, "cases": []}
    rng = np.random.default_rng(2024)

    w = syn.CONFIGS["c3"]
    d = syn.generate(w)
    F, N = w.n_flights, w.n_frames
    for qpf in (0, 10, 100, 1000):
        fl = np.repeat(np.arange(F, dtype=np.int32), qpf)
        q = queries_at(rng, d["x_true"], d["y_true"], d["frame_yaw_deg"], fl, rng.integers(0, N, fl.size).astype(np.int32))
        out["cases"].append(run_case(f"c3_{qpf}_per_flight", w, d, q, reps, o, 200))
    del d

    w = syn.CONFIGS["c2"]
    d = syn.generate(w)
    frames = np.arange(int(w.rate_hz) - 1, w.n_frames, int(w.rate_hz), dtype=np.int32)     # one per second
    q = queries_at(rng, d["x_true"], d["y_true"], d["frame_yaw_deg"], np.zeros(frames.size, np.int32), frames)
    out["cases"].append(run_case("c2_one_per_second", w, d, q, reps, o, 40))
    del d

    ir = syn.C5_RES.index("0.02")                                                           # 1000 x 1000
    w = syn.c5_workload(ir, 8)
    d = syn.generate(w)
    F, N = w.n_flights, w.n_frames
    fl = np.repeat(np.arange(F, dtype=np.int32), 100)
    q = queries_at(rng, d["x_true"], d["y_true"], d["frame_yaw_deg"], fl, rng.integers(0, N, fl.size).astype(np.int32))
    out["cases"].append(run_case(f"c5_{w.W}_100_per_flight", w, d, q, reps, o, 100))
    print(json.dumps(out))


if __name__ == "__main__":
    main()
