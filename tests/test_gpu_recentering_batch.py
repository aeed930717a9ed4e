"""uqs_replay_recentering_dev: many flights per call, each recentred exactly as log_tick() does, against the oracle
flight by flight (grid bytes, final origin bits, event count, event list, ray-cell updates), on both routes: the
sub-tile engine in each flight's global frame (route A) and the segment loop (route B)."""
import ctypes
import os
import subprocess
import sys

import numpy as np
import pytest
import torch

from conftest import first_diff

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


@pytest.fixture()
def dev(gpu):
    """Engine and tuning back to their defaults afterwards."""
    try:
        yield torch.device("cuda:0")
    finally:
        gpu.set_engine(0, 0)
        gpu.set_tuning(0, 0, 0)


def oracle_events(oracle, p, x, y):
    """The oracle's recenter decisions (orc_recentre_if_needed on a 2x2 grid: the decision reads only the poses,
    size_m, res_m and the running origin) -> [[frame, sx, sy], ...]."""
    L = oracle.L
    L.orc_recentre_if_needed.argtypes = [ctypes.c_void_p, ctypes.c_void_p, ctypes.c_float, ctypes.c_float,
                                         ctypes.POINTER(ctypes.c_int), ctypes.POINTER(ctypes.c_int)]
    q = p.copy()
    q.W = q.H = 2
    g = np.zeros(4, np.int8)
    sx, sy = ctypes.c_int(0), ctypes.c_int(0)
    out = []
    for i in range(x.size):
        if L.orc_recentre_if_needed(ctypes.byref(q), g.ctypes.data, x[i], y[i], ctypes.byref(sx), ctypes.byref(sy)):
            out.append((i, sx.value, sy.value))
    return np.asarray(out, np.int32).reshape(-1, 3)


def oracle_fleet(oracle, p, x, y, yaw, r):
    F = x.shape[0]
    grids = np.empty((F, p.H, p.W), np.int8)
    origins = np.empty((F, 2), np.float32)
    events, U = [], 0
    for f in range(F):
        g, o, n, u = oracle.replay_recentering(p, x[f], y[f], yaw[f], r[f])
        grids[f], origins[f] = g, o
        ev = oracle_events(oracle, p, x[f], y[f])
        assert ev.shape[0] == n
        events.append(ev)
        U += u
    return grids, origins, events, U


def run(gpu, p, x, y, yaw, r, max_events=64):
    F, N = x.shape
    t = [torch.from_numpy(np.ascontiguousarray(a, np.float32)).cuda() for a in (x, y, yaw, r.reshape(F, N, 32))]
    grids = torch.full((F, p.H, p.W), 55, dtype=torch.int8, device="cuda")
    origins = torch.zeros((F, 2), dtype=torch.float32, device="cuda")
    n_ev = torch.zeros(F, dtype=torch.int32, device="cuda")
    events = torch.full((F, max(max_events, 1), 3), -7, dtype=torch.int32, device="cuda")
    torch.cuda.synchronize()
    l0 = gpu.kernel_launches()
    st = gpu.replay_recentering_dev(p, F, N, *(a.data_ptr() for a in t), grids.data_ptr(), origins.data_ptr(), n_ev.data_ptr(),
                                    events.data_ptr() if max_events else 0, max_events, want_stats=True)
    launches = gpu.kernel_launches() - l0
    torch.cuda.synchronize()
    return grids.cpu().numpy(), origins.cpu().numpy(), n_ev.cpu().numpy(), events.cpu().numpy(), st, launches


def check(got, want, what, max_events=64):
    grids, origins, n_ev, events, st, _ = got
    wg, wo, wev, U = want
    for f in range(grids.shape[0]):
        assert np.array_equal(grids[f], wg[f]), (what, f, first_diff(grids[f], wg[f]))
        assert origins[f].view(np.uint32).tolist() == wo[f].view(np.uint32).tolist(), (what, f, origins[f], wo[f])
        assert n_ev[f] == wev[f].shape[0], (what, f, n_ev[f], wev[f].shape[0])
        k = min(int(n_ev[f]), max_events)
        assert np.array_equal(events[f, :k], wev[f][:k]), (what, f)
    assert st["ray_cell_updates"] == U, what


def fleet(synth, F, N, W, res, size, seed):
    """wandering_log-style drifts with per-flight speed and heading, plus the special flights listed below."""
    w = synth.Workload("wander", seed, F, N, W, res, size, 50.0)
    d = synth.generate(w)
    p = w.params()
    rng = np.random.default_rng(seed)
    t = (np.arange(N, dtype=np.float32) / np.float32(50.0))[None]
    speed = rng.uniform(0.5, 6.0, (F, 1)).astype(np.float32)
    head = rng.uniform(-np.pi, np.pi, (F, 1)).astype(np.float32)
    x = (d["x_true"] + speed * np.cos(head) * t).astype(np.float32)
    y = (d["y_true"] + speed * np.sin(head) * t).astype(np.float32)
    size = float(p.size_m)
    x[0], y[0] = d["x_true"][0], d["y_true"][0]                       # 0, 1: never recenter
    x[1], y[1] = d["x_true"][1], d["y_true"][1]
    x[2] += np.float32(0.8 * size)                                     # 2: first pose far from the origin: event at frame 0
    tri = np.minimum(t[0], t[0, -1] - t[0])                            # 3: out and back over erased cells
    x[3] = d["x_true"][3] + np.float32(3.0) * tri
    y[3] = d["y_true"][3] - np.float32(1.5) * tri
    x[4, N // 3:] += np.float32(0.9 * size)                            # 4: a jump beyond max_shift (clamped shifts)
    y[4, N // 2:] -= np.float32(1.7 * size)
    x[5] = d["x_true"][5] + np.float32(2.5) * t[0]                     # 5: diagonal drift
    y[5] = d["y_true"][5] + np.float32(2.5) * t[0]
    x[6, 10], y[6, 11], x[6, 12], y[6, 13] = np.nan, np.nan, np.inf, -np.inf     # 6: NaN and Inf poses
    x[6, 40:44] = np.inf
    r = d["ranges"].copy()
    m = rng.random(r.shape)
    r[m < 0.03] = np.nan                                               # beams with no return, too short, out of range
    r[(m >= 0.03) & (m < 0.05)] = rng.uniform(0.0, 0.05, ((m >= 0.03) & (m < 0.05)).sum()).astype(np.float32)
    r[(m >= 0.05) & (m < 0.07)] = np.float32(9.0)
    return p, x, y, d["yaw_deg"], r


ROUTE_A = [(0, (0, 0, 1)), (1, (0, 0, 1)), (0, (40, 40, 1)), (1, (24, 56, 1))]     # (engine, (sw, sh, time slices))
ROUTE_B = [(3, (0, 0, 0)), (0, (0, 0, 4)), (1, (40, 40, 7))]


@pytest.mark.parametrize("geom", [(400, "0.05", 20.0), (500, "0.10", 50.0)])
def test_fleet_on_both_routes(gpu, oracle, synth, dev, geom):
    W, res, size = geom
    F, N = 256, 1200
    p, x, y, yaw, r = fleet(synth, F, N, W, res, size, seed=7 + W)
    want = oracle_fleet(oracle, p, x, y, yaw, r)
    n_ev = np.array([e.shape[0] for e in want[2]])
    assert n_ev[:2].tolist() == [0, 0] and want[2][2][0, 0] == 0 and (n_ev[2:] > 0).mean() > 0.8
    half = np.float32(p.size_m) * np.float32(0.5)
    cap = int(np.float32(np.float32(half / np.float32(p.res_m)) * np.float32(0.5)))    # max_shift, uav_local_nav.c:337
    assert np.abs(want[2][4][:, 1:]).max() == cap                      # flight 4's shifts were clamped
    results = []
    for engine, tune in ROUTE_A + ROUTE_B:
        gpu.set_engine(engine, 0)
        gpu.set_tuning(*tune)
        got = run(gpu, p, x, y, yaw, r)
        check(got, want, (engine, tune))
        route_a = (engine, tune) in ROUTE_A
        assert (got[5] < 16) == route_a, (engine, tune, got[5])         # route B launches per flight and segment
        results.append(got[0])
    assert all(np.array_equal(results[0], g) for g in results)
    # flights that never recenter equal uqs_replay_dev at the fixed origin
    gpu.set_engine(0, 0)
    gpu.set_tuning(0, 0, 0)
    plain, _ = gpu.replay(p, x[:2], y[:2], yaw[:2], r[:2])
    assert np.array_equal(plain, results[0][:2])


def test_one_long_log_old_and_new_call(gpu, oracle, synth, dev):
    w = synth.Workload("wander", 3, 1, 30000, 400, "0.05", 20.0, 50.0)
    d = synth.generate(w)
    p = w.params()
    t = np.arange(30000, dtype=np.float32) / np.float32(50.0)
    x = (d["x_true"][0] + np.float32(1.3) * t * np.cos(t / np.float32(90.0))).astype(np.float32)
    y = (d["y_true"][0] + np.float32(1.1) * t * np.sin(t / np.float32(70.0))).astype(np.float32)
    want_g, want_o, n, U = oracle.replay_recentering(p, x, y, d["yaw_deg"][0], d["ranges"][0])
    wev = oracle_events(oracle, p, x, y)
    assert n > 50
    grid, origin, events, st = gpu.replay_recentering(p, x, y, d["yaw_deg"][0], d["ranges"][0])
    assert np.array_equal(grid, want_g), first_diff(grid, want_g)
    assert np.float32(origin[0]) == np.float32(want_o[0]) and np.float32(origin[1]) == np.float32(want_o[1])
    assert np.array_equal(events, wev[:256]) and st["ray_cell_updates"] == U
    # the event count is no longer capped: the C call reports every event
    L = gpu.lib()
    g2 = np.empty((p.H, p.W), np.int8)
    o2 = np.zeros(2, np.float32)
    n2 = ctypes.c_int(-1)
    ev2 = np.zeros((8, 3), np.int32)
    rc = L.uqs_replay_recentering(ctypes.byref(p), 30000, *(a.ctypes.data for a in (x, y, d["yaw_deg"][0], d["ranges"][0], g2, o2)),
                                  ctypes.byref(n2), ev2.ctypes.data, 8, None)
    assert rc == 0 and n2.value == n and np.array_equal(ev2, wev[:8]) and np.array_equal(g2, want_g)
    for engine, tune in [(0, (0, 0, 0)), (0, (0, 0, 1)), (3, (0, 0, 0))]:
        gpu.set_engine(engine, 0)
        gpu.set_tuning(*tune)
        got = run(gpu, p, x[None], y[None], d["yaw_deg"][:1], d["ranges"][:1], max_events=4096)
        check(got, (want_g[None], np.asarray(want_o, np.float32)[None], [wev], U), (engine, tune), max_events=4096)


@pytest.mark.parametrize("case", ["long rays", "clamp excludes 0"])
def test_inputs_that_take_the_segment_route(gpu, oracle, synth, dev, case):
    if case == "long rays":
        w = synth.Workload("wander", 5, 4, 300, 1200, "0.0035", 4.2, 50.0)
    else:
        w = synth.Workload("wander", 6, 4, 600, 400, "0.05", 20.0, 50.0)
    d = synth.generate(w)
    p = w.params()
    if case == "clamp excludes 0":
        p.lo_min, p.lo_max = 5, 60
    t = (np.arange(d["x_true"].shape[1], dtype=np.float32) / np.float32(50.0))[None]
    x = (d["x_true"] + np.float32(2.0) * t).astype(np.float32)
    y = (d["y_true"] - np.float32(1.0) * t).astype(np.float32)
    want = oracle_fleet(oracle, p, x, y, d["yaw_deg"], d["ranges"])
    assert sum(e.shape[0] for e in want[2]) > 0
    for engine in (0, 1):
        gpu.set_engine(engine, 0)
        gpu.set_tuning(0, 0, 1)
        got = run(gpu, p, x, y, d["yaw_deg"], d["ranges"])
        check(got, want, (case, engine))
        assert got[5] >= 16


def test_engine_2_refused_max_events_and_bad_arguments(gpu, oracle, synth, dev):
    p, x, y, yaw, r = fleet(synth, 8, 400, 400, "0.05", 20.0, seed=11)
    want = oracle_fleet(oracle, p, x, y, yaw, r)
    gpu.set_engine(2, 0)
    with pytest.raises(gpu.UqsError) as e:
        run(gpu, p, x, y, yaw, r)
    assert e.value.code == gpu.ERR_BAD_ARG and "engine 2" in str(e.value)
    gpu.set_engine(0, 0)
    for cap in (0, 1, 2):
        got = run(gpu, p, x, y, yaw, r, max_events=cap)
        check(got, want, cap, max_events=cap)
        assert (got[3][:, cap:] == -7).all()
    # bad arguments: nothing is written
    F, N = x.shape
    t = [torch.from_numpy(a).cuda() for a in (x, y, yaw, r)]
    outs = [torch.full((F, p.H, p.W), 9, dtype=torch.int8, device="cuda"), torch.full((F, 2), 9.0, device="cuda"),
            torch.full((F,), 9, dtype=torch.int32, device="cuda"), torch.full((F, 4, 3), 9, dtype=torch.int32, device="cuda")]
    ptr = [a.data_ptr() for a in t] + [o.data_ptr() for o in outs]
    L = gpu.lib()
    bad = [dict(F=0), dict(N=-1), dict(i=0), dict(i=3), dict(i=4), dict(i=5), dict(i=6), dict(max_events=-1),
           dict(max_events=4, i=7)]
    torch.cuda.synchronize()
    for b in bad:
        args = list(ptr)
        if "i" in b:
            args[b["i"]] = None
        rc = L.uqs_replay_recentering_dev(ctypes.byref(p), b.get("F", F), b.get("N", N), *args, b.get("max_events", 4), None)
        assert rc == gpu.ERR_BAD_ARG, b
    torch.cuda.synchronize()
    assert all(bool((o == 9).all()) for o in outs)


def test_many_flights_across_internal_chunks(gpu, oracle, synth, dev):
    """65535 + 45 flights: the ray set-up takes at most 65535 flights per launch, so the call spans two chunks."""
    F, N = 65535 + 45, 24
    p = gpu.make_params(64, 64, 0.05, size_m=3.2)
    rng = np.random.default_rng(4)
    t = np.arange(N, dtype=np.float32)[None] * np.float32(0.1)
    x = (rng.uniform(-1, 1, (F, 1)) + rng.uniform(-1, 1, (F, 1)) * t).astype(np.float32)
    y = (rng.uniform(-1, 1, (F, 1)) + rng.uniform(-1, 1, (F, 1)) * t).astype(np.float32)
    yaw = rng.uniform(-180, 180, (F, N)).astype(np.float32)
    r = rng.uniform(0.1, 2.0, (F, N, 32)).astype(np.float32)
    got = run(gpu, p, x, y, yaw, r, max_events=8)
    grids, origins, n_ev, events, st, launches = got
    assert launches < 24
    for f in list(range(0, 40)) + list(range(65500, F)):
        g, o, n, _ = oracle.replay_recentering(p, x[f], y[f], yaw[f], r[f])
        ev = oracle_events(oracle, p, x[f], y[f])
        assert np.array_equal(grids[f], g), (f, first_diff(grids[f], g))
        assert origins[f].tolist() == list(np.float32(o)) and n_ev[f] == n and np.array_equal(events[f, :min(n, 8)], ev[:8]), f
    assert n_ev.sum() > F


def test_under_the_bounds_checked_build(pkg):
    """This file once more under -DUQS_DEBUG_BOUNDS (every shared-memory access of the engines checked against its
    region), without the many-flight case."""
    dbg = os.path.join(ROOT, "micro-quad-slam_b200", "libuqs_mapping_dbg.so")
    assert os.path.exists(dbg)
    env = dict(os.environ, UQS_LIBRARY=dbg)
    res = subprocess.run([sys.executable, "-m", "pytest", os.path.abspath(__file__), "-q", "-x", "-m", "gpu", "-k",
                          "not many_flights and not bounds_checked", "-p", "no:cacheprovider"], capture_output=True, text=True,
                         env=env, timeout=2400, cwd=ROOT)
    tail = res.stdout[-3000:] + res.stderr[-2000:]
    assert res.returncode == 0 and "UQS_DEBUG_BOUNDS" not in res.stdout + res.stderr, tail
    assert " passed" in res.stdout and "failed" not in res.stdout, tail
