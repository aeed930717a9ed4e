"""uqs_replay_recentering_frontier_dev: frontier queries answered at their frame on recentred maps, inside the batch
replay with recentering.  Every score against the oracle's frame-by-frame statement (recentering_scores_at_frames,
pinned in tests/test_recentering_frontier_cpu.py); grids, origins, events and stats against uqs_replay_recentering_dev byte for
byte; both routes, every engine and tuning of tests/test_gpu_recentering_batch.py, and queries placed where the order of
events and probes decides the score."""
import ctypes
import os
import subprocess
import sys

import numpy as np
import pytest
import torch

from conftest import first_diff
from test_frontier_replay_cpu import hostile_queries
from test_gpu_recentering_batch import ROUTE_A, ROUTE_B, fleet
from test_gpu_recentering_batch import run as run_plain
from test_recentering_frontier_cpu import events_of, recentering_scores_at_frames

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
OFFSETS = np.array([-90.0, 0.0, 90.0], np.float32)


@pytest.fixture()
def dev(gpu):
    try:
        yield torch.device("cuda:0")
    finally:
        gpu.set_engine(0, 0)
        gpu.set_tuning(0, 0, 0)


def run(gpu, p, x, y, yaw, r, q, max_events=64):
    """(grids, origins, n_events, events, stats, launches, scores) of uqs_replay_recentering_frontier_dev"""
    F, N = x.shape
    t = [torch.from_numpy(np.ascontiguousarray(a, np.float32)).cuda() for a in (x, y, yaw, r.reshape(F, N, 32))]
    grids = torch.full((F, p.H, p.W), 55, dtype=torch.int8, device="cuda")
    origins = torch.zeros((F, 2), dtype=torch.float32, device="cuda")
    n_ev = torch.zeros(F, dtype=torch.int32, device="cuda")
    events = torch.full((F, max(max_events, 1), 3), -7, dtype=torch.int32, device="cuda")
    tq = torch.from_numpy(np.ascontiguousarray(q).view(np.uint8)).cuda() if q.size else None
    ts = torch.full((max(q.size, 1),), -12345, dtype=torch.int32, device="cuda")
    torch.cuda.synchronize()
    l0 = gpu.kernel_launches()
    st = gpu.replay_recentering_frontier_dev(p, F, N, *(a.data_ptr() for a in t), grids.data_ptr(), origins.data_ptr(),
                                             n_ev.data_ptr(), events.data_ptr() if max_events else 0, max_events, q.size,
                                             tq.data_ptr() if q.size else 0, ts.data_ptr() if q.size else 0, want_stats=True)
    launches = gpu.kernel_launches() - l0
    torch.cuda.synchronize()
    return (grids.cpu().numpy(), origins.cpu().numpy(), n_ev.cpu().numpy(), events.cpu().numpy(), st, launches,
            ts.cpu().numpy()[:q.size])


def same_as_plain(got, plain, what):
    for a, b, name in zip(got[:5], plain[:5], ("grids", "origins", "n_events", "events", "stats")):
        if isinstance(a, np.ndarray):
            assert np.array_equal(a.view(np.uint8), b.view(np.uint8)), (what, name, first_diff(a, b) if name == "grids" else "")
        else:
            assert a == b, (what, name)


def assert_scores(got, want, q, what):
    bad = np.flatnonzero(got != want)
    assert bad.size == 0, f"{what}: {bad.size} of {q.size} scores differ; first query {q[bad[0]]}: got {got[bad[0]]} want {want[bad[0]]}"


class Walk:
    """One flight stepped frame by frame with the oracle: the grid kept at chosen frames, and, in global coordinates
    (window cell + S), the last frame at which each non-zero cell left the window."""

    def __init__(self, oracle, p, x, y, yaw, r, keep=()):
        L = oracle.L
        L.orc_recentre_if_needed.argtypes = [ctypes.c_void_p, ctypes.c_void_p, ctypes.c_float, ctypes.c_float,
                                             ctypes.POINTER(ctypes.c_int), ctypes.POINTER(ctypes.c_int)]
        L.orc_recenter_shift.argtypes = [ctypes.c_void_p, ctypes.c_void_p, ctypes.c_int, ctypes.c_int]
        L.orc_recenter_shift.restype = None
        ev = events_of(oracle, p, x, y)
        S = np.concatenate([[[0, 0]], np.cumsum(ev[:, 1:], axis=0)]).astype(np.int64)
        self.smin = S.min(axis=0)
        span = S.max(axis=0) - self.smin
        self.erased = np.full((p.H + span[1], p.W + span[0]), -1, np.int32)
        self.grids, self.origins, self.S = {}, [], []
        s = p.copy()
        grid = np.zeros((p.H, p.W), np.int8)
        Sx = Sy = 0
        sx, sy = ctypes.c_int(0), ctypes.c_int(0)
        for i in range(x.size):
            before = grid.copy()
            if L.orc_recentre_if_needed(ctypes.byref(s), grid.ctypes.data, x[i], y[i], ctypes.byref(sx), ctypes.byref(sy)):
                kept = np.zeros_like(before, bool)          # source cells some destination reads
                kept[max(sy.value, 0):p.H + min(sy.value, 0), max(sx.value, 0):p.W + min(sx.value, 0)] = True
                gy, gx = np.nonzero((before != 0) & ~kept)
                self.erased[gy + Sy - self.smin[1], gx + Sx - self.smin[0]] = i
                Sx += sx.value
                Sy += sy.value
            L.orc_frame(ctypes.byref(s), grid.ctypes.data, x[i], y[i], yaw[i], r[i].ctypes.data)
            self.origins.append((np.float32(s.origin_x), np.float32(s.origin_y)))
            self.S.append((Sx, Sy))
            if i in keep:
                self.grids[i] = grid.copy()
        self.events = ev


def sample_cells(oracle, p, origin, qx, qy, yaw, off):
    """Window cells of a query's samples (numpy float32 angles: close to, not always exactly, the restated sincosf)."""
    q = p.copy()
    q.origin_x, q.origin_y = origin
    out = []
    step = np.float32(p.res_m) * np.float32(2.0)
    for fan in (0.0, 15.0, -15.0):
        a = np.float32(np.float32(np.float32(yaw) + np.float32(off)) + np.float32(fan)) * np.float32(np.float32(np.pi) / np.float32(180.0))
        cs, sn = np.float32(np.cos(np.float64(a))), np.float32(np.sin(np.float64(a)))
        d = step
        while d <= np.float32(2.5):
            ok, gx, gy = oracle.world_to_grid(q, np.float32(qx + d * cs), np.float32(qy + d * sn))
            if not ok:
                break
            out.append((gx, gy))
            d = np.float32(d + step)
    return out


def hazard_queries(oracle, pkg, p, x, y, yaw, r, flights, rng):
    """Queries on `flights` where the order of events and probes decides the score:
    hazard 2 -- at frame e - 1, posed in the strip the event at frame e erases, with the grid at e - 1 kept;
    hazard 1 -- at frames after an event, posed where the flight was before it (cells erased and re-entered)."""
    out, walks = [], {}
    for f in flights:
        ev = events_of(oracle, p, x[f], y[f])
        walks[f] = w = Walk(oracle, p, x[f], y[f], yaw[f], r[f], keep=set(int(e) - 1 for e in ev[:, 0] if e > 0))
        half = np.array([p.W // 2, p.H // 2])
        for e, sx, sy in ev:
            if e == 0:
                continue
            ox, oy = w.origins[e - 1]
            gx = sx // 2 if sx > 0 else p.W - 1 + sx // 2 if sx < 0 else rng.integers(0, p.W)
            gy = sy // 2 if sy > 0 else p.H - 1 + sy // 2 if sy < 0 else rng.integers(0, p.H)
            for k in range(6):
                jx, jy = rng.integers(-2, 3, 2)
                qx = np.float32(ox + np.float32(int(gx + jx) - half[0]) * np.float32(p.res_m)) if sx else x[f, e - 1]
                qy = np.float32(oy + np.float32(int(gy + jy) - half[1]) * np.float32(p.res_m)) if sy else y[f, e - 1]
                out.append((f, e - 1, qx, qy, rng.uniform(-180, 180), rng.choice(OFFSETS)))
        for e in ev[:, 0]:
            for p_fr in (e, e + 1, e + 7, e + 40):
                if p_fr >= x.shape[1]:
                    continue
                for j in rng.integers(0, max(p_fr, 1), 3):                  # where the flight was before
                    out.append((f, p_fr, x[f, j], y[f, j], rng.uniform(-180, 180), rng.choice(OFFSETS)))
                # on cells that left the window at or before p_fr and are inside it again
                (Sx, Sy), (ox, oy) = w.S[p_fr], w.origins[p_fr]
                x0, y0 = Sx - w.smin[0], Sy - w.smin[1]
                era = w.erased[y0:y0 + p.H, x0:x0 + p.W]
                cy, cx = np.nonzero((era >= 0) & (era <= p_fr))
                for k in rng.permutation(cy.size)[:6]:
                    out.append((f, p_fr, np.float32(ox + np.float32(int(cx[k]) - half[0]) * np.float32(p.res_m)),
                                np.float32(oy + np.float32(int(cy[k]) - half[1]) * np.float32(p.res_m)),
                                rng.uniform(-180, 180), rng.choice(OFFSETS)))
    a = np.array(out, dtype=object)
    q = pkg.make_queries(a[:, 0].astype(np.int32), a[:, 1].astype(np.int32), a[:, 2].astype(np.float32),
                         a[:, 3].astype(np.float32), a[:, 4].astype(np.float32), a[:, 5].astype(np.float32))
    return q, walks


def check_hazards_are_hit(oracle, p, q, walks):
    """Hazard 2: some strip queries score differently on their grid shifted out and back (the erased cells zeroed).
    Hazard 1: some queries sample a non-zero cell that left the window at or before their frame."""
    L = oracle.L
    differ = reentered = 0
    for i in range(q.size):
        f, fr = int(q["flight"][i]), int(q["frame"][i])
        w = walks[f]
        if fr in w.grids and fr + 1 in set(int(e) for e in w.events[:, 0]):
            e = w.events[w.events[:, 0] == fr + 1][0]
            g = w.grids[fr]
            s = p.copy()
            s.origin_x, s.origin_y = w.origins[fr]
            g2 = g.copy()
            L.orc_recenter_shift(ctypes.byref(p), g2.ctypes.data, int(e[1]), int(e[2]))
            L.orc_recenter_shift(ctypes.byref(p), g2.ctypes.data, -int(e[1]), -int(e[2]))
            args = (q["x"][i], q["y"][i], q["yaw_deg"][i], q["offset_deg"][i])
            differ += oracle.frontier_score(s, g, *args) != oracle.frontier_score(s, g2, *args)
        Sx, Sy = w.S[fr]
        for gx, gy in sample_cells(oracle, p, w.origins[fr], q["x"][i], q["y"][i], q["yaw_deg"][i], q["offset_deg"][i]):
            if 0 <= w.erased[gy + Sy - w.smin[1], gx + Sx - w.smin[0]] <= fr:
                reentered += 1
                break
    assert differ > 0 and reentered > 0, (differ, reentered)
    return differ, reentered


@pytest.mark.parametrize("geom", [(400, "0.05", 20.0), (500, "0.10", 50.0)])
def test_fleet_on_both_routes(gpu, oracle, pkg, synth, dev, geom):
    W, res, size = geom
    F, N = 64, 1200
    p, x, y, yaw, r = fleet(synth, F, N, W, res, size, seed=7 + W)
    rng = np.random.default_rng(W)
    hq, walks = hazard_queries(oracle, pkg, p, x, y, yaw, r, [2, 3, 4, 5, 6, 9], rng)
    around = []
    for f in range(F):
        ev = events_of(oracle, p, x[f], y[f])[:, 0]
        fr = np.unique(np.concatenate([ev, np.maximum(ev - 1, 0)])).astype(np.int32)
        around.append(pkg.make_queries(f, fr, x[f, fr], y[f, fr], yaw[f, fr], rng.choice(OFFSETS, fr.size)))
    pile = pkg.make_queries(3, N // 2, x[3, N // 2], y[3, N // 2], rng.uniform(-180, 180, 300).astype(np.float32),
                            rng.choice(OFFSETS, 300))
    q = np.concatenate([hostile_queries(rng, pkg, p, x, y, yaw, 1500), hq, pile] + around)
    q = np.concatenate([q, q[rng.integers(0, q.size, 200)]])
    q = q[rng.permutation(q.size)]
    assert 2 in q["flight"][q["frame"] == 0] and np.isnan(q["yaw_deg"]).any()
    want = recentering_scores_at_frames(oracle, p, x, y, yaw, r, q)
    assert len(set(want.tolist())) > 30
    check_hazards_are_hit(oracle, p, hq, walks)
    for engine, tune in ROUTE_A + ROUTE_B:
        gpu.set_engine(engine, 0)
        gpu.set_tuning(*tune)
        got = run(gpu, p, x, y, yaw, r, q)
        assert_scores(got[6], want, q, (engine, tune))
        same_as_plain(got, run_plain(gpu, p, x, y, yaw, r), (engine, tune))
        if (engine, tune) in ROUTE_A:
            few = run(gpu, p, x, y, yaw, r, q[:7])
            assert few[5] == got[5] < 24, (engine, tune, few[5], got[5])
            assert_scores(few[6], want[:7], q[:7], (engine, tune, "few"))
    # flights that never recentre: the same scores as uqs_replay_frontier_dev at the fixed origin
    gpu.set_engine(0, 0)
    gpu.set_tuning(0, 0, 0)
    q01 = q[q["flight"] < 2]
    _, s_fixed, _ = gpu.replay_frontier(p, x[:2], y[:2], yaw[:2], r[:2], q01)
    assert np.array_equal(run(gpu, p, x[:2], y[:2], yaw[:2], r[:2], q01)[6], s_fixed)


def test_no_queries_bad_queries_and_bad_arguments(gpu, oracle, pkg, synth, dev):
    p, x, y, yaw, r = fleet(synth, 8, 400, 400, "0.05", 20.0, seed=11)
    F, N = x.shape
    empty = pkg.make_queries([], [], [], [], [], [])
    same_as_plain(run(gpu, p, x, y, yaw, r, empty), run_plain(gpu, p, x, y, yaw, r), "no queries")
    t = [torch.from_numpy(np.ascontiguousarray(a)).cuda() for a in (x, y, yaw, r)]
    outs = [torch.full((F, p.H, p.W), 9, dtype=torch.int8, device="cuda"), torch.full((F, 2), 9.0, device="cuda"),
            torch.full((F,), 9, dtype=torch.int32, device="cuda"), torch.full((F, 4, 3), 9, dtype=torch.int32, device="cuda"),
            torch.full((4,), 9, dtype=torch.int32, device="cuda")]
    L = pkg.lib()
    for bad in ((8, 0), (-1, 0), (0, N), (1, -5)):
        q = pkg.make_queries([0, 1, bad[0], 0], [3, 5, bad[1], N], 0.0, 0.0, 0.0, 0.0)
        tq = torch.from_numpy(q.view(np.uint8)).cuda()
        with pytest.raises(pkg.UqsError) as e:
            gpu.replay_recentering_frontier_dev(p, F, N, *(a.data_ptr() for a in t), *(o.data_ptr() for o in outs[:4]), 4, 4,
                                                tq.data_ptr(), outs[4].data_ptr(), want_stats=True)
        assert e.value.code == pkg.ERR_BAD_ARG and "query 2" in str(e.value)
    q = pkg.make_queries([0, 1], [3, 5], 0.0, 0.0, 0.0, 0.0)
    tq = torch.from_numpy(q.view(np.uint8)).cuda()
    ptr = [a.data_ptr() for a in t] + [o.data_ptr() for o in outs[:4]]
    torch.cuda.synchronize()
    for i in list(range(8)) + [8, 9]:
        args = list(ptr) + [tq.data_ptr(), outs[4].data_ptr()]
        args[i] = None
        rc = L.uqs_replay_recentering_frontier_dev(ctypes.byref(p), F, N, *args[:8], 4, 2, *args[8:], None)
        assert rc == gpu.ERR_BAD_ARG, i
    gpu.set_engine(2, 0)
    with pytest.raises(pkg.UqsError) as e:
        gpu.replay_recentering_frontier_dev(p, F, N, *ptr, 4, 2, tq.data_ptr(), outs[4].data_ptr(), want_stats=True)
    assert e.value.code == pkg.ERR_BAD_ARG and "engine 2" in str(e.value)
    torch.cuda.synchronize()
    assert all(bool((o == 9).all()) for o in outs)
    # host-buffer form, with and without the grid and origin outputs
    gpu.set_engine(0, 0)
    q = hostile_queries(np.random.default_rng(4), pkg, p, x, y, yaw, 300)
    grids, origins, scores, st = gpu.replay_recentering_frontier(p, x, y, yaw, r, q)
    plain = run_plain(gpu, p, x, y, yaw, r)
    assert np.array_equal(grids, plain[0]) and np.array_equal(origins, plain[1]) and st == plain[4]
    assert_scores(scores, recentering_scores_at_frames(oracle, p, x, y, yaw, r, q), q, "host form")
    assert np.array_equal(gpu.replay_recentering_frontier(p, x, y, yaw, r, q, want_grids=False)[2], scores)


def test_dropin_route_agrees(gpu, oracle, pkg, synth, dev):
    """map_recentre_if_needed + map_update_from_beams + frontier_score_dir, as log_tick and control_tick call them, give
    what the batch call gives at the same instants."""
    from test_next_rows_cpu import wandering_log
    w, d, x, y = wandering_log(synth, n=900, speed=9.0)
    p = w.params()
    yaw, r = d["yaw_deg"][0], d["ranges"][0]
    di = gpu.DropIn(p)
    di.hover_init(float(x[0]), float(y[0]))
    q = p.copy()
    q.origin_x, q.origin_y = x[0], y[0]
    inst = []
    for i in range(900):
        di.set_beams(r[i])
        di.map_recentre_if_needed(x[i], y[i])
        di.map_update_from_beams(x[i], y[i], yaw[i])
        if i % 30 == 29:
            for off in (-90.0, 0.0, 90.0):
                inst.append((i, off, di.frontier_score_dir(x[i], y[i], yaw[i], off)))
    qs = pkg.make_queries(0, [i for i, _, _ in inst], [x[i] for i, _, _ in inst], [y[i] for i, _, _ in inst],
                          [yaw[i] for i, _, _ in inst], [o for _, o, _ in inst])
    grids, origins, scores, _ = gpu.replay_recentering_frontier(q, x[None], y[None], yaw[None], r[None], qs)
    assert np.array_equal(grids[0], di.grid()) and np.float32(origins[0, 0]) == np.float32(di.origin()[0])
    assert len(events_of(oracle, q, x, y)) >= 2
    assert scores.tolist() == [s for _, _, s in inst]


def test_one_long_log_one_query_per_second(gpu, oracle, pkg, synth, dev):
    w = synth.Workload("wander", 3, 1, 30000, 400, "0.05", 20.0, 50.0)
    d = synth.generate(w)
    p = w.params()
    t = np.arange(30000, dtype=np.float32) / np.float32(50.0)
    x = (d["x_true"][0] + np.float32(1.3) * t * np.cos(t / np.float32(90.0))).astype(np.float32)[None]
    y = (d["y_true"][0] + np.float32(1.1) * t * np.sin(t / np.float32(70.0))).astype(np.float32)[None]
    yaw, r = d["yaw_deg"][:1], d["ranges"][:1]
    fr = np.arange(49, 30000, 50, dtype=np.int32)
    rng = np.random.default_rng(2)
    q = pkg.make_queries(0, fr, x[0, fr], y[0, fr], yaw[0, fr], rng.choice(OFFSETS, fr.size))
    q = q[rng.permutation(q.size)]
    assert len(events_of(oracle, p, x[0], y[0])) > 50
    want = recentering_scores_at_frames(oracle, p, x, y, yaw, r, q)
    assert len(set(want.tolist())) > 20
    for engine, tune in [(0, (0, 0, 0)), (3, (0, 0, 0))]:
        gpu.set_engine(engine, 0)
        gpu.set_tuning(*tune)
        got = run(gpu, p, x, y, yaw, r, q, max_events=4096)
        assert_scores(got[6], want, q, (engine, tune))
        same_as_plain(got, run_plain(gpu, p, x, y, yaw, r, max_events=4096), (engine, tune))
        assert got[5] >= 16                                          # the segment route


def test_many_flights_across_internal_chunks(gpu, oracle, pkg, synth, dev):
    """65535 + 45 flights: queries on flights either side of the ray set-up's 65535-flight chunk boundary."""
    F, N = 65535 + 45, 24
    p = gpu.make_params(64, 64, 0.05, size_m=3.2)
    rng = np.random.default_rng(4)
    tt = np.arange(N, dtype=np.float32)[None] * np.float32(0.1)
    x = (rng.uniform(-1, 1, (F, 1)) + rng.uniform(-1, 1, (F, 1)) * tt).astype(np.float32)
    y = (rng.uniform(-1, 1, (F, 1)) + rng.uniform(-1, 1, (F, 1)) * tt).astype(np.float32)
    yaw = rng.uniform(-180, 180, (F, N)).astype(np.float32)
    r = rng.uniform(0.1, 2.0, (F, N, 32)).astype(np.float32)
    fl = np.repeat(np.arange(65525, 65545, dtype=np.int32), 30)
    fr = rng.integers(0, N, fl.size).astype(np.int32)
    q = pkg.make_queries(fl, fr, x[fl, fr], y[fl, fr], yaw[fl, fr], rng.choice(OFFSETS, fl.size))
    got = run(gpu, p, x, y, yaw, r, q, max_events=8)
    assert got[5] < 24
    assert_scores(got[6], recentering_scores_at_frames(oracle, p, x, y, yaw, r, q), q, "many flights")
    assert got[2][65525:65545].sum() > 0


def test_under_the_bounds_checked_build(pkg):
    """This file once more under -DUQS_DEBUG_BOUNDS (the probe reads of the recentering sub-tile engine checked against
    the warp's sub-tile), without the many-flight case."""
    dbg = os.path.join(ROOT, "micro-quad-slam_b200", "libuqs_mapping_dbg.so")
    assert os.path.exists(dbg)
    env = dict(os.environ, UQS_LIBRARY=dbg)
    res = subprocess.run([sys.executable, "-m", "pytest", os.path.abspath(__file__), "-q", "-x", "-m", "gpu", "-k",
                          "not many_flights and not bounds_checked", "-p", "no:cacheprovider"], capture_output=True, text=True,
                         env=env, timeout=2400, cwd=ROOT)
    tail = res.stdout[-3000:] + res.stderr[-2000:]
    assert res.returncode == 0 and "UQS_DEBUG_BOUNDS" not in res.stdout + res.stderr, tail
    assert " passed" in res.stdout and "failed" not in res.stdout, tail
