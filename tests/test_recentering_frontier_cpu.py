"""Frontier queries at their frame on recentred maps (uqs_replay_recentering_frontier) on the CPU: the statement
"score after log_tick() of frames 0..frame, at the running origin" as a frame-by-frame composition of the already-pinned
orc_recentre_if_needed, orc_frame and orc_frontier_score_dir, pinned on every machine to orc_replay_recentering replayed
up to each query's frame and, where it is built, to the reference's own code; the no-device errors of both entry
points."""
import ctypes

import numpy as np
import pytest

from conftest import have_ref
from test_frontier_replay_cpu import hostile_queries


def recentering_walk(oracle, p, x, y, yaw, ranges, queries):
    """One flight's log_tick() with recentering (orc_recentre_if_needed, then orc_frame), every query of frame i (the
    flight field is not read) scored by orc_frontier_score_dir on the running grid and origin right after frame i.
    Returns (grid, origin (x, y), n_events, updates, scores in input order); p is not modified."""
    L = oracle.L
    L.orc_recentre_if_needed.argtypes = [ctypes.c_void_p, ctypes.c_void_p, ctypes.c_float, ctypes.c_float,
                                         ctypes.POINTER(ctypes.c_int), ctypes.POINTER(ctypes.c_int)]
    x, y, yaw = (np.ascontiguousarray(a, np.float32).ravel() for a in (x, y, yaw))
    ranges = np.ascontiguousarray(ranges, np.float32).reshape(x.size, 32)
    s = p.copy()
    grid = np.zeros((p.H, p.W), np.int8)
    order = np.argsort(queries["frame"], kind="stable")
    scores = np.zeros(queries.size, np.int32)
    n_ev = U = k = 0
    for i in range(x.size):
        n_ev += L.orc_recentre_if_needed(ctypes.byref(s), grid.ctypes.data, x[i], y[i], None, None)
        U += L.orc_frame(ctypes.byref(s), grid.ctypes.data, x[i], y[i], yaw[i], ranges[i].ctypes.data)
        while k < order.size and queries["frame"][order[k]] <= i:
            q = queries[order[k]]
            if q["frame"] == i:
                scores[order[k]] = oracle.frontier_score(s, grid, q["x"], q["y"], q["yaw_deg"], q["offset_deg"])
            k += 1
    return grid, (float(s.origin_x), float(s.origin_y)), int(n_ev), int(U), scores


def recentering_scores_at_frames(oracle, p, x, y, yaw, ranges, queries):
    """Scores of ``queries`` (QUERY_DTYPE, input order) against each flight's recentred map right after the query's
    frame, flight by flight (each flight walked up to its last query's frame)."""
    scores = np.zeros(queries.size, np.int32)
    for f in np.unique(queries["flight"]):
        mine = np.flatnonzero(queries["flight"] == f)
        n = int(queries["frame"][mine].max()) + 1
        scores[mine] = recentering_walk(oracle, p, x[f, :n], y[f, :n], yaw[f, :n], ranges[f, :n], queries[mine])[4]
    return scores


def drifting(synth, F, N, W, res, size, seed):
    """wandering_log-style poses drifting away from the origin: every flight recentres several times."""
    w = synth.Workload("wander", seed, F, N, W, res, size, 50.0)
    d = synth.generate(w)
    rng = np.random.default_rng(seed)
    t = (np.arange(N, dtype=np.float32) / np.float32(50.0))[None]
    speed = rng.uniform(2.0, 6.0, (F, 1)).astype(np.float32)
    head = rng.uniform(-np.pi, np.pi, (F, 1)).astype(np.float32)
    x = (d["x_true"] + speed * np.cos(head) * t).astype(np.float32)
    y = (d["y_true"] + speed * np.sin(head) * t).astype(np.float32)
    return w.params(), x, y, d["yaw_deg"], np.ascontiguousarray(d["ranges"])


def queries_around_events(rng, pkg, oracle, p, x, y, yaw, n):
    """hostile_queries plus, for every event of every flight, queries at the event's frame and the frame before."""
    q = [hostile_queries(rng, pkg, p, x, y, yaw, n)]
    for f in range(x.shape[0]):
        frames = events_of(oracle, p, x[f], y[f])[:, 0]
        fr = np.unique(np.concatenate([frames, np.maximum(frames - 1, 0)])).astype(np.int32)
        q.append(pkg.make_queries(f, fr, x[f, fr], y[f, fr], yaw[f, fr], rng.choice([-90.0, 0.0, 90.0], fr.size)))
    q = np.concatenate(q)
    return q[rng.permutation(q.size)]


def events_of(oracle, p, x, y):
    """[[frame, sx, sy], ...] of one flight: orc_recentre_if_needed on a 2x2 grid (the decision reads the poses only)."""
    L = oracle.L
    L.orc_recentre_if_needed.argtypes = [ctypes.c_void_p, ctypes.c_void_p, ctypes.c_float, ctypes.c_float,
                                         ctypes.POINTER(ctypes.c_int), ctypes.POINTER(ctypes.c_int)]
    q = p.copy()
    q.W = q.H = 2
    g = np.zeros(4, np.int8)
    sx, sy = ctypes.c_int(0), ctypes.c_int(0)
    out = [(i, sx.value, sy.value) for i in range(x.size)
           if L.orc_recentre_if_needed(ctypes.byref(q), g.ctypes.data, x[i], y[i], ctypes.byref(sx), ctypes.byref(sy))]
    return np.asarray(out, np.int32).reshape(-1, 3)


def test_statement_equals_replays_up_to_each_frame(oracle, pkg, synth):
    """The frame-by-frame statement against orc_replay_recentering replayed over frames 0..f for every query frame f,
    scored at the origin that replay ends on; and its final grid, origin, events and updates against the whole log."""
    p, x, y, yaw, r = drifting(synth, 3, 400, 400, "0.05", 20.0, seed=21)
    x[2, 0] += np.float32(0.8 * p.size_m)                       # an event at frame 0
    rng = np.random.default_rng(5)
    q = queries_around_events(rng, pkg, oracle, p, x, y, yaw, 150)
    got = recentering_scores_at_frames(oracle, p, x, y, yaw, r, q)
    assert len(set(got.tolist())) > 10
    for f in range(3):
        mine = np.flatnonzero(q["flight"] == f)
        for fr in np.unique(q["frame"][mine]):
            g, o, _, _ = oracle.replay_recentering(p, x[f, :fr + 1], y[f, :fr + 1], yaw[f, :fr + 1], r[f, :fr + 1])
            s = p.copy()
            s.origin_x, s.origin_y = np.float32(o[0]), np.float32(o[1])
            for k in mine[q["frame"][mine] == fr]:
                assert got[k] == oracle.frontier_score(s, g, q["x"][k], q["y"][k], q["yaw_deg"][k], q["offset_deg"][k]), (f, fr, k)
        g2, o2, n2, u2, _ = recentering_walk(oracle, p, x[f], y[f], yaw[f], r[f], q[mine])
        g3, o3, n3, u3 = oracle.replay_recentering(p, x[f], y[f], yaw[f], r[f])
        assert np.array_equal(g2, g3) and (o2, n2, u2) == (o3, n3, u3) and n2 > 0


def test_oracle_equals_reference(orc_mod, oracle, pkg, synth):
    if not have_ref(orc_mod, 400, 400, "0.05"):
        pytest.skip("oracle/_ref not built (needs the reference source)")
    ref = orc_mod.Reference(400, 400, "0.05")
    p, x, y, yaw, r = drifting(synth, 2, 700, 400, "0.05", 20.0, seed=33)
    rng = np.random.default_rng(8)
    q = queries_around_events(rng, pkg, oracle, p, x, y, yaw, 200)
    got = recentering_scores_at_frames(oracle, p, x, y, yaw, r, q)
    for f in range(2):
        ref.reset(0.0, 0.0)
        mine = sorted(np.flatnonzero(q["flight"] == f), key=lambda i: int(q["frame"][i]))
        done = 0
        for i in mine:
            while done <= q["frame"][i]:
                ref.frame(x[f, done], y[f, done], yaw[f, done], r[f, done], allow_recenter=True)
                done += 1
            assert got[i] == ref.frontier_score(q["x"][i], q["y"][i], q["yaw_deg"][i], q["offset_deg"][i]), i
    assert len(set(got.tolist())) > 10


def test_symbols_are_exported(pkg):
    names = pkg.exported_symbols()
    assert "uqs_replay_recentering_frontier_dev" in names and "uqs_replay_recentering_frontier" in names


def test_entry_points_fail_without_a_device(pkg):
    import torch
    if torch.cuda.is_available():
        pytest.skip("a GPU is present")
    with pytest.raises(pkg.UqsError):
        pkg.init(0)
    p = pkg.make_params(400, 400, 0.05, size_m=20.0)
    z = np.zeros((1, 4), np.float32)
    q = pkg.make_queries(0, 0, 0.0, 0.0, 0.0, 0.0)
    with pytest.raises(pkg.UqsError) as e:
        pkg.replay_recentering_frontier(p, z, z, z, np.zeros((1, 4, 32), np.float32), q)
    assert e.value.code == pkg.ERR_NOT_INIT
    L = pkg.lib()
    st = pkg.Stats()
    good = [ctypes.c_void_p(16)] * 8
    for F, N, bufs, nq in [(1, 4, good, 1), (1, 4, good, 0), (0, 4, good, 1), (1, 4, [None] * 8, 1), (1, 4, good, -1)]:
        rc = L.uqs_replay_recentering_frontier_dev(ctypes.byref(p), F, N, *bufs, 0, nq, ctypes.c_void_p(16), ctypes.c_void_p(16),
                                                   ctypes.byref(st))
        assert rc == pkg.ERR_NOT_INIT, (F, N, nq)
    rc = L.uqs_replay_recentering_frontier(ctypes.byref(p), 1, 4, *([ctypes.c_void_p(16)] * 6), 1, ctypes.c_void_p(16),
                                           ctypes.c_void_p(16), ctypes.byref(st))
    assert rc == pkg.ERR_NOT_INIT
