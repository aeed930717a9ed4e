"""uqs_replay_frontier[_dev] on the device: every score against the oracle's statement of "the map as it stood after
the query's frame" (pinned to the reference in tests/test_frontier_replay_cpu.py), every grid and the stats against
uqs_replay_dev on the same inputs, byte for byte -- across the engines, their geometries and time slices, hostile
queries, start grids, and the full-size drift ensemble."""
import multiprocessing as mp
import os
import subprocess
import sys

import numpy as np
import pytest
import torch

from conftest import first_diff
from test_frontier_replay_cpu import hostile_queries, oracle_scores_at_frames
from test_next_rows_cpu import wandering_log

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


@pytest.fixture()
def dev(gpu):
    gpu.set_stream(torch.cuda.current_stream().cuda_stream)
    yield torch.device("cuda:0")
    gpu.set_stream(None)
    gpu.set_engine(0, 0)
    gpu.set_tuning(0, 0, 0)


def both(gpu, p, x, y, yaw, ranges, q, start=None):
    """(grids of uqs_replay_dev, grids of uqs_replay_frontier_dev, their stats, the scores)"""
    d = torch.device("cuda:0")
    F, N = x.shape
    t = [torch.from_numpy(np.ascontiguousarray(a, np.float32)).to(d) for a in (x, y, yaw, ranges)]
    g0 = torch.zeros((F, p.H, p.W), dtype=torch.int8, device=d) if start is None else torch.from_numpy(start).to(d)
    g1 = g0.clone()
    acc = start is not None
    st0 = gpu.replay_dev(p, F, N, *(a.data_ptr() for a in t), g0.data_ptr(), accumulate=acc, want_stats=True)
    tq = torch.from_numpy(np.ascontiguousarray(q).view(np.uint8)).to(d)
    ts = torch.full((q.size,), -12345, dtype=torch.int32, device=d)
    st1 = gpu.replay_frontier_dev(p, F, N, *(a.data_ptr() for a in t), g1.data_ptr(), q.size, tq.data_ptr(), ts.data_ptr(),
                                  accumulate=acc, want_stats=True)
    return g0.cpu().numpy(), g1.cpu().numpy(), st0, st1, ts.cpu().numpy()


def check(gpu, oracle, p, x, y, yaw, ranges, q, start=None, want=None):
    g0, g1, st0, st1, scores = both(gpu, p, x, y, yaw, ranges, q, start)
    assert np.array_equal(g0, g1), first_diff(g1, g0)
    assert st0 == st1
    if want is None:
        want = oracle_scores_at_frames(oracle, p, x, y, yaw, ranges, q, start)
    bad = np.flatnonzero(scores != want)
    assert bad.size == 0, f"{bad.size} of {q.size} scores differ; first query {q[bad[0]]}: got {scores[bad[0]]} want {want[bad[0]]}"
    return g1, scores, want


def small(synth, F=6, N=900, seed_cfg="c1"):
    w = synth.scaled(synth.CONFIGS[seed_cfg], n_flights=F, n_samples=N)
    d = synth.generate(w)
    return w.params(), d["x_true"], d["y_true"], d["frame_yaw_deg"], np.ascontiguousarray(d["ranges"])


@pytest.mark.parametrize("engine,warps", [(0, 0), (1, 0), (2, 4), (2, 8), (2, 16), (2, 32), (3, 0)])
def test_engines_and_resident_warps(gpu, oracle, pkg, synth, dev, engine, warps):
    p, x, y, yaw, r = small(synth)
    r[5] = np.nan                                                # a flight without an accepted ray (empty box)
    gpu.set_engine(engine, warps)
    q = hostile_queries(np.random.default_rng(100 + engine * 40 + warps), pkg, p, x, y, yaw, 1500)
    _, scores, _ = check(gpu, oracle, p, x, y, yaw, r, q)
    assert len(set(scores.tolist())) > 20


@pytest.mark.parametrize("sw,sh", [(16, 16), (40, 56), (64, 100), (400, 8), (7, 33)])
def test_subtile_sizes(gpu, oracle, pkg, synth, dev, sw, sh):
    p, x, y, yaw, r = small(synth, F=3)
    gpu.set_engine(1, 0)
    gpu.set_tuning(sw, sh, 1)
    q = hostile_queries(np.random.default_rng(sw * 7 + sh), pkg, p, x, y, yaw, 900)
    check(gpu, oracle, p, x, y, yaw, r, q)


@pytest.mark.parametrize("S", [1, 2, 7, 64])
def test_time_slices_on_a_long_log(gpu, oracle, pkg, synth, dev, S):
    w = synth.scaled(synth.CONFIGS["c2"], n_samples=24000)
    d = synth.generate(w)
    p, x, y, yaw, r = w.params(), d["x_true"], d["y_true"], d["frame_yaw_deg"], np.ascontiguousarray(d["ranges"])
    N = x.shape[1]
    gpu.set_engine(1, 0)
    gpu.set_tuning(0, 0, S)
    rng = np.random.default_rng(S)
    gps = ((N + 31) // 32 + S - 1) // S
    edges = [e for s in range(1, S) for e in (s * gps * 32 - 1, s * gps * 32) if e < N]
    frames = np.concatenate([rng.integers(0, N, 600), [0, N - 1], edges]).astype(np.int32)
    q = pkg.make_queries(0, frames, x[0, frames], y[0, frames], yaw[0, frames], rng.choice([-90.0, 0.0, 90.0], frames.size))
    q = q[rng.permutation(q.size)]
    _, scores, _ = check(gpu, oracle, p, x, y, yaw, r, q)
    assert len(set(scores.tolist())) > 20


@pytest.mark.parametrize("engine", [0, 1, 2])
def test_accumulate_onto_start_grids(gpu, oracle, pkg, synth, dev, engine):
    p, x, y, yaw, r = small(synth, F=4, N=600)
    gpu.set_engine(engine, 0)
    rng = np.random.default_rng(9 + engine)
    start = rng.integers(-60, 60, (4, p.H, p.W)).astype(np.int8)
    q = hostile_queries(rng, pkg, p, x, y, yaw, 800)
    check(gpu, oracle, p, x, y, yaw, r, q, start)
    start[2, 10:50, 10:50] = 127                                 # outside [lo_min, lo_max]: the unrestricted engine
    start[1, 200, 200] = -128
    check(gpu, oracle, p, x, y, yaw, r, q, start)


def test_bad_queries_and_no_queries(gpu, oracle, pkg, synth, dev):
    p, x, y, yaw, r = small(synth, F=2, N=300)
    F, N = x.shape
    d = torch.device("cuda:0")
    t = [torch.from_numpy(np.ascontiguousarray(a, np.float32)).to(d) for a in (x, y, yaw, r)]
    for bad in ((2, 0), (-1, 0), (0, N), (1, -5)):
        q = pkg.make_queries([0, 1, bad[0], 0], [3, 5, bad[1], N], 0.0, 0.0, 0.0, 0.0)
        start = np.full((F, p.H, p.W), 7, np.int8)
        g = torch.from_numpy(start).to(d)
        tq = torch.from_numpy(q.view(np.uint8)).to(d)
        ts = torch.zeros(4, dtype=torch.int32, device=d)
        with pytest.raises(pkg.UqsError) as e:
            gpu.replay_frontier_dev(p, F, N, *(a.data_ptr() for a in t), g.data_ptr(), 4, tq.data_ptr(), ts.data_ptr(),
                                    accumulate=True, want_stats=True)
        assert e.value.code == pkg.ERR_BAD_ARG and "query 2" in str(e.value)
        assert np.array_equal(g.cpu().numpy(), start)
    g0 = torch.zeros((F, p.H, p.W), dtype=torch.int8, device=d)
    g1 = torch.full((F, p.H, p.W), 3, dtype=torch.int8, device=d)
    st0 = gpu.replay_dev(p, F, N, *(a.data_ptr() for a in t), g0.data_ptr(), want_stats=True)
    st1 = gpu.replay_frontier_dev(p, F, N, *(a.data_ptr() for a in t), g1.data_ptr(), 0, 0, 0, want_stats=True)
    assert st0 == st1 and torch.equal(g0, g1)
    # host-buffer form
    q = hostile_queries(np.random.default_rng(4), pkg, p, x, y, yaw, 300)
    grids, scores, st = gpu.replay_frontier(p, x, y, yaw, r, q)
    assert np.array_equal(grids, g0.cpu().numpy()) and st == st0
    assert np.array_equal(scores, oracle_scores_at_frames(oracle, p, x, y, yaw, r, q))


def test_dropin_route_agrees(gpu, oracle, pkg, synth, dev):
    """frontier_score_dir between map_update_from_beams calls (one flight, one process-wide grid, no recentering)
    gives what the batch call gives for the same instants."""
    w, d, x, y = wandering_log(synth, n=900, speed=0.0)
    p = w.params()
    yaw, r = d["yaw_deg"][0], d["ranges"][0]
    di = gpu.DropIn(p)
    di.hover_init(float(x[0]), float(y[0]))
    q = p.copy()
    q.origin_x, q.origin_y = x[0], y[0]
    inst = []
    for i in range(900):
        di.set_beams(r[i])
        di.map_update_from_beams(x[i], y[i], yaw[i])
        if i % 150 == 149:
            for off in (-90.0, 0.0, 90.0):
                inst.append((i, off, di.frontier_score_dir(x[i], y[i], yaw[i], off)))
    qs = pkg.make_queries(0, [i for i, _, _ in inst], [x[i] for i, _, _ in inst], [y[i] for i, _, _ in inst],
                          [yaw[i] for i, _, _ in inst], [o for _, o, _ in inst])
    grids, scores, _ = gpu.replay_frontier(q, x[None], y[None], yaw[None], r[None], qs)
    assert np.array_equal(grids[0], di.grid())
    assert scores.tolist() == [s for _, _, s in inst]


_FULL = {}          # the full-size inputs, inherited by the forked oracle workers


def _oracle_chunk(k):
    from oracle import orc
    p, x, y, yaw, r, qs, bounds = (_FULL[n] for n in ("p", "x", "y", "yaw", "r", "qs", "bounds"))
    f0 = 64 * k
    sub = qs[bounds[k]:bounds[k + 1]].copy()
    sub["flight"] -= f0
    return oracle_scores_at_frames(orc.Oracle(), p, x[f0:f0 + 64], y[f0:f0 + 64], yaw[f0:f0 + 64], r[f0:f0 + 64], sub)


def test_full_size_drift_ensemble_100_queries_per_flight(gpu, oracle, pkg, synth, dev):
    """All 4096 flights of config 3, 100 queries each at random frames; every score equals the oracle's (forked over
    the host's cores)."""
    w = synth.CONFIGS["c3"]
    d = synth.generate(w)
    p = w.params()
    x, y, yaw, r = d["x_true"], d["y_true"], d["frame_yaw_deg"], d["ranges"]
    F, N = x.shape
    rng = np.random.default_rng(3)
    fl = np.repeat(np.arange(F, dtype=np.int32), 100)
    fr = rng.integers(0, N, fl.size).astype(np.int32)
    q = pkg.make_queries(fl, fr, x[fl, fr], y[fl, fr], yaw[fl, fr], rng.choice([-90.0, 0.0, 90.0], fl.size))
    q = q[rng.permutation(q.size)]
    g0, g1, st0, st1, scores = both(gpu, p, x, y, yaw, r, q)
    assert np.array_equal(g0, g1) and st0 == st1
    del g0, g1
    order = np.argsort(q["flight"], kind="stable")
    qs = q[order]
    bounds = np.searchsorted(qs["flight"], np.arange(0, F + 1, 64))
    _FULL.update(p=p, x=x, y=y, yaw=yaw, r=r, qs=qs, bounds=bounds)
    try:
        with mp.get_context("fork").Pool(os.cpu_count()) as pool:
            want_sorted = np.concatenate(pool.map(_oracle_chunk, range(len(bounds) - 1)))
    finally:
        _FULL.clear()
    want = np.empty_like(want_sorted)
    want[order] = want_sorted
    bad = np.flatnonzero(scores != want)
    assert bad.size == 0, f"{bad.size} of {q.size} scores differ; first query {q[bad[0]]}"


def test_under_the_bounds_checked_build(pkg):
    """The probe reads of shared memory are checked against the same regions as the updates (-DUQS_DEBUG_BOUNDS)."""
    dbg = os.path.join(ROOT, "micro-quad-slam_b200", "libuqs_mapping_dbg.so")
    assert os.path.exists(dbg)
    env = dict(os.environ, UQS_LIBRARY=dbg)
    res = subprocess.run([sys.executable, "-m", "pytest", os.path.abspath(__file__), "-q", "-x", "-m", "gpu", "-k",
                          "not full_size and not bounds_checked", "-p", "no:cacheprovider"], capture_output=True, text=True,
                         env=env, timeout=1500, cwd=ROOT)
    tail = res.stdout[-3000:] + res.stderr[-2000:]
    assert res.returncode == 0 and "UQS_DEBUG_BOUNDS" not in res.stdout + res.stderr, tail
    assert " passed" in res.stdout and "failed" not in res.stdout, tail
