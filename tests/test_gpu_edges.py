"""Edges of the replay that the plainer tests do not reach, each against the CPU oracle byte for byte:

* frontier queries (uqs_replay_frontier_dev) on random geometries, cell sizes and log-odds constants, on the
  automatic routes to the unrestricted kernel, with time slices over several flights and with the resident-engine
  knobs left on;
* calls of more than 65535 flights, which replay_device cuts into internal chunks (grids, stats, engine choice and
  frontier probes per chunk);
* the resident engine's measurement knobs (uqs_set_k0_bias, uqs_set_resident_pitch_mod), which must not change a byte,
  and the collision bound K0 as the resident engine receives it with a bias."""
import os
import subprocess
import sys

import numpy as np
import pytest
import torch

from conftest import first_diff
from test_frontier_replay_cpu import hostile_queries, oracle_scores_at_frames
from test_gpu_frontier_replay import both
from test_gpu_parity import _walk_cells

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
LAYOUTS = {"default": (0, 0), "fan": (1, 0), "decode warp": (0, 1)}      # (fan layout, decode warp)


@pytest.fixture()
def dev(gpu):
    """The library on torch's current stream; every engine, tuning and knob back to its default afterwards."""
    gpu.set_stream(torch.cuda.current_stream().cuda_stream)
    try:
        yield torch.device("cuda:0")
    finally:
        gpu.set_stream(None)
        gpu.set_engine(0, 0)
        gpu.set_tuning(0, 0, 0)
        gpu.set_fan_layout(-1)
        gpu.set_decode_warp(-1)
        gpu.set_k0_bias(0)
        gpu.set_resident_pitch_mod(-1)


def frontier_samples(res):
    """Samples per frontier ray: d = 2 res, 4 res, ... <= 2.5 m accumulated in binary32, as the reference's loop."""
    step = np.float32(np.float32(res) * np.float32(2.0))
    n, d = 0, step
    while d <= np.float32(2.5):
        n += 1
        d = np.float32(d + step)
    return n


def check_all(gpu, p, x, y, yaw, r, q, want, U, want_scores, start=None, what=None):
    """uqs_replay_dev and uqs_replay_frontier_dev of the same call: both grids equal the oracle's, the stats agree with
    each other and with the oracle's update count, every score equals the oracle's."""
    g0, g1, st0, st1, scores = both(gpu, p, x, y, yaw, r, q, start)
    assert np.array_equal(g0, want), (what, "replay_dev", first_diff(g0, want))
    assert np.array_equal(g1, want), (what, "replay_frontier_dev", first_diff(g1, want))
    assert st0 == st1 and st0["ray_cell_updates"] == U, (what, st0, st1, U)
    bad = np.flatnonzero(scores != want_scores)
    assert bad.size == 0, (what, f"{bad.size} of {q.size} scores differ; first query {q[bad[0]]}: got {scores[bad[0]]} "
                                 f"want {want_scores[bad[0]]}")
    return scores


def oracle_with_start(oracle, p, x, y, yaw, r, start=None):
    """(grids, updates) of the oracle, each flight from its start grid (zero when ``start`` is None)."""
    if start is None:
        return oracle.replay_flights(p, x, y, yaw, r)
    grids = np.array(start, np.int8)
    U = 0
    for f in range(x.shape[0]):
        U += oracle.replay(p, x[f], y[f], yaw[f], r[f], grids[f])[1]
    return grids, U


# ----------------------------------------------------------------------------------------------
# A. frontier queries on random geometries and sensor constants
# ----------------------------------------------------------------------------------------------
RES = (0.02, 0.05, 0.1, 0.25, 0.7, 1.25, 1.3)           # 1.25: one sample per ray (d = 2.5); 1.3: none (s_max = 0)
N_SEEDS = 28


def random_log(gpu, seed):
    rng = np.random.default_rng(7000 + seed)
    W = int(rng.choice([62, 90, 101, 128, 250, 333, 400]))
    H = int(rng.choice([58, 96, 127, 200, 260, 400]))
    res = RES[seed % len(RES)]
    p = gpu.make_params(W, H, res, W * res)
    p.fov_deg = np.float32(rng.choice([2.0, 10.0, 63.0, 90.0, 120.0, 170.0]))
    p.max_range_m = np.float32(rng.choice([1.0, 4.0, 6.0]))
    p.origin_x, p.origin_y = np.float32(rng.uniform(-1, 1)), np.float32(rng.uniform(-1, 1))
    p.lo_free, p.lo_occ = int(rng.choice([1, 2, 5])), int(rng.choice([3, 6, 20]))
    # lo_max = 7: no cell can score "occupied" (> 10); lo_min = -5: none can score "free" (< -10)
    p.lo_min, p.lo_max = int(rng.choice([-80, -128, -5])), int(rng.choice([80, 127, 7]))
    F, N = int(rng.choice([1, 2, 5])), int(rng.choice([40, 333, 700]))
    half_x, half_y = 0.5 * W * res, 0.5 * H * res
    mode = rng.integers(3)
    if mode == 0:      # hover
        x = (p.origin_x + 0.01 * rng.standard_normal((F, N))).astype(np.float32)
        y = (p.origin_y + 0.01 * rng.standard_normal((F, N))).astype(np.float32)
    elif mode == 1:    # jumps all over (and beyond) the map
        x = rng.uniform(-1.2 * half_x, 1.2 * half_x, (F, N)).astype(np.float32)
        y = rng.uniform(-1.2 * half_y, 1.2 * half_y, (F, N)).astype(np.float32)
    else:              # smooth drift
        t = np.linspace(0, 1, N, dtype=np.float32)
        x = (np.float32(0.7 * half_x) * np.cos(6 * t) + np.zeros((F, 1), np.float32)).astype(np.float32)
        y = (np.float32(0.7 * half_y) * np.sin(4 * t) + np.zeros((F, 1), np.float32)).astype(np.float32)
    yaw = rng.uniform(-360, 360, (F, N)).astype(np.float32)
    r = rng.uniform(0.0, float(p.max_range_m) * 1.1, (F, N, 32)).astype(np.float32)
    r[rng.random(r.shape) < 0.1] = np.nan
    r[rng.random(r.shape) < 0.1] = np.float32(rng.uniform(0.04, 3 * res))       # very short rays
    return rng, p, x, y, yaw, r


def test_random_seeds_cover_every_frontier_route(gpu):
    """The seeds below reach a sampling ray of none, one and many samples, and both clamp constants that make a
    score class unreachable."""
    logs = [random_log(gpu, s)[1] for s in range(N_SEEDS)]
    s_max = [frontier_samples(p.res_m) for p in logs]
    assert s_max.count(0) >= 3 and s_max.count(1) >= 3 and sum(s > 1 for s in s_max) >= 15
    assert sum(p.lo_max == 7 for p in logs) >= 3 and sum(p.lo_min == -5 for p in logs) >= 3


@pytest.mark.parametrize("seed", range(N_SEEDS))
def test_frontier_queries_on_random_geometry_and_constants(gpu, oracle, pkg, dev, seed):
    """Every engine of the plain stress test (sub-tiles with 1 and 3 time slices, auto, resident at 4/16/32 warps,
    the unrestricted kernel), hostile queries, grids and stats equal to the oracle and to uqs_replay_dev."""
    rng, p, x, y, yaw, r = random_log(gpu, seed)
    q = hostile_queries(rng, pkg, p, x, y, yaw, 400)
    want, U = oracle.replay_flights(p, x, y, yaw, r)
    want_scores = oracle_scores_at_frames(oracle, p, x, y, yaw, r, q)
    if frontier_samples(p.res_m) == 0:
        assert not want_scores.any()
    cases = [(1, 0, 1), (1, 0, 3), (0, 0, 0), (2, 4, 0), (2, 16, 0), (2, 32, 0), (3, 0, 0)]
    for engine, nw, slices in cases:
        gpu.set_engine(engine, nw)
        gpu.set_tuning(0, 0, slices)
        what = ((engine, nw, slices), dict(W=p.W, H=p.H, res=float(p.res_m), fov=float(p.fov_deg), lo=(p.lo_min, p.lo_max)))
        check_all(gpu, p, x, y, yaw, r, q, want, U, want_scores, what=what)


def synth_log(synth, F, N, cfg="c1"):
    w = synth.scaled(synth.CONFIGS[cfg], n_flights=F, n_samples=N)
    d = synth.generate(w)
    return w.params(), d["x_true"], d["y_true"], d["frame_yaw_deg"], np.ascontiguousarray(d["ranges"])


@pytest.mark.parametrize("lo", [(5, 60), (-60, -3)])
@pytest.mark.parametrize("engine", [0, 2])
def test_frontier_queries_with_a_clamp_range_excluding_zero(gpu, oracle, pkg, synth, dev, engine, lo):
    """A clamp range without 0 sends engines 0 and 2 to the unrestricted kernel by themselves (probes included)."""
    p, x, y, yaw, r = synth_log(synth, 3, 500)
    p.lo_min, p.lo_max = lo
    q = hostile_queries(np.random.default_rng([engine, lo[0] + 128]), pkg, p, x, y, yaw, 600)
    want, U = oracle.replay_flights(p, x, y, yaw, r)
    want_scores = oracle_scores_at_frames(oracle, p, x, y, yaw, r, q)
    gpu.set_engine(engine, 0)
    check_all(gpu, p, x, y, yaw, r, q, want, U, want_scores)
    start = np.random.default_rng(3).integers(-100, 100, (3, p.H, p.W)).astype(np.int8)
    want, U = oracle_with_start(oracle, p, x, y, yaw, r, start)
    check_all(gpu, p, x, y, yaw, r, q, want, U, oracle_scores_at_frames(oracle, p, x, y, yaw, r, q, start), start)


@pytest.mark.parametrize("engine", [0, 2])
def test_frontier_queries_with_rays_longer_than_1024_cells(gpu, oracle, pkg, dev, engine):
    """1400 x 1200 cells of 3 mm with a 4 m range: rays of up to ~1400 cells, the unrestricted kernel by itself."""
    p = gpu.make_params(1400, 1200, 0.003)
    rng = np.random.default_rng(11)
    F, N = 2, 150
    x = rng.uniform(-1.5, 1.5, (F, N)).astype(np.float32)
    y = rng.uniform(-1.2, 1.2, (F, N)).astype(np.float32)
    yaw = rng.uniform(-180, 180, (F, N)).astype(np.float32)
    r = rng.uniform(0.05, 4.4, (F, N, 32)).astype(np.float32)
    r[rng.random(r.shape) < 0.1] = np.nan
    q = hostile_queries(rng, pkg, p, x, y, yaw, 300)
    want, U = oracle.replay_flights(p, x, y, yaw, r)
    cells, origin = oracle.beam_cells(p, x, y, yaw, r)
    ok = cells[..., 0] >= 0
    longest = np.abs(cells - origin[:, None, :]).max(axis=2)[ok].max()
    assert longest > 1024, longest
    gpu.set_engine(engine, 0)
    scores = check_all(gpu, p, x, y, yaw, r, q, want, U, oracle_scores_at_frames(oracle, p, x, y, yaw, r, q))
    assert len(set(scores.tolist())) > 20


@pytest.mark.parametrize("S", [2, 5])
def test_frontier_queries_on_time_slices_of_several_flights(gpu, oracle, pkg, synth, dev, S):
    """Sub-tile engine with S forced time slices over 3 flights: queries on the first and last frame of every slice
    of every flight, so that the slice composition of probes reads maps at flight indices 1 and 2."""
    p, x, y, yaw, r = synth_log(synth, 3, 2000)
    F, N = x.shape
    gps = ((N + 31) // 32 + S - 1) // S
    edges = sorted({e for s in range(S) for e in (s * gps * 32, min((s + 1) * gps * 32, N) - 1) if e < N})
    rng = np.random.default_rng(S)
    fl = np.repeat(np.arange(F), len(edges) + 200)
    fr = np.concatenate([np.concatenate([edges, rng.integers(0, N, 200)]) for _ in range(F)]).astype(np.int32)
    q = pkg.make_queries(fl, fr, x[fl, fr], y[fl, fr], yaw[fl, fr], rng.choice([-90.0, 0.0, 90.0], fl.size))
    q = q[rng.permutation(q.size)]
    want, U = oracle.replay_flights(p, x, y, yaw, r)
    gpu.set_engine(1, 0)
    gpu.set_tuning(0, 0, S)
    scores = check_all(gpu, p, x, y, yaw, r, q, want, U, oracle_scores_at_frames(oracle, p, x, y, yaw, r, q))
    assert len(set(scores.tolist())) > 20


@pytest.mark.parametrize("engine,warps", [(0, 0), (2, 4), (2, 8), (2, 32)])
def test_frontier_queries_ignore_the_resident_layout_knobs(gpu, oracle, pkg, synth, dev, engine, warps):
    """uqs_set_fan_layout(1) and uqs_set_decode_warp(1) left on during query calls: the same grids and scores."""
    p, x, y, yaw, r = synth_log(synth, 6, 600, "c3")
    q = hostile_queries(np.random.default_rng(warps), pkg, p, x, y, yaw, 900)
    want, U = oracle.replay_flights(p, x, y, yaw, r)
    want_scores = oracle_scores_at_frames(oracle, p, x, y, yaw, r, q)
    gpu.set_engine(engine, warps)
    for fan, dec in ((1, 0), (0, 1), (1, 1)):
        gpu.set_fan_layout(fan)
        gpu.set_decode_warp(dec)
        check_all(gpu, p, x, y, yaw, r, q, want, U, want_scores, what=(fan, dec))


# ----------------------------------------------------------------------------------------------
# B. more than 65535 flights in one call (internal chunks of at most 65535: gridDim.y of the ray set-up)
# ----------------------------------------------------------------------------------------------
def many_flights_log(T, N=40):
    """65535 + T flights of N frames on a 48 x 48 grid of 10 cm cells with a 1 m range, seeded poses and ranges."""
    F = 65535 + T
    rng = np.random.default_rng(65535 + T)
    p_args = (48, 48, 0.1)
    x = (rng.uniform(-1.5, 1.5, (F, 1)) + np.cumsum(rng.normal(0, 0.05, (F, N)), axis=1)).astype(np.float32)
    y = (rng.uniform(-1.5, 1.5, (F, 1)) + np.cumsum(rng.normal(0, 0.05, (F, N)), axis=1)).astype(np.float32)
    yaw = rng.uniform(-180, 180, (F, N)).astype(np.float32)
    r = rng.uniform(0.03, 1.1, (F, N, 32)).astype(np.float32)
    r[rng.random(r.shape) < 0.1] = np.nan
    return p_args, x, y, yaw, r


@pytest.mark.parametrize("tail", ["resident", "sub-tiles"])
def test_many_flights_across_internal_chunks(gpu, oracle, pkg, dev, tail):
    """65535 + T flights: T = ceil(SMs/4) leaves the last chunk resident under engine 0, one fewer sends it to the
    sub-tile engine inside the same call.  Engines 0, 1 and 3, fresh and onto seeded start grids, each with frontier
    queries on flights 0, 65534, 65535, 65536 and the last one at frames 0, 31, 32 and the last, plus random ones;
    once more on engine 1 with two time slices (probes of the second chunk in slice maps).  Grids and stats equal the
    oracle's.  Peak memory, measured on a B200: 2.3 GB of host memory (the test process) and 2.8 GB of device memory;
    about 15 s per case."""
    T = -(-gpu.sm_count() // 4) - (tail == "sub-tiles")
    (W, H, res), x, y, yaw, r = many_flights_log(T)
    p = gpu.make_params(W, H, res)
    p.max_range_m = 1.0
    F, N = x.shape
    rng = np.random.default_rng(T)
    fl = np.repeat(np.array([0, 65534, 65535, 65536, F - 1]), 12)
    fr = np.tile(np.repeat(np.array([0, 31, 32, N - 1]), 3), 5)
    off = np.tile(np.array([-90.0, 0.0, 90.0]), 20)
    fl = np.concatenate([fl, rng.integers(0, F, 400), rng.integers(65535, F, 100)])
    fr = np.concatenate([fr, rng.integers(0, N, 500)])
    off = np.concatenate([off, rng.choice([-90.0, 0.0, 90.0], 500)])
    q = pkg.make_queries(fl, fr, x[fl, fr], y[fl, fr], yaw[fl, fr], off)
    q = q[rng.permutation(q.size)]
    start = rng.integers(-70, 70, (F, H, W)).astype(np.int8)
    for acc in (None, start):
        want, U = oracle_with_start(oracle, p, x, y, yaw, r, acc)
        want_scores = oracle_scores_at_frames(oracle, p, x, y, yaw, r, q, acc)
        for engine, slices in ((0, 0), (1, 0), (3, 0)) + (((1, 2),) if acc is None else ()):
            gpu.set_engine(engine, 0)
            gpu.set_tuning(0, 0, slices)
            check_all(gpu, p, x, y, yaw, r, q, want, U, want_scores, acc, what=(engine, slices, acc is not None))
        del want


# ----------------------------------------------------------------------------------------------
# C. the resident engine's measurement knobs, and K0 with a bias
# ----------------------------------------------------------------------------------------------
def parallel_beams_log(F=8, N=120, seed=5):
    """400 x 400 cells of 5 cm, 2-degree fans and ranges of 6 to 20 cm: the eight beams of a sensor quantise to
    directions that are often exactly parallel, and share cells up to the shorter one's end.  In every other frame all
    32 beams have one range, which keeps the quantised directions in angular order (the frames K0 is computed for from
    neighbours alone).  Half of the flights hover, the others drift a few cells per frame (so that cells stay inside
    the clamp and a lost update shows)."""
    rng = np.random.default_rng(seed)
    x = np.where(np.arange(F)[:, None] % 2 == 0, 0.01 * rng.standard_normal((F, N)),
                 np.cumsum(rng.normal(0, 0.15, (F, N)), axis=1)).astype(np.float32)
    y = np.where(np.arange(F)[:, None] % 2 == 0, 0.01 * rng.standard_normal((F, N)),
                 np.cumsum(rng.normal(0, 0.15, (F, N)), axis=1)).astype(np.float32)
    yaw = rng.uniform(-180, 180, (F, N)).astype(np.float32)
    r = rng.uniform(0.06, 0.2, (F, N, 32)).astype(np.float32)
    r[:, ::2] = r[:, ::2, :1]
    r[rng.random(r.shape) < 0.05] = np.nan
    return x, y, yaw, r


def parallel_params(gpu):
    p = gpu.make_params(400, 400, 0.05)
    p.fov_deg = 2.0
    p.lo_min, p.lo_max = -128, 127
    return p


def shared_steps(cells, origin):
    """Per frame: the last step at which two beams share a cell (brute force on the reference's walk; -1: none), the
    longest beam in steps (-1: no accepted beam), and whether the pose is on the grid."""
    n = origin.shape[0]
    last, mmax = np.full(n, -1), np.full(n, -1)
    for f in range(n):
        if origin[f, 0] < 0:
            continue
        beams = [(int(cells[f, b, 0] - origin[f, 0]), int(cells[f, b, 1] - origin[f, 1])) for b in range(32) if cells[f, b, 0] >= 0]
        walks = [_walk_cells(dx, dy) for dx, dy in beams]
        mmax[f] = max((len(w) - 1 for w in walks), default=-1)
        for i in range(len(walks)):
            for j in range(i + 1, len(walks)):
                for k in range(min(len(walks[i]), len(walks[j]))):
                    if walks[i][k] == walks[j][k]:
                        last[f] = max(last[f], k)
    return last, mmax, origin[:, 0] >= 0


@pytest.mark.parametrize("bias", [0, 1, 8])
def test_collision_bound_k0_with_a_bias_by_brute_force(gpu, dev, bias):
    """K0 as the resident engine receives it with uqs_set_k0_bias(b): still above every shared step (brute force),
    and exactly the unbiased K0 plus b, capped at the longest beam's last step + 1 -- on parallel short beams, on
    ordinary frames and on wide fans whose beams are out of angular order (the all-pairs bound)."""
    rng = np.random.default_rng(78)
    logs = [(parallel_params(gpu),) + tuple(a.reshape(-1, *a.shape[2:]) for a in parallel_beams_log(F=2, N=150))]
    for fov, rmax in ((63.0, 4.0), (170.0, 0.6)):
        p = gpu.make_params(400, 400, 0.05)
        p.fov_deg, p.max_range_m = fov, rmax
        n = 150
        r = rng.uniform(0.06, rmax * 1.1, (n, 32)).astype(np.float32)
        short = rng.random(n) < 0.4
        r[short] = rng.uniform(0.06, 0.3, (int(short.sum()), 32)).astype(np.float32)
        r[rng.random((n, 32)) < 0.1] = np.nan
        logs.append((p, rng.uniform(-2, 2, n).astype(np.float32), rng.uniform(-2, 2, n).astype(np.float32),
                     rng.uniform(-180, 180, n).astype(np.float32), r))
    parallel = unsorted = 0
    for p, x, y, yaw, r in logs:
        cells, origin = gpu.beam_cells(p, x, y, yaw, r)
        last, mmax, on = shared_steps(cells, origin)
        gpu.set_k0_bias(0)
        k0_plain, srt = gpu.frame_bounds(p, x, y, yaw, r)
        gpu.set_k0_bias(bias)
        k0, _ = gpu.frame_bounds(p, x, y, yaw, r)
        assert np.array_equal(k0[~on], np.full((~on).sum(), -1))
        bad = np.flatnonzero(on & (last >= k0))
        assert bad.size == 0, f"frame {bad[0]}: beams share a cell at step {last[bad[0]]}, K0 = {k0[bad[0]]} (bias {bias})"
        expect = np.minimum(k0_plain + bias, mmax + 1)
        bad = np.flatnonzero(on & (k0 != expect))
        assert bad.size == 0, f"frame {bad[0]}: K0 {k0[bad[0]]} with bias {bias}, {k0_plain[bad[0]]} without, longest beam {mmax[bad[0]]}"
        parallel += int((on & (last >= 1)).sum())
        unsorted += int((on & (srt == 0)).sum())
    assert parallel > 100 and unsorted > 10, (parallel, unsorted)


@pytest.mark.parametrize("layout", list(LAYOUTS))
@pytest.mark.parametrize("warps", [4, 8, 16, 32])
def test_k0_bias_gives_identical_bytes(gpu, oracle, dev, warps, layout):
    """Resident engine with K0 biased by 0..8 steps on a log whose sorted frames have exactly parallel neighbouring
    beams (checked by brute force first): grids and stats equal the oracle's for every bias."""
    p = parallel_params(gpu)
    x, y, yaw, r = parallel_beams_log()
    cells, origin = gpu.beam_cells(p, x.ravel(), y.ravel(), yaw.ravel(), r.reshape(-1, 32))
    last, _, on = shared_steps(cells, origin)
    k0, srt = gpu.frame_bounds(p, x.ravel(), y.ravel(), yaw.ravel(), r.reshape(-1, 32))
    assert not (on & (last >= k0)).any()
    assert int((on & (last >= 1) & (srt == 1)).sum()) > 100
    want, U = oracle.replay_flights(p, x, y, yaw, r)
    gpu.set_engine(2, warps)
    gpu.set_fan_layout(LAYOUTS[layout][0])
    gpu.set_decode_warp(LAYOUTS[layout][1])
    for bias in range(9):
        gpu.set_k0_bias(bias)
        got, st = gpu.replay(p, x, y, yaw, r)
        assert np.array_equal(got, want), (bias, first_diff(got, want))
        assert st["ray_cell_updates"] == U


def full_box_log():
    """Poses all over a 560 x 400 grid, corners included: the touched box of each flight is the whole grid, which
    fits the resident engine's shared memory with the built-in row pitch and not with most others.  40 flights: enough
    for engine 0 to choose the resident engine whenever the box fits."""
    p_args = (560, 400, 0.05)
    rng = np.random.default_rng(560)
    F, N = 40, 400
    x = rng.uniform(-14.0, 13.95, (F, N)).astype(np.float32)
    y = rng.uniform(-10.0, 9.95, (F, N)).astype(np.float32)
    x[:, :4] = np.array([-14.0, 13.95, -14.0, 13.95], np.float32)
    y[:, :4] = np.array([-10.0, -10.0, 9.95, 9.95], np.float32)
    yaw = rng.uniform(-180, 180, (F, N)).astype(np.float32)
    r = rng.uniform(0.1, 4.4, (F, N, 32)).astype(np.float32)
    r[:, :4] = 0.5
    r[rng.random(r.shape) < 0.1] = np.nan
    return p_args, x, y, yaw, r


@pytest.mark.parametrize("box", ["small", "whole grid"])
@pytest.mark.parametrize("layout", list(LAYOUTS))
def test_resident_pitch_mod_gives_identical_bytes(gpu, oracle, pkg, dev, layout, box):
    """Row pitch of the resident box forced to m words mod 32: the same bytes at every warp count, or -- when the
    wider pitch no longer fits shared memory -- UQS_ERR_BAD_ARG from engine 2 and the same bytes from engine 0."""
    if box == "small":
        p = parallel_params(gpu)
        x, y, yaw, r = parallel_beams_log(F=4)
    else:
        (W, H, res), x, y, yaw, r = full_box_log()
        p = gpu.make_params(W, H, res)
    want, U = oracle.replay_flights(p, x, y, yaw, r)
    gpu.set_fan_layout(LAYOUTS[layout][0])
    gpu.set_decode_warp(LAYOUTS[layout][1])
    refused = []
    for m in (-1, 0, 1, 2, 15, 16, 31):
        gpu.set_resident_pitch_mod(m)
        for warps in (4, 8, 16, 32):
            gpu.set_engine(2, warps)
            try:
                got, st = gpu.replay(p, x, y, yaw, r)
            except pkg.UqsError as e:
                assert e.code == pkg.ERR_BAD_ARG and "does not fit" in str(e), (m, warps, e.code, str(e))
                refused.append((m, warps))
                gpu.set_engine(0, warps)
                got, st = gpu.replay(p, x, y, yaw, r)
            assert np.array_equal(got, want), (m, warps, first_diff(got, want))
            assert st["ray_cell_updates"] == U
    assert not any(m == -1 for m, _ in refused), refused
    if box == "small":
        assert not refused, refused
    else:
        assert any(w == 4 for _, w in refused), refused


# ----------------------------------------------------------------------------------------------
def test_under_the_bounds_checked_build(pkg):
    """This file once more under -DUQS_DEBUG_BOUNDS (every shared-memory access of the engines checked against its
    region): the pitch and K0 variants change the resident layout and collision paths.  The >65535-flight cases are
    left out."""
    dbg = os.path.join(ROOT, "micro-quad-slam_b200", "libuqs_mapping_dbg.so")
    assert os.path.exists(dbg)
    env = dict(os.environ, UQS_LIBRARY=dbg)
    res = subprocess.run([sys.executable, "-m", "pytest", os.path.abspath(__file__), "-q", "-x", "-m", "gpu", "-k",
                          "not many_flights and not bounds_checked", "-p", "no:cacheprovider"], capture_output=True, text=True,
                         env=env, timeout=2400, cwd=ROOT)
    tail = res.stdout[-3000:] + res.stderr[-2000:]
    assert res.returncode == 0 and "UQS_DEBUG_BOUNDS" not in res.stdout + res.stderr, tail
    assert " passed" in res.stdout and "failed" not in res.stdout, tail
