"""Frontier queries at their frame (uqs_replay_frontier) on the CPU: the oracle's statement of "the score against the
map as it stood after frame f" pinned to the reference's own code, the uqs_query layout, and the no-device errors."""
import ctypes
import os
import subprocess

import numpy as np
import pytest

from conftest import have_ref

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def oracle_scores_at_frames(oracle, p, x, y, yaw, ranges, queries, start=None):
    """Scores of ``queries`` (QUERY_DTYPE) in input order: each flight replayed by the oracle segment by segment up to
    every distinct query frame, frontier_score_dir on the grid as it stands then.  ``start``: [F,H,W] start grids."""
    scores = np.zeros(queries.size, np.int32)
    for f in np.unique(queries["flight"]):
        grid = np.zeros((p.H, p.W), np.int8) if start is None else np.array(start[f], np.int8)
        mine = np.flatnonzero(queries["flight"] == f)
        mine = mine[np.argsort(queries["frame"][mine], kind="stable")]
        done = 0
        for i in mine:
            q = queries[i]
            upto = int(q["frame"]) + 1
            if upto > done:
                oracle.replay(p, x[f, done:upto], y[f, done:upto], yaw[f, done:upto], ranges[f, done:upto], grid=grid)
                done = upto
            scores[i] = oracle.frontier_score(p, grid, q["x"], q["y"], q["yaw_deg"], q["offset_deg"])
    return scores


def hostile_queries(rng, pkg, p, x, y, yaw, n):
    """Queries at random frames from each flight's own poses and from hostile ones: off the grid, on its edge, NaN and
    huge yaw, far from the trajectory; duplicates and a pile-up at one frame; shuffled."""
    F, N = x.shape
    fl = rng.integers(0, F, n)
    fr = rng.integers(0, N, n)
    qx, qy, qyaw = x[fl, fr].copy(), y[fl, fr].copy(), yaw[fl, fr].copy()
    off = rng.choice(np.array([-90.0, 0.0, 90.0], np.float32), n)
    edge = np.float32((p.W // 2 - 1) * np.float32(p.res_m))                          # last column
    k = n // 8
    qx[:k] = np.float32(1e6)                                                       # off the grid
    qx[k:2 * k] = edge + p.origin_x                                                # on the grid's edge
    qyaw[2 * k:2 * k + k // 2] = np.float32("nan")
    qyaw[2 * k + k // 2:3 * k] = np.float32(1e30)
    qx[3 * k:4 * k] = rng.uniform(-0.45, 0.45, k).astype(np.float32) * np.float32(p.W * p.res_m)   # anywhere on the grid
    qy[3 * k:4 * k] = rng.uniform(-0.45, 0.45, k).astype(np.float32) * np.float32(p.H * p.res_m)
    fr[4 * k:4 * k + k // 2] = fr[4 * k]                                           # many at one frame
    fl[4 * k:4 * k + k // 2] = fl[4 * k]
    fr[0], fr[1], fr[2], fr[3] = 0, N - 1, 0, N - 1
    q = pkg.make_queries(fl, fr, qx, qy, qyaw, off)
    q = np.concatenate([q, q[: n // 10]])                                          # duplicates
    return q[rng.permutation(q.size)]


def test_oracle_statement_equals_reference(orc_mod, oracle, pkg, synth):
    if not have_ref(orc_mod, 400, 400, "0.05"):
        pytest.skip("oracle/_ref not built (needs /root/reference)")
    ref = orc_mod.Reference(400, 400, "0.05")
    w = synth.scaled(synth.CONFIGS["c1"], n_flights=2, n_samples=700)
    d = synth.generate(w)
    p = w.params()
    x, y, yaw, r = d["x_true"], d["y_true"], d["frame_yaw_deg"], d["ranges"]
    rng = np.random.default_rng(31)
    q = hostile_queries(rng, pkg, p, x, y, yaw, 160)
    start = rng.integers(-20, 20, (2, p.H, p.W)).astype(np.int8)
    for st in (None, start):
        got = oracle_scores_at_frames(oracle, p, x, y, yaw, r, q, st)
        for f in range(2):
            ref.reset(0.0, 0.0)
            if st is not None:
                ref.set_grid(st[f])
            mine = sorted(np.flatnonzero(q["flight"] == f), key=lambda i: int(q["frame"][i]))
            done = 0
            for i in mine:
                while done <= q["frame"][i]:
                    ref.frame(x[f, done], y[f, done], yaw[f, done], r[f, done])
                    done += 1
                assert got[i] == ref.frontier_score(q["x"][i], q["y"][i], q["yaw_deg"][i], q["offset_deg"][i]), i
    assert len(set(got.tolist())) > 10


def test_query_struct_layout_matches_header(pkg, tmp_path):
    src = ('#include <stdio.h>\n#include <stddef.h>\n#include "uqs_mapping.h"\nint main(void){printf("%zu %zu %zu %zu %zu %zu %zu",'
           ' sizeof(uqs_query), offsetof(uqs_query,flight), offsetof(uqs_query,frame), offsetof(uqs_query,x),'
           ' offsetof(uqs_query,y), offsetof(uqs_query,yaw_deg), offsetof(uqs_query,offset_deg));return 0;}\n')
    exe = str(tmp_path / "uqs_query_layout")
    r = subprocess.run(["gcc", "-std=c99", "-I", os.path.join(ROOT, "include"), "-x", "c", "-", "-o", exe], input=src, text=True,
                       capture_output=True)
    assert r.returncode == 0, r.stderr
    out = [int(v) for v in subprocess.check_output([exe], text=True).split()]
    D = pkg.QUERY_DTYPE
    assert out == [24, 0, 4, 8, 12, 16, 20] == [D.itemsize] + [D.fields[n][1] for n in D.names]


def test_make_queries(pkg):
    q = pkg.make_queries([0, 1], 5, [1.5, 2.5], 0.0, 90.0, [-90.0, 90.0])
    assert q.dtype == pkg.QUERY_DTYPE and q.size == 2
    assert q["frame"].tolist() == [5, 5] and q["x"].tolist() == [1.5, 2.5] and q["offset_deg"].tolist() == [-90.0, 90.0]


def test_entry_points_fail_without_a_device(pkg):
    import torch
    if torch.cuda.is_available():
        pytest.skip("a GPU is present")
    with pytest.raises(pkg.UqsError):
        pkg.init(0)
    p = pkg.make_params(400, 400, 0.05)
    z = np.zeros((1, 4), np.float32)
    q = pkg.make_queries(0, 0, 0.0, 0.0, 0.0, 0.0)
    with pytest.raises(pkg.UqsError) as e:
        pkg.replay_frontier(p, z, z, z, np.zeros((1, 4, 32), np.float32), q)
    assert e.value.code == pkg.ERR_NOT_INIT
    L = pkg.lib()
    st = pkg.Stats()
    rc = L.uqs_replay_frontier_dev(ctypes.byref(p), 1, 4, None, None, None, None, None, 0, 0, None, None, ctypes.byref(st))
    assert rc == pkg.ERR_NOT_INIT
