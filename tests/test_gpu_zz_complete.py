"""COMPLETE parity at full BASELINE size: every flight of configs 3 and 5 and the whole logs of configs 2 and 4,
device result against the reference's own code (oracle/_ref), compared through 64-bit digests per grid (the
digest function itself is pinned against numpy below and against the oracle's restatement of it).  Where oracle/_ref is
not built, the device is compared with the digests stored in tests/golden/full_size/digests.npz, which the CPU
restatement computed from the same logs (tests/golden/make_complete_digests.py).

The reference needs ~5 s (C3) and ~25 s (C5) on 16 cores, ~15 s (C2) and ~80 s (C4) on one: the two single-log
jobs are started in the background by conftest.py when the session begins and are collected here, in the file
pytest runs last."""
import importlib
import json
import os
import sys
import time

import numpy as np
import pytest
import torch

sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))
import ref_jobs  # noqa: E402

from conftest import background_reference_job, have_ref  # noqa: E402

pytestmark = pytest.mark.gpu
GOLDEN = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "full_size", "digests.npz")


def _golden(key):
    with np.load(GOLDEN) as z:
        return z[key]


@pytest.fixture()
def dev(gpu):
    gpu.set_stream(torch.cuda.current_stream().cuda_stream)
    yield torch.device("cuda:0")
    gpu.set_stream(None)
    gpu.set_engine(0, 0)
    gpu.set_tuning(0, 0, 0)


def _numpy_digest(g):
    m = np.uint64
    with np.errstate(over="ignore"):
        z = ((np.arange(g.size, dtype=m) << m(8)) | g.reshape(-1).view(np.uint8).astype(m)) + m(0x9E3779B97F4A7C15)
        z = (z ^ (z >> m(30))) * m(0xBF58476D1CE4E5B9)
        z = (z ^ (z >> m(27))) * m(0x94D049BB133111EB)
        return int((z ^ (z >> m(31))).sum(dtype=m))


def test_digest_function_device_host_oracle_numpy(gpu, oracle, dev):
    rng = np.random.default_rng(11)
    g = rng.integers(-128, 128, (5, 333, 417), dtype=np.int8)
    g[1] = 0
    t = torch.from_numpy(g).to(dev)
    got = gpu.grid_hashes_dev(t.data_ptr(), 5, 333 * 417)
    for i in range(5):
        want = _numpy_digest(g[i])
        assert int(got[i]) == want == gpu.grid_hash(g[i]) == oracle.grid_hash64(g[i])
    g2 = g[0].copy()
    g2[100, 100] ^= 1
    assert gpu.grid_hash(g2) != gpu.grid_hash(g[0])
    g3 = g[0].copy()
    g3[5, 5], g3[5, 6] = g[0][5, 6], g[0][5, 5]                  # position-sensitive
    assert g[0][5, 5] == g[0][5, 6] or gpu.grid_hash(g3) != gpu.grid_hash(g[0])


def _mismatch(kind, idx, got, want):
    bad = np.flatnonzero(got != want)
    return f"{kind}: {bad.size} of {want.size} grids differ from the expected ones; first: {idx(int(bad[0])) if bad.size else None}"


def test_c3_every_one_of_the_4096_flights(gpu, orc_mod, synth, dev):
    w = synth.CONFIGS["c3"]
    d = synth.generate(w)
    p = w.params()
    F, N = w.n_flights, w.n_frames
    args = [torch.from_numpy(d[k].view(np.int32) if k == "t_ms" else d[k]).to(dev) for k in ("t_ms", "of_rate_x", "of_rate_y", "h_m", "yaw_deg", "of_q")]
    tx = torch.empty((F, N), dtype=torch.float32, device=dev)
    ty = torch.empty_like(tx)
    tr = torch.from_numpy(d["ranges"]).to(dev)
    g = torch.empty((F, p.H, p.W), dtype=torch.int8, device=dev)
    gpu.pose_integrate_dev(F, N, *(a.data_ptr() for a in args), tx.data_ptr(), ty.data_ptr(), 0)
    st = gpu.replay_dev(p, F, N, tx.data_ptr(), ty.data_ptr(), args[4].data_ptr(), tr.data_ptr(), g.data_ptr(), want_stats=True)
    got = gpu.grid_hashes_dev(g.data_ptr(), F, p.W * p.H)
    if have_ref(orc_mod, w.W, w.W, w.res):
        t0 = time.perf_counter()
        want = ref_jobs.flights_digests([(synth.scaled(w, n_flights=1), f) for f in range(F)], w.W, w.res, flow=True)
        print(f"reference code: {F} flights (P0 statement + mapping) in {time.perf_counter() - t0:.1f} s on {os.cpu_count()} cores")
    else:
        want = _golden("c3")
    assert np.array_equal(got, want), _mismatch("config 3", lambda i: f"flight {i}", got, want)
    assert st["frames"] == F * N and st["domain_errors"] == 0


def test_c5_every_one_of_the_16384_flights(gpu, orc_mod, synth, dev):
    """256 configs x 64 flights; the 16 noise levels of a resolution share the geometry (one device call, one
    reference build)."""
    t_ref = 0.0
    total = 0
    golden = _golden("c5")
    for ir, res in enumerate(synth.C5_RES):
        W = synth.c5_width(res)
        ws = [synth.c5_workload(ir, isg) for isg in range(16)]
        ds = [synth.generate(w) for w in ws]
        p = ws[0].params()
        F, N = 16 * 64, ws[0].n_frames
        cat = lambda k: np.ascontiguousarray(np.concatenate([q[k] for q in ds], axis=0))
        t = [torch.from_numpy(cat(k)).to(dev) for k in ("x_true", "y_true", "frame_yaw_deg", "ranges")]
        g = torch.empty((F, p.H, p.W), dtype=torch.int8, device=dev)
        gpu.replay_dev(p, F, N, *(a.data_ptr() for a in t), g.data_ptr())
        got = gpu.grid_hashes_dev(g.data_ptr(), F, p.W * p.H)
        if have_ref(orc_mod, W, W, res):
            t0 = time.perf_counter()
            want = ref_jobs.flights_digests([(synth.scaled(ws[i // 64], n_flights=1), i % 64) for i in range(F)], W, res, flow=False)
            t_ref += time.perf_counter() - t0
        else:
            want = golden[ir]
        assert np.array_equal(got, want), _mismatch(f"config 5, {W}x{W} @ {res} m", lambda i: f"noise level {i // 64}, flight {i % 64}", got, want)
        total += F
        del t, g
    print(f"reference code: {total} flights in {t_ref:.1f} s on {os.cpu_count()} cores")
    assert total == 16384


def _collect(name):
    """The reference's digest of one long log, or the stored one where the background job was not started."""
    job = background_reference_job(name)
    if job is None:
        return {"digest": int(_golden(name)), "frames": int(_golden(name + "_frames")), "seconds": None}
    proc, path = job
    proc.wait(timeout=900)
    assert proc.returncode == 0, f"reference job {name} failed"
    with open(path) as f:
        return json.load(f)


def test_c2_the_whole_one_hour_log(gpu, synth, dev):
    ref = _collect("c2")
    w = synth.CONFIGS["c2"]
    d = synth.generate(w)
    p = w.params()
    grids, px, py, st = gpu.replay_flow(p, d["t_ms"], d["of_rate_x"], d["of_rate_y"], d["h_m"], d["yaw_deg"], d["of_q"], d["ranges"])
    if ref["seconds"] is not None:
        print(f"reference code: {ref['frames']} frames in {ref['seconds']:.1f} s on one core")
    assert gpu.grid_hash(grids[0]) == ref["digest"], "config 2: the device grid's digest differs from the expected one"
    assert st["frames"] == w.n_frames == ref["frames"]


@pytest.mark.slow
def test_c4_the_whole_building_sweep(gpu, synth, dev):
    w = synth.CONFIGS["c4"]
    d = synth.generate(w)
    p = w.params()
    x, y = synth.frame_poses(d, d["x_true"], d["y_true"])
    t = [torch.from_numpy(np.ascontiguousarray(a)).to(dev) for a in (x, y, d["frame_yaw_deg"], d["ranges"])]
    g = torch.empty((1, p.H, p.W), dtype=torch.int8, device=dev)
    st = gpu.replay_dev(p, 1, w.n_frames, *(a.data_ptr() for a in t), g.data_ptr(), want_stats=True)
    got = int(gpu.grid_hashes_dev(g.data_ptr(), 1, p.W * p.H)[0])
    # the banded form (what every rank of a multi-GPU run executes for its band) on the same device
    g2 = torch.full_like(g, 3)
    gpu.replay_banded_dev(p, w.n_frames, *(a.data_ptr() for a in t), g2.data_ptr(), gather=True)
    torch.cuda.synchronize()
    assert torch.equal(g, g2)
    ref = _collect("c4")
    if ref["seconds"] is not None:
        print(f"reference code: {ref['frames']} frames in {ref['seconds']:.1f} s on one core")
    assert got == ref["digest"], "config 4: the device grid's digest differs from the expected one"
    assert st["frames"] == ref["frames"] == 2 * 1048576
