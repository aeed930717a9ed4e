"""Generate tests/golden/full_size/digests.npz: the 64-bit digest of every grid of BASELINE configurations 2-5 at full
size, computed on the CPU with the plain-C restatement (oracle/uqs_oracle.c), from the same seeded logs and pose
sources that tests/ref_jobs.py feeds the reference's own code.  test_gpu_zz_complete.py compares the device against
these digests wherever the reference's libraries (oracle/_ref) are not built.

    python tests/golden/make_complete_digests.py        # about 17 core-minutes; one forked worker per host core

The device result of the same commit was equal to every digest when the file was written.
"""
import importlib
import multiprocessing as mp
import os
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, ROOT)
from oracle import orc  # noqa: E402

synth = importlib.import_module("micro-quad-slam_b200.synth")
OUT = os.path.join(os.path.dirname(os.path.abspath(__file__)), "full_size", "digests.npz")


def _flight_digest(o, w, fid, flow):
    d = synth.generate(w, flight_id0=fid, n_flights=1, n_threads=1)
    if flow:
        x, y = o.pose_integrate(d["t_ms"][0], d["of_rate_x"][0], d["of_rate_y"][0], d["h_m"][0], d["yaw_deg"][0], d["of_q"][0])
    else:
        x, y = d["x_true"][0], d["y_true"][0]
    g, _ = o.replay(w.params(), x, y, d["frame_yaw_deg"][0], d["ranges"][0])
    return o.grid_hash64(g)


def _worker(c, cores, flights, flow, out):
    o = orc.Oracle()
    for i in range(c, len(flights), cores):
        w, fid = flights[i]
        out[i] = _flight_digest(o, w, fid, flow)


def flights_digests(flights, flow, cores):
    ctx = mp.get_context("fork")
    out = ctx.Array("Q", len(flights), lock=False)
    procs = [ctx.Process(target=_worker, args=(c, cores, flights, flow, out)) for c in range(cores)]
    for p in procs:
        p.start()
    for p in procs:
        p.join()
    if any(p.exitcode != 0 for p in procs):
        raise RuntimeError("worker failed")
    return np.frombuffer(out, dtype=np.uint64).copy()


def single_log(name):
    """Config 2 (P0 + mapping) or config 4 (true poses, two frames per sample): (digest, frames)."""
    o = orc.Oracle()
    w = synth.CONFIGS[name]
    d = synth.generate(w)
    if name == "c2":
        x, y = o.pose_integrate(d["t_ms"][0], d["of_rate_x"][0], d["of_rate_y"][0], d["h_m"][0], d["yaw_deg"][0], d["of_q"][0])
    else:
        xs, ys = synth.frame_poses(d, d["x_true"], d["y_true"])
        x, y = xs[0], ys[0]
    g, _ = o.replay(w.params(), x, y, d["frame_yaw_deg"][0], d["ranges"][0])
    return o.grid_hash64(g), int(np.asarray(x).size)


def _single_worker(name, out):
    out[0], out[1] = single_log(name)


def main():
    orc.build()
    cores = os.cpu_count() or 1
    t0 = time.perf_counter()
    # the two long single logs run beside the many-flight jobs
    ctx = mp.get_context("fork")
    single = {k: ctx.Array("Q", 2, lock=False) for k in ("c2", "c4")}
    procs = [ctx.Process(target=_single_worker, args=(k, a)) for k, a in single.items()]
    for p in procs:
        p.start()
    w3 = synth.CONFIGS["c3"]
    c3 = flights_digests([(synth.scaled(w3, n_flights=1), f) for f in range(w3.n_flights)], True, cores)
    print(f"c3: {c3.size} flights, {time.perf_counter() - t0:.0f} s", flush=True)
    c5 = np.empty((len(synth.C5_RES), 1024), np.uint64)
    for ir in range(len(synth.C5_RES)):
        ws = [synth.c5_workload(ir, isg) for isg in range(16)]
        c5[ir] = flights_digests([(synth.scaled(ws[i // 64], n_flights=1), i % 64) for i in range(1024)], False, cores)
    print(f"c5: {c5.size} flights, {time.perf_counter() - t0:.0f} s", flush=True)
    for p in procs:
        p.join()
    if any(p.exitcode != 0 for p in procs):
        raise RuntimeError("single-log worker failed")
    np.savez_compressed(OUT, c3=c3, c5=c5, c2=np.uint64(single["c2"][0]), c2_frames=np.int64(single["c2"][1]),
                        c4=np.uint64(single["c4"][0]), c4_frames=np.int64(single["c4"][1]))
    print(f"wrote {OUT} in {time.perf_counter() - t0:.0f} s: c2 {single['c2'][0]:016x}, c4 {single['c4'][0]:016x}")


if __name__ == "__main__":
    main()
