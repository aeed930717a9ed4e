"""The overlapped schedule of device replays on the resident engine (uqs_set_setup_overlap): the ray set-up of each
chunk of flights runs beside the previous chunk's replay.  Only the schedule changes, so every call here must give the
grids and stats of the serial schedule (uqs_set_setup_overlap(0)) byte for byte, and the calls that cannot overlap --
a single wave of flights, a row band, a box that leaves no room beside the replay's CTAs, the sub-tile engine -- must
take the serial schedule.  The serial schedule itself is checked against the oracle by the other GPU tests."""
import numpy as np
import pytest
import torch

from conftest import first_diff
from test_gpu_edges import many_flights_log, synth_log


def test_the_library_exports_the_schedule_knob(pkg):
    L = pkg.lib()
    assert hasattr(L, "uqs_set_setup_overlap") and hasattr(L, "uqs_setup_overlap_chunks")
    assert "uqs_set_setup_overlap" in pkg.exported_symbols()


@pytest.fixture()
def dev(gpu):
    gpu.set_stream(torch.cuda.current_stream().cuda_stream)
    try:
        yield torch.device("cuda:0")
    finally:
        gpu.set_stream(None)
        gpu.set_engine(0, 0)
        gpu.set_k0_bias(0)
        gpu.set_setup_overlap(-1)
        gpu.set_host_chunk(0)


def overlapping(gpu):
    """Flights of a call that takes the overlapped schedule under engine 2 with 8 warps per CTA (4 CTAs per SM beside
    one set-up block, whatever the box): a first chunk of 4 CTAs per SM, then one chunk of 2 waves (replay_device)."""
    gpu.set_engine(2, 8)
    return gpu.sm_count() * 4 * 3


def both_schedules(gpu, p, x, y, yaw, r, start=None, row0=0, rows=None):
    """(grids, stats, chunks set up beside a replay) of the serial and then the overlapped schedule."""
    out = []
    F, N = x.shape
    d = {k: torch.as_tensor(np.ascontiguousarray(v)).cuda() for k, v in (("x", x), ("y", y), ("yaw", yaw), ("r", r))}
    for waves in (0, 2):
        gpu.set_setup_overlap(waves)
        g = torch.as_tensor(start).cuda() if start is not None else torch.full((F, p.H, p.W), 77, dtype=torch.int8, device="cuda")
        st = gpu.replay_dev(p, F, N, d["x"].data_ptr(), d["y"].data_ptr(), d["yaw"].data_ptr(), d["r"].data_ptr(), g.data_ptr(),
                            accumulate=start is not None, row0=row0, rows=rows, want_stats=True)
        torch.cuda.synchronize()
        out.append((g.cpu().numpy(), st, gpu.setup_overlap_chunks()))
    (g0, s0, c0), (g1, s1, c1) = out
    assert c0 == 0
    assert np.array_equal(g0, g1), first_diff(g0, g1)
    assert s0 == s1, (s0, s1)
    return g1, s1, c1


@pytest.mark.gpu
@pytest.mark.parametrize("extra", [0, 37, 2 * 148 * 4 + 5])
def test_flights_beyond_one_wave(gpu, synth, dev, extra):
    """Enough c3 flights for the overlapped schedule (chunks beside a replay): no byte changes; flight counts that
    are not a multiple of the later chunks' size included."""
    F = overlapping(gpu) + extra
    p, x, y, yaw, r = synth_log(synth, F, 200, "c3")
    _, st, chunks = both_schedules(gpu, p, x, y, yaw, r)
    assert chunks >= 1 and st["ray_cell_updates"] > 0


@pytest.mark.gpu
@pytest.mark.parametrize("F", [1, 100, 1024])
def test_few_flights_keep_the_serial_schedule(gpu, synth, dev, F):
    """Less than a first chunk and one later chunk of flights: serial."""
    p, x, y, yaw, r = synth_log(synth, F, 300, "c3")
    assert both_schedules(gpu, p, x, y, yaw, r)[2] == 0


@pytest.mark.gpu
@pytest.mark.parametrize("warps", [4, 8, 16])
def test_warps_per_cta(gpu, synth, dev, warps):
    """The resident engine forced to 4, 8 or 16 warps per CTA (4: the replay's CTAs leave no room for a set-up block)."""
    p, x, y, yaw, r = synth_log(synth, overlapping(gpu) + 300, 160, "c3")
    gpu.set_engine(2, warps)
    chunks = both_schedules(gpu, p, x, y, yaw, r)[2]
    assert chunks == 0 if warps == 4 else chunks >= 1


@pytest.mark.gpu
def test_accumulate_and_k0_bias(gpu, synth, dev):
    """Onto seeded start grids (accumulate = 1), and with a K0 bias of 3 steps."""
    F = overlapping(gpu) + 200
    p, x, y, yaw, r = synth_log(synth, F, 160, "c3")
    start = np.random.default_rng(5).integers(p.lo_min, p.lo_max + 1, (F, p.H, p.W)).astype(np.int8)
    assert both_schedules(gpu, p, x, y, yaw, r, start=start)[2] >= 1
    gpu.set_k0_bias(3)
    assert both_schedules(gpu, p, x, y, yaw, r)[2] >= 1


@pytest.mark.gpu
def test_row_band_keeps_the_serial_schedule(gpu, synth, dev):
    """A row band cannot be resident: the sub-tile engine, serial."""
    F = overlapping(gpu) + 50
    gpu.set_engine(0, 0)
    p, x, y, yaw, r = synth_log(synth, F, 120, "c3")
    assert both_schedules(gpu, p, x, y, yaw, r, row0=p.H // 4, rows=p.H // 2)[2] == 0


@pytest.mark.gpu
def test_sub_tile_engine_is_unaffected(gpu, synth, dev):
    F = overlapping(gpu) + 50
    gpu.set_engine(1, 0)
    p, x, y, yaw, r = synth_log(synth, F, 120, "c3")
    assert both_schedules(gpu, p, x, y, yaw, r)[2] == 0


@pytest.mark.gpu
def test_a_box_with_no_room_beside_it_takes_the_serial_schedule(gpu, dev):
    """Flights over all of a 472 x 472 grid: one resident CTA of ~229 KB per SM leaves less shared memory than a
    set-up block needs."""
    p = gpu.make_params(472, 472, 0.1)
    rng = np.random.default_rng(472)
    F, N = overlapping(gpu) + 100, 60
    x = rng.uniform(-23.0, 23.0, (F, N)).astype(np.float32)
    y = rng.uniform(-23.0, 23.0, (F, N)).astype(np.float32)
    yaw = rng.uniform(-180, 180, (F, N)).astype(np.float32)
    r = rng.uniform(0.05, 4.2, (F, N, 32)).astype(np.float32)
    gpu.set_engine(2, 16)
    assert both_schedules(gpu, p, x, y, yaw, r)[2] == 0


@pytest.mark.gpu
def test_millimetre_ranges_through_one_host_chunk(gpu, synth, dev):
    """u16 millimetre ranges (uqs_replay_flow_mm), all flights in one chunk of the host-buffer call."""
    F = overlapping(gpu) + 120
    w = synth.on_mm_lattice(synth.scaled(synth.CONFIGS["c3"], n_flights=F, n_samples=200))
    d = synth.generate(w)
    p = w.params()
    mm = synth.ranges_to_mm(d["ranges"])
    args = (d["t_ms"], d["of_rate_x"], d["of_rate_y"], d["h_m"], d["yaw_deg"], d["of_q"])
    gpu.set_host_chunk(F)
    out = []
    for waves in (0, 2):
        gpu.set_setup_overlap(waves)
        g, _, _, st = gpu.replay_flow_mm(p, *args, mm, want_poses=False)
        out.append((g, st, gpu.setup_overlap_chunks()))
    assert out[0][2] == 0 and out[1][2] >= 1
    assert np.array_equal(out[0][0], out[1][0]), first_diff(out[0][0], out[1][0])
    assert out[0][1] == out[1][1]


@pytest.mark.gpu
def test_more_than_65535_flights(gpu, dev):
    """65535 + SMs/4 flights: internal chunks of the scratch budget, each scheduled on its own."""
    T = -(-gpu.sm_count() // 4)
    (W, H, res), x, y, yaw, r = many_flights_log(T)
    p = gpu.make_params(W, H, res)
    p.max_range_m = 1.0
    gpu.set_engine(2, 8)
    assert both_schedules(gpu, p, x, y, yaw, r)[2] >= 1
