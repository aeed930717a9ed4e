"""micro-quad-slam_b200 -- Python binding of libuqs_mapping.so (the product is the C/CUDA library).

The host side of the path is plain C behind ``include/uqs_mapping.h``; this module
only loads that shared library with ctypes so that pytest and ``bench.py`` can call the
same C ABI a C harness would.  Function names and argument meaning follow the
reference's mapping symbols (``uav_local_nav.c:205-306``) and the batch entry points of
the header.  There is no Python or CPU implementation of the path in here: if the
library is missing or no CUDA device is usable, calls raise ``UqsError``.

The directory name contains hyphens, so import it with
``importlib.import_module("micro-quad-slam_b200")``.
"""
from __future__ import annotations

import ctypes as C
import os
from typing import Optional

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.environ.get("UQS_LIBRARY") or os.path.join(_HERE, "libuqs_mapping.so")   # override: kernel-variant experiments (tools/)
SYNTH_LIB_PATH = os.path.join(_HERE, "libuqs_synth.so")

BEAMS_PER_FRAME = 32

OK, ERR_NO_DEVICE, ERR_CUDA, ERR_BAD_ARG, ERR_NOT_INIT, ERR_DOMAIN, ERR_NOMEM, ERR_NO_NCCL, ERR_NCCL = range(9)
COMM_ID_BYTES = 128


class UqsError(RuntimeError):
    def __init__(self, code: int, msg: str):
        super().__init__(f"uqs error {code}: {msg}")
        self.code = code


class Params(C.Structure):
    """``uqs_params`` -- run-time form of the reference's grid/sensor constants."""

    _fields_ = [
        ("W", C.c_int32), ("H", C.c_int32),
        ("res_m", C.c_float), ("size_m", C.c_float),
        ("origin_x", C.c_float), ("origin_y", C.c_float),
        ("max_range_m", C.c_float), ("fov_deg", C.c_float),
        ("min_range_m", C.c_float), ("hit_margin_m", C.c_float),
        ("lo_free", C.c_int32), ("lo_occ", C.c_int32), ("lo_min", C.c_int32), ("lo_max", C.c_int32),
    ]

    def copy(self) -> "Params":
        q = Params()
        C.memmove(C.byref(q), C.byref(self), C.sizeof(Params))
        return q


class Stats(C.Structure):
    _fields_ = [
        ("ray_cell_updates", C.c_uint64), ("rays_accepted", C.c_uint64), ("rays_skipped", C.c_uint64),
        ("frames", C.c_uint64), ("domain_errors", C.c_uint64),
    ]

    def as_dict(self) -> dict:
        return {k: int(getattr(self, k)) for k, _ in self._fields_}


def make_params(W: int, H: int, res_m: float, size_m: Optional[float] = None, origin=(0.0, 0.0)) -> Params:
    """Reference defaults (uav_local_nav.c:117-118, 194-197) with the given geometry."""
    p = Params()
    p.W, p.H = int(W), int(H)
    p.res_m = np.float32(res_m)
    p.size_m = np.float32(size_m if size_m is not None else W * res_m)
    p.origin_x, p.origin_y = np.float32(origin[0]), np.float32(origin[1])
    p.max_range_m, p.fov_deg = 4.0, 63.0
    p.min_range_m, p.hit_margin_m = np.float32(0.05), np.float32(0.05)
    p.lo_free, p.lo_occ, p.lo_min, p.lo_max = 1, 6, -80, 80
    return p


_lib = None

_EXPORTS = [
    # batch API
    "uqs_params_default", "uqs_init", "uqs_shutdown", "uqs_last_error", "uqs_device_sm_count",
    "uqs_set_stream", "uqs_use_own_stream", "uqs_sync", "uqs_set_tuning", "uqs_set_engine", "uqs_set_fan_layout", "uqs_set_decode_warp", "uqs_set_k0_bias", "uqs_set_resident_pitch_mod", "uqs_set_setup_overlap", "uqs_setup_overlap_chunks", "uqs_kernel_launches",
    "uqs_set_profiling", "uqs_profile_collect", "uqs_profile_timeline", "uqs_set_host_chunk",
    "uqs_pose_integrate", "uqs_pose_integrate_dev", "uqs_replay", "uqs_replay_dev", "uqs_replay_flow",
    "uqs_beam_cells", "uqs_frame_bounds", "uqs_sincosf_batch", "uqs_measure_rmw_peak", "uqs_measure_atoms_peak",
    "uqs_beams_from_scans", "uqs_beams_from_scans_dev", "uqs_replay_recentering", "uqs_frontier_scores",
    "uqs_replay_frontier", "uqs_replay_frontier_dev", "uqs_replay_recentering_dev",
    "uqs_replay_recentering_frontier", "uqs_replay_recentering_frontier_dev",
    "uqs_scanlog_read", "uqs_scanlog_count", "uqs_navlog_read", "map_recenter_shift", "map_recentre_if_needed", "frontier_score_dir",
    # multi-GPU
    "uqs_flight_shard", "uqs_row_band", "uqs_comm_unique_id", "uqs_comm_init_rank", "uqs_comm_destroy", "uqs_comm_nranks",
    "uqs_comm_rank", "uqs_nccl_version", "uqs_set_band_balance", "uqs_band_edges", "uqs_balanced_row_bands_dev", "uqs_replay_banded_dev", "uqs_replay_banded", "uqs_multi_init", "uqs_multi_count",
    "uqs_multi_select", "uqs_multi_shutdown", "uqs_multi_replay_banded", "uqs_multi_grid_dev",
    "uqs_grid_hashes_dev", "uqs_grid_hash", "uqs_set_copy_only", "uqs_replay_flow_mm", "uqs_replay_flow_boxed", "uqs_unpack_boxed",
    # drop-in symbols
    "uqs_dropin_configure", "uqs_dropin_flush", "uqs_dropin_upload", "map_reset",
    "occ_grid", "map_inited", "map_origin_x", "map_origin_y", "tof_beams_m", "pending_kf_flags",
    "world_to_grid", "raycast_update", "map_update_from_beams",
]


def exported_symbols():
    return list(_EXPORTS)


def lib() -> C.CDLL:
    """Load libuqs_mapping.so (built in-tree by ``__graft_entry__.build()``)."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise UqsError(ERR_NO_DEVICE, f"{LIB_PATH} is missing: build it (python -c 'import __graft_entry__ as g; "
                       "g.build()'); there is no fallback implementation")
    L = C.CDLL(LIB_PATH)
    fp, ip, vp = C.POINTER(C.c_float), C.c_int, C.c_void_p
    L.uqs_last_error.restype = C.c_char_p
    L.uqs_init.argtypes = [ip]
    L.uqs_set_stream.argtypes = [vp]
    L.uqs_set_tuning.argtypes = [ip, ip, ip]
    L.uqs_set_engine.argtypes = [ip, ip]
    L.uqs_set_fan_layout.argtypes = [ip]
    L.uqs_set_resident_pitch_mod.argtypes = [ip]
    L.uqs_set_decode_warp.argtypes = [ip]
    L.uqs_set_k0_bias.argtypes = [ip]
    L.uqs_set_setup_overlap.argtypes = [ip]
    L.uqs_set_profiling.argtypes = [ip]
    L.uqs_profile_collect.argtypes = [C.POINTER(C.c_double), C.POINTER(C.c_int)]
    L.uqs_profile_timeline.argtypes = [C.POINTER(C.c_double), ip]
    L.uqs_kernel_launches.restype = C.c_ulonglong
    L.uqs_pose_integrate.argtypes = [ip, ip] + [vp] * 8 + [ip]
    L.uqs_pose_integrate_dev.argtypes = [ip, ip] + [vp] * 8 + [ip]
    L.uqs_replay.argtypes = [C.POINTER(Params), ip, ip, vp, vp, vp, vp, vp, C.POINTER(Stats)]
    L.uqs_replay_dev.argtypes = [C.POINTER(Params), ip, ip, vp, vp, vp, vp, vp, ip, ip, ip, C.POINTER(Stats)]
    L.uqs_replay_flow.argtypes = [C.POINTER(Params), ip, ip] + [vp] * 10 + [C.POINTER(Stats)]
    L.uqs_beam_cells.argtypes = [C.POINTER(Params), ip, vp, vp, vp, vp, vp, vp]
    L.uqs_frame_bounds.argtypes = [C.POINTER(Params), ip, vp, vp, vp, vp, vp, vp]
    L.uqs_sincosf_batch.argtypes = [C.c_size_t, vp, vp, vp]
    L.uqs_measure_rmw_peak.argtypes = [C.POINTER(C.c_double)]
    L.uqs_measure_atoms_peak.argtypes = [C.POINTER(C.c_double)]
    L.uqs_beams_from_scans.argtypes = [C.c_longlong, vp, C.c_float, vp, vp]
    L.uqs_replay_recentering.argtypes = [C.POINTER(Params), ip, vp, vp, vp, vp, vp, vp, C.POINTER(C.c_int), vp, ip, C.POINTER(Stats)]
    L.uqs_replay_recentering_dev.argtypes = [C.POINTER(Params), ip, ip] + [vp] * 8 + [ip, C.POINTER(Stats)]
    L.uqs_frontier_scores.argtypes = [C.POINTER(Params), vp, ip, vp, vp, vp, vp, vp]
    L.uqs_replay_frontier.argtypes = [C.POINTER(Params), ip, ip, vp, vp, vp, vp, vp, ip, vp, vp, C.POINTER(Stats)]
    L.uqs_replay_frontier_dev.argtypes = [C.POINTER(Params), ip, ip, vp, vp, vp, vp, vp, ip, ip, vp, vp, C.POINTER(Stats)]
    L.uqs_replay_recentering_frontier_dev.argtypes = [C.POINTER(Params), ip, ip] + [vp] * 8 + [ip, ip, vp, vp, C.POINTER(Stats)]
    L.uqs_replay_recentering_frontier.argtypes = [C.POINTER(Params), ip, ip] + [vp] * 6 + [ip, vp, vp, C.POINTER(Stats)]
    L.uqs_scanlog_read.restype = C.c_long
    L.uqs_scanlog_read.argtypes = [C.c_char_p, ip, C.c_long] + [vp] * 11
    L.uqs_scanlog_count.restype = C.c_long
    L.uqs_scanlog_count.argtypes = [C.c_char_p, ip]
    L.uqs_navlog_read.restype = C.c_long
    L.uqs_navlog_read.argtypes = [C.c_char_p, C.c_long] + [vp] * 12
    L.uqs_flight_shard.argtypes = [ip, ip, ip, C.POINTER(C.c_int), C.POINTER(C.c_int)]
    L.uqs_flight_shard.restype = None
    L.uqs_row_band.argtypes = [ip, ip, ip, ip, C.POINTER(C.c_int), C.POINTER(C.c_int)]
    L.uqs_row_band.restype = None
    L.uqs_set_band_balance.argtypes = [ip]
    L.uqs_band_edges.argtypes = [C.POINTER(C.c_int)]
    L.uqs_balanced_row_bands_dev.argtypes = [C.POINTER(Params), ip, vp, vp, ip, C.POINTER(C.c_int)]
    L.uqs_comm_unique_id.argtypes = [vp]
    L.uqs_comm_init_rank.argtypes = [vp, ip, ip]
    L.uqs_replay_banded_dev.argtypes = [C.POINTER(Params), ip, vp, vp, vp, vp, vp, ip, C.POINTER(Stats)]
    L.uqs_replay_banded.argtypes = [C.POINTER(Params), ip, vp, vp, vp, vp, vp, C.POINTER(Stats)]
    L.uqs_multi_init.argtypes = [ip, C.POINTER(C.c_int)]
    L.uqs_multi_select.argtypes = [ip]
    L.uqs_multi_shutdown.restype = None
    L.uqs_multi_replay_banded.argtypes = [C.POINTER(Params), ip, vp, vp, vp, vp, vp, C.POINTER(Stats)]
    L.uqs_multi_grid_dev.argtypes = [ip]
    L.uqs_multi_grid_dev.restype = C.c_void_p
    L.uqs_replay_flow_mm.argtypes = [C.POINTER(Params), ip, ip] + [vp] * 10 + [C.POINTER(Stats)]
    L.uqs_replay_flow_boxed.argtypes = [C.POINTER(Params), ip, ip] + [vp] * 11 + [C.c_size_t, C.POINTER(C.c_size_t), vp, vp, C.POINTER(Stats)]
    L.uqs_unpack_boxed.argtypes = [C.POINTER(Params), ip, vp, vp, vp, vp]
    L.uqs_grid_hashes_dev.argtypes = [vp, ip, C.c_size_t, vp]
    L.uqs_grid_hash.argtypes = [vp, C.c_size_t]
    L.uqs_grid_hash.restype = C.c_uint64
    L.uqs_set_copy_only.argtypes = [ip]
    L.map_recenter_shift.argtypes = [ip, ip]
    L.map_recenter_shift.restype = None
    L.map_recentre_if_needed.argtypes = [C.c_float, C.c_float]
    L.map_recentre_if_needed.restype = None
    L.frontier_score_dir.argtypes = [C.c_float] * 4
    L.uqs_dropin_configure.argtypes = [C.POINTER(Params)]
    L.world_to_grid.argtypes = [C.c_float, C.c_float, C.POINTER(C.c_int), C.POINTER(C.c_int)]
    L.world_to_grid.restype = C.c_bool
    L.raycast_update.argtypes = [C.c_float] * 4 + [C.c_bool]
    L.raycast_update.restype = None
    L.map_update_from_beams.argtypes = [C.c_float] * 3
    L.map_update_from_beams.restype = None
    L.map_reset.restype = None
    L.uqs_dropin_flush.restype = None
    _lib = L
    return L


def _check(rc: int):
    if rc != OK:
        raise UqsError(rc, lib().uqs_last_error().decode(errors="replace"))


def init(device: int = 0):
    _check(lib().uqs_init(int(device)))


def shutdown():
    lib().uqs_shutdown()


def sync():
    _check(lib().uqs_sync())


def set_stream(ptr: Optional[int]):
    """Run on the given cudaStream_t (int handle; 0 = legacy default stream); None = library stream."""
    if ptr is None:
        _check(lib().uqs_use_own_stream())
    else:
        _check(lib().uqs_set_stream(C.c_void_p(ptr)))


def set_tuning(subtile_w: int = 0, subtile_h: int = 0, time_slices: int = 0):
    _check(lib().uqs_set_tuning(subtile_w, subtile_h, time_slices))


def set_engine(engine: int = 0, flight_warps: int = 0):
    """0 auto, 1 warp-owned sub-tiles, 2 grid resident per CTA (identical results)."""
    _check(lib().uqs_set_engine(engine, flight_warps))


def set_fan_layout(on: int = -1):
    """Lane layout of the resident engine's free-space steps: 0 = 32 beams x 1 step, 1 = 8 beams x 4 steps, -1 = default."""
    _check(lib().uqs_set_fan_layout(int(on)))


def set_decode_warp(on: int = -1):
    """Resident engine: 1 = a dedicated producer warp decodes frames for the consumer warps, 0 = shared decode, -1 = default."""
    _check(lib().uqs_set_decode_warp(int(on)))


def set_k0_bias(steps: int = 0):
    _check(lib().uqs_set_k0_bias(int(steps)))


def set_resident_pitch_mod(words_mod32: int = -1):
    _check(lib().uqs_set_resident_pitch_mod(int(words_mod32)))


def set_setup_overlap(waves: int = -1):
    """Resident device replays: n > 0 = chunks of n resident waves, each one's ray set-up beside the previous chunk's
    replay; 0 = set-up of all flights, then their replay; -1 = default (identical results)."""
    _check(lib().uqs_set_setup_overlap(int(waves)))


def setup_overlap_chunks() -> int:
    """Chunks of the last device replay whose ray set-up ran beside a replay (0: the serial schedule)."""
    return int(lib().uqs_setup_overlap_chunks())


def set_host_chunk(flights: int = 0):
    _check(lib().uqs_set_host_chunk(int(flights)))


def set_profiling(on: bool):
    _check(lib().uqs_set_profiling(1 if on else 0))


def profile_collect():
    """(ms, counts) per kernel family [pose, ray set-up, replay] since the last call; synchronises."""
    ms, cnt = (C.c_double * 3)(), (C.c_int * 3)()
    _check(lib().uqs_profile_collect(ms, cnt))
    return list(ms), list(cnt)


def profile_timeline(max_spans: int = 4096):
    """[(kind, start_ms, end_ms)] of the spans recorded since the last profile_collect(); kinds 0 pose, 1 ray
    set-up, 2 replay, 3 H2D, 4 D2H."""
    buf = (C.c_double * (3 * max_spans))()
    n = lib().uqs_profile_timeline(buf, max_spans)
    return [(int(buf[3 * i]), buf[3 * i + 1], buf[3 * i + 2]) for i in range(max(n, 0))]


def kernel_launches() -> int:
    return int(lib().uqs_kernel_launches())


def sm_count() -> int:
    return int(lib().uqs_device_sm_count())


def _f32(a, shape=None):
    a = np.ascontiguousarray(a, dtype=np.float32)
    if shape is not None and a.shape != shape:
        raise ValueError(f"expected shape {shape}, got {a.shape}")
    return a


def _ptr(a: np.ndarray) -> C.c_void_p:
    return C.c_void_p(a.ctypes.data)


def replay(p: Params, x, y, yaw_deg, ranges, out: Optional[np.ndarray] = None):
    """``uqs_replay``: x,y,yaw [F,N], ranges [F,N,32] -> (grids [F,H,W] int8, stats dict)."""
    x = _f32(x)
    if x.ndim == 1:
        x = x[None]
    F, N = x.shape
    y, yaw_deg = _f32(y).reshape(F, N), _f32(yaw_deg).reshape(F, N)
    ranges = _f32(ranges).reshape(F, N, BEAMS_PER_FRAME)
    grids = out if out is not None else np.empty((F, p.H, p.W), np.int8)
    st = Stats()
    _check(lib().uqs_replay(C.byref(p), F, N, _ptr(x), _ptr(y), _ptr(yaw_deg), _ptr(ranges), _ptr(grids), C.byref(st)))
    return grids, st.as_dict()


def replay_flow(p: Params, t_ms, of_rate_x, of_rate_y, h_m, yaw_deg, of_q, ranges, want_poses=True,
                out: Optional[np.ndarray] = None):
    """``uqs_replay_flow``: P0 then the replay, one frame per flow sample."""
    t_ms = np.ascontiguousarray(t_ms, dtype=np.uint32)
    if t_ms.ndim == 1:
        t_ms = t_ms[None]
    F, N = t_ms.shape
    rx, ry, h, yaw = (_f32(a).reshape(F, N) for a in (of_rate_x, of_rate_y, h_m, yaw_deg))
    q = np.ascontiguousarray(of_q, dtype=np.uint8).reshape(F, N)
    ranges = _f32(ranges).reshape(F, N, BEAMS_PER_FRAME)
    grids = out if out is not None else np.empty((F, p.H, p.W), np.int8)
    px = np.empty((F, N), np.float32) if want_poses else None
    py = np.empty((F, N), np.float32) if want_poses else None
    st = Stats()
    _check(lib().uqs_replay_flow(C.byref(p), F, N, _ptr(t_ms), _ptr(rx), _ptr(ry), _ptr(h), _ptr(yaw), _ptr(q),
                                 _ptr(ranges), _ptr(grids), _ptr(px) if want_poses else None,
                                 _ptr(py) if want_poses else None, C.byref(st)))
    return grids, px, py, st.as_dict()


def _flow_args(t_ms, of_rate_x, of_rate_y, h_m, yaw_deg, of_q):
    t_ms = np.ascontiguousarray(t_ms, dtype=np.uint32)
    if t_ms.ndim == 1:
        t_ms = t_ms[None]
    F, N = t_ms.shape
    rx, ry, h, yaw = (_f32(a).reshape(F, N) for a in (of_rate_x, of_rate_y, h_m, yaw_deg))
    q = np.ascontiguousarray(of_q, dtype=np.uint8).reshape(F, N)
    return F, N, t_ms, rx, ry, h, yaw, q


def replay_flow_mm(p: Params, t_ms, of_rate_x, of_rate_y, h_m, yaw_deg, of_q, ranges_mm, want_poses=True,
                   out: Optional[np.ndarray] = None):
    """``uqs_replay_flow_mm``: as replay_flow with ranges as u16 millimetres (0xFFFF = no return)."""
    F, N, t_ms, rx, ry, h, yaw, q = _flow_args(t_ms, of_rate_x, of_rate_y, h_m, yaw_deg, of_q)
    mm = np.ascontiguousarray(ranges_mm, dtype=np.uint16).reshape(F, N, BEAMS_PER_FRAME)
    grids = out if out is not None else np.empty((F, p.H, p.W), np.int8)
    px = np.empty((F, N), np.float32) if want_poses else None
    py = np.empty((F, N), np.float32) if want_poses else None
    st = Stats()
    _check(lib().uqs_replay_flow_mm(C.byref(p), F, N, _ptr(t_ms), _ptr(rx), _ptr(ry), _ptr(h), _ptr(yaw), _ptr(q), _ptr(mm),
                                    _ptr(grids), _ptr(px) if want_poses else None, _ptr(py) if want_poses else None, C.byref(st)))
    return grids, px, py, st.as_dict()


def replay_flow_boxed(p: Params, t_ms, of_rate_x, of_rate_y, h_m, yaw_deg, of_q, ranges=None, ranges_mm=None,
                      packed: Optional[np.ndarray] = None, boxes: Optional[np.ndarray] = None, offsets: Optional[np.ndarray] = None):
    """``uqs_replay_flow_boxed``: returns (boxes [F,4] int32, offsets [F] uint64, packed int8, bytes used, stats)."""
    F, N, t_ms, rx, ry, h, yaw, q = _flow_args(t_ms, of_rate_x, of_rate_y, h_m, yaw_deg, of_q)
    if (ranges is None) == (ranges_mm is None):
        raise ValueError("exactly one of ranges / ranges_mm")
    r = _f32(ranges).reshape(F, N, BEAMS_PER_FRAME) if ranges is not None else None
    mm = np.ascontiguousarray(ranges_mm, dtype=np.uint16).reshape(F, N, BEAMS_PER_FRAME) if ranges_mm is not None else None
    boxes = boxes if boxes is not None else np.empty((F, 4), np.int32)
    offsets = offsets if offsets is not None else np.empty(F, np.uint64)
    packed = packed if packed is not None else np.empty(F * p.W * p.H, np.int8)
    used = C.c_size_t(0)
    st = Stats()
    _check(lib().uqs_replay_flow_boxed(C.byref(p), F, N, _ptr(t_ms), _ptr(rx), _ptr(ry), _ptr(h), _ptr(yaw), _ptr(q),
                                       _ptr(r) if r is not None else None, _ptr(mm) if mm is not None else None,
                                       _ptr(boxes), _ptr(offsets), _ptr(packed), packed.nbytes, C.byref(used), None, None, C.byref(st)))
    return boxes, offsets, packed, int(used.value), st.as_dict()


def unpack_boxed(p: Params, boxes, offsets, packed, out: Optional[np.ndarray] = None):
    """``uqs_unpack_boxed``: dense [F,H,W] grids from the boxed form."""
    F = boxes.shape[0]
    grids = out if out is not None else np.empty((F, p.H, p.W), np.int8)
    _check(lib().uqs_unpack_boxed(C.byref(p), F, _ptr(boxes), _ptr(offsets), _ptr(packed), _ptr(grids)))
    return grids


def pose_integrate(t_ms, of_rate_x, of_rate_y, h_m, yaw_deg, of_q, mode: int = 0):
    """``uqs_pose_integrate`` (P0, builder-defined): returns x, y [F,N] float32."""
    t_ms = np.ascontiguousarray(t_ms, dtype=np.uint32)
    if t_ms.ndim == 1:
        t_ms = t_ms[None]
    F, N = t_ms.shape
    rx, ry, h, yaw = (_f32(a).reshape(F, N) for a in (of_rate_x, of_rate_y, h_m, yaw_deg))
    q = np.ascontiguousarray(of_q, dtype=np.uint8).reshape(F, N)
    xo, yo = np.empty((F, N), np.float32), np.empty((F, N), np.float32)
    _check(lib().uqs_pose_integrate(F, N, _ptr(t_ms), _ptr(rx), _ptr(ry), _ptr(h), _ptr(yaw), _ptr(q), _ptr(xo),
                                    _ptr(yo), int(mode)))
    return xo, yo


def replay_dev(p: Params, n_flights: int, n_frames: int, x_ptr: int, y_ptr: int, yaw_ptr: int, ranges_ptr: int,
               grids_ptr: int, accumulate: bool = False, row0: int = 0, rows: Optional[int] = None,
               want_stats: bool = False):
    """``uqs_replay_dev`` on raw device pointers (e.g. ``tensor.data_ptr()``); asynchronous unless stats are asked."""
    st = Stats()
    _check(lib().uqs_replay_dev(C.byref(p), n_flights, n_frames, C.c_void_p(x_ptr), C.c_void_p(y_ptr),
                                C.c_void_p(yaw_ptr), C.c_void_p(ranges_ptr), C.c_void_p(grids_ptr),
                                1 if accumulate else 0, row0, p.H if rows is None else rows,
                                C.byref(st) if want_stats else None))
    return st.as_dict() if want_stats else None


def pose_integrate_dev(n_flights, n_samples, t_ptr, rx_ptr, ry_ptr, h_ptr, yaw_ptr, q_ptr, xo_ptr, yo_ptr, mode=0):
    _check(lib().uqs_pose_integrate_dev(n_flights, n_samples, *(C.c_void_p(v) for v in
                                        (t_ptr, rx_ptr, ry_ptr, h_ptr, yaw_ptr, q_ptr, xo_ptr, yo_ptr)), int(mode)))


def beam_cells(p: Params, x, y, yaw_deg, ranges):
    """End cell of every beam (A3/A6 parity hook): returns cells [N,32,2], origin [N,2] (int32, -1 = dropped)."""
    x, y, yaw_deg = _f32(x).ravel(), _f32(y).ravel(), _f32(yaw_deg).ravel()
    N = x.size
    ranges = _f32(ranges).reshape(N, BEAMS_PER_FRAME)
    cells = np.empty((N, BEAMS_PER_FRAME, 2), np.int32)
    origin = np.empty((N, 2), np.int32)
    _check(lib().uqs_beam_cells(C.byref(p), N, _ptr(x), _ptr(y), _ptr(yaw_deg), _ptr(ranges), _ptr(cells), _ptr(origin)))
    return cells, origin


def frame_bounds(p: Params, x, y, yaw_deg, ranges):
    """Collision bound parity hook: (K0 [N], sorted [N]) per frame as the ray set-up writes them (-1 = pose off grid)."""
    x, y, yaw_deg = _f32(x).ravel(), _f32(y).ravel(), _f32(yaw_deg).ravel()
    N = x.size
    ranges = _f32(ranges).reshape(N, BEAMS_PER_FRAME)
    k0, srt = np.empty(N, np.int32), np.empty(N, np.int32)
    _check(lib().uqs_frame_bounds(C.byref(p), N, _ptr(x), _ptr(y), _ptr(yaw_deg), _ptr(ranges), _ptr(k0), _ptr(srt)))
    return k0, srt


def sincosf_batch(ang):
    ang = _f32(ang).ravel()
    s, c = np.empty_like(ang), np.empty_like(ang)
    _check(lib().uqs_sincosf_batch(ang.size, _ptr(ang), _ptr(s), _ptr(c)))
    return s, c


def beams_from_scans(raw, max_range_m: float = 4.0):
    """N1: raw [n,512] u8 (u16 LE mm, F/R/B/L x 8x8) -> (beams [n,32], dir_min [n,4])."""
    raw = np.ascontiguousarray(raw, np.uint8).reshape(-1, 512)
    n = raw.shape[0]
    beams, dmin = np.empty((n, 32), np.float32), np.empty((n, 4), np.float32)
    _check(lib().uqs_beams_from_scans(n, _ptr(raw), max_range_m, _ptr(beams), _ptr(dmin)))
    return beams, dmin


def replay_recentering(p: Params, x, y, yaw_deg, ranges):
    """N2: one log with the reference's recentering honoured -> (grid, origin, events [[frame,sx,sy]...], stats)."""
    x, y, yaw_deg = _f32(x).ravel(), _f32(y).ravel(), _f32(yaw_deg).ravel()
    n = x.size
    ranges = _f32(ranges).reshape(n, BEAMS_PER_FRAME)
    grid = np.empty((p.H, p.W), np.int8)
    origin = np.zeros(2, np.float32)
    n_ev = C.c_int(0)
    ev = np.zeros((256, 3), np.int32)
    st = Stats()
    _check(lib().uqs_replay_recentering(C.byref(p), n, _ptr(x), _ptr(y), _ptr(yaw_deg), _ptr(ranges), _ptr(grid), _ptr(origin),
                                        C.byref(n_ev), _ptr(ev), 256, C.byref(st)))
    return grid, (float(origin[0]), float(origin[1])), ev[:min(n_ev.value, 256)].copy(), st.as_dict()


def replay_recentering_dev(p: Params, n_flights: int, n_frames: int, x_ptr: int, y_ptr: int, yaw_ptr: int, ranges_ptr: int,
                           grids_ptr: int, origins_ptr: int, n_events_ptr: int, events_ptr: int = 0, max_events: int = 0,
                           want_stats: bool = False):
    """``uqs_replay_recentering_dev`` on raw device pointers (e.g. ``tensor.data_ptr()``): grids int8 [F,H,W], origins
    float32 [F,2], n_events int32 [F], events int32 [F,max_events,3] (0 = none); asynchronous unless stats are asked."""
    st = Stats()
    _check(lib().uqs_replay_recentering_dev(C.byref(p), n_flights, n_frames, C.c_void_p(x_ptr), C.c_void_p(y_ptr),
                                            C.c_void_p(yaw_ptr), C.c_void_p(ranges_ptr), C.c_void_p(grids_ptr),
                                            C.c_void_p(origins_ptr), C.c_void_p(n_events_ptr),
                                            C.c_void_p(events_ptr) if events_ptr else None, int(max_events),
                                            C.byref(st) if want_stats else None))
    return st.as_dict() if want_stats else None


def replay_recentering_flights(p: Params, x, y, yaw_deg, ranges, max_events: int = 64):
    """N2 for many flights from host arrays (x, y, yaw [F,N], ranges [F,N,32]), staged through torch on the current
    device -> (grids [F,H,W] int8, origins [F,2] float32, n_events [F] int32, events [F,max_events,3] int32, stats).
    events[f, k] is meaningful for k < min(n_events[f], max_events)."""
    import torch
    x = _f32(x)
    if x.ndim == 1:
        x = x[None]
    F, N = x.shape
    dev = torch.device("cuda", torch.cuda.current_device())
    t = [torch.from_numpy(a).to(dev) for a in (x, _f32(y).reshape(F, N), _f32(yaw_deg).reshape(F, N),
                                               _f32(ranges).reshape(F, N, BEAMS_PER_FRAME))]
    grids = torch.empty((F, p.H, p.W), dtype=torch.int8, device=dev)
    origins = torch.empty((F, 2), dtype=torch.float32, device=dev)
    n_ev = torch.empty(F, dtype=torch.int32, device=dev)
    events = torch.zeros((F, max(max_events, 0), 3), dtype=torch.int32, device=dev)
    torch.cuda.synchronize()
    st = replay_recentering_dev(p, F, N, *(a.data_ptr() for a in t), grids.data_ptr(), origins.data_ptr(), n_ev.data_ptr(),
                                events.data_ptr() if max_events > 0 else 0, max_events, want_stats=True)
    torch.cuda.synchronize()
    return grids.cpu().numpy(), origins.cpu().numpy(), n_ev.cpu().numpy(), events.cpu().numpy(), st


def frontier_scores(p: Params, grid, x, y, yaw_deg, offset_deg):
    """N3: frontier_score_dir for n queries against one grid."""
    g = np.ascontiguousarray(grid, np.int8).reshape(p.H, p.W)
    x, y, yaw_deg, offset_deg = (_f32(a).ravel() for a in (x, y, yaw_deg, offset_deg))
    out = np.empty(x.size, np.int32)
    _check(lib().uqs_frontier_scores(C.byref(p), _ptr(g), x.size, _ptr(x), _ptr(y), _ptr(yaw_deg), _ptr(offset_deg), _ptr(out)))
    return out


# ``uqs_query``: 24 bytes, no padding (include/uqs_mapping.h)
QUERY_DTYPE = np.dtype([("flight", "<i4"), ("frame", "<i4"), ("x", "<f4"), ("y", "<f4"), ("yaw_deg", "<f4"),
                        ("offset_deg", "<f4")])


def make_queries(flight, frame, x, y, yaw_deg, offset_deg) -> np.ndarray:
    """Array of ``uqs_query`` records from six broadcastable columns."""
    cols = np.broadcast_arrays(*(np.asarray(a) for a in (flight, frame, x, y, yaw_deg, offset_deg)))
    q = np.empty(cols[0].size, QUERY_DTYPE)
    for name, c in zip(QUERY_DTYPE.names, cols):
        q[name] = c.ravel()
    return q


def replay_frontier(p: Params, x, y, yaw_deg, ranges, queries, want_grids: bool = True):
    """``uqs_replay_frontier``: the replay of ``replay`` plus frontier_score_dir for every query against its flight's
    grid after frames 0..frame.  Returns (grids [F,H,W] int8 or None, scores [n] int32, stats dict)."""
    x = _f32(x)
    if x.ndim == 1:
        x = x[None]
    F, N = x.shape
    y, yaw_deg = _f32(y).reshape(F, N), _f32(yaw_deg).reshape(F, N)
    ranges = _f32(ranges).reshape(F, N, BEAMS_PER_FRAME)
    q = np.ascontiguousarray(queries, QUERY_DTYPE)
    grids = np.empty((F, p.H, p.W), np.int8) if want_grids else None
    scores = np.empty(q.size, np.int32)
    st = Stats()
    _check(lib().uqs_replay_frontier(C.byref(p), F, N, _ptr(x), _ptr(y), _ptr(yaw_deg), _ptr(ranges),
                                     _ptr(grids) if grids is not None else None, q.size, _ptr(q) if q.size else None,
                                     _ptr(scores) if q.size else None, C.byref(st)))
    return grids, scores, st.as_dict()


def replay_frontier_dev(p: Params, n_flights: int, n_frames: int, x_ptr: int, y_ptr: int, yaw_ptr: int, ranges_ptr: int,
                        grids_ptr: int, n_queries: int, queries_ptr: int, scores_ptr: int, accumulate: bool = False,
                        want_stats: bool = False):
    """``uqs_replay_frontier_dev`` on raw device pointers (queries: ``QUERY_DTYPE`` records, scores: int32);
    asynchronous unless stats are asked."""
    st = Stats()
    _check(lib().uqs_replay_frontier_dev(C.byref(p), n_flights, n_frames, C.c_void_p(x_ptr), C.c_void_p(y_ptr),
                                         C.c_void_p(yaw_ptr), C.c_void_p(ranges_ptr), C.c_void_p(grids_ptr),
                                         1 if accumulate else 0, int(n_queries), C.c_void_p(queries_ptr),
                                         C.c_void_p(scores_ptr), C.byref(st) if want_stats else None))
    return st.as_dict() if want_stats else None


def replay_recentering_frontier(p: Params, x, y, yaw_deg, ranges, queries, want_grids: bool = True):
    """``uqs_replay_recentering_frontier``: the replay of ``replay_recentering_flights`` plus frontier_score_dir for every
    query against its flight's recentred map at its frame, in the window of the origin the flight had then.  Returns
    (grids [F,H,W] int8 or None, origins [F,2] float32 or None, scores [n] int32, stats dict)."""
    x = _f32(x)
    if x.ndim == 1:
        x = x[None]
    F, N = x.shape
    y, yaw_deg = _f32(y).reshape(F, N), _f32(yaw_deg).reshape(F, N)
    ranges = _f32(ranges).reshape(F, N, BEAMS_PER_FRAME)
    q = np.ascontiguousarray(queries, QUERY_DTYPE)
    grids = np.empty((F, p.H, p.W), np.int8) if want_grids else None
    origins = np.empty((F, 2), np.float32) if want_grids else None
    scores = np.empty(q.size, np.int32)
    st = Stats()
    _check(lib().uqs_replay_recentering_frontier(C.byref(p), F, N, _ptr(x), _ptr(y), _ptr(yaw_deg), _ptr(ranges),
                                                 _ptr(grids) if grids is not None else None,
                                                 _ptr(origins) if origins is not None else None, q.size,
                                                 _ptr(q) if q.size else None, _ptr(scores) if q.size else None, C.byref(st)))
    return grids, origins, scores, st.as_dict()


def replay_recentering_frontier_dev(p: Params, n_flights: int, n_frames: int, x_ptr: int, y_ptr: int, yaw_ptr: int,
                                    ranges_ptr: int, grids_ptr: int, origins_ptr: int, n_events_ptr: int, events_ptr: int,
                                    max_events: int, n_queries: int, queries_ptr: int, scores_ptr: int,
                                    want_stats: bool = False):
    """``uqs_replay_recentering_frontier_dev`` on raw device pointers: the buffers of ``replay_recentering_dev`` plus
    queries (``QUERY_DTYPE`` records) and scores (int32); asynchronous unless stats are asked."""
    st = Stats()
    _check(lib().uqs_replay_recentering_frontier_dev(C.byref(p), n_flights, n_frames, C.c_void_p(x_ptr), C.c_void_p(y_ptr),
                                                     C.c_void_p(yaw_ptr), C.c_void_p(ranges_ptr), C.c_void_p(grids_ptr),
                                                     C.c_void_p(origins_ptr), C.c_void_p(n_events_ptr),
                                                     C.c_void_p(events_ptr) if events_ptr else None, int(max_events),
                                                     int(n_queries), C.c_void_p(queries_ptr) if queries_ptr else None,
                                                     C.c_void_p(scores_ptr) if scores_ptr else None,
                                                     C.byref(st) if want_stats else None))
    return st.as_dict() if want_stats else None


def navlog_read(path: str) -> dict:
    """N4: navlog.csv -> SoA numpy arrays (the columns P0 and the mapper consume; host file I/O in the C library)."""
    L = lib()
    n = L.uqs_navlog_read(path.encode(), 0, *([None] * 12))
    if n < 0:
        raise UqsError(ERR_BAD_ARG, f"cannot read nav log {path} (code {n})")
    f32 = ("yaw_deg", "alt_m", "x_m", "y_m", "vx_mps", "vy_mps", "rf_m")
    d = {"t_ms": np.empty(n, np.uint32), **{k: np.empty(n, np.float32) for k in f32}, "of_q": np.empty(n, np.uint8),
         "of_rate_x": np.empty(n, np.float32), "of_rate_y": np.empty(n, np.float32), "tof4": np.empty((n, 4), np.float32)}
    order = ("t_ms",) + f32 + ("of_q", "of_rate_x", "of_rate_y", "tof4")
    got = L.uqs_navlog_read(path.encode(), n, *(_ptr(d[k]) for k in order))
    if got != n:
        raise UqsError(ERR_BAD_ARG, f"nav log {path} changed while reading ({got} != {n})")
    return d


def scanlog_read(path: str, keep_nan_pose: bool = False) -> dict:
    """N4: scanlog.bin -> SoA numpy arrays (host file I/O in the C library)."""
    L = lib()
    n = L.uqs_scanlog_count(path.encode(), int(keep_nan_pose))
    if n < 0:
        raise UqsError(ERR_BAD_ARG, f"cannot read scan log {path} (code {n})")
    d = {"host_ms": np.empty(n, np.uint32), "scan_ms": np.empty(n, np.uint32), "x_m": np.empty(n, np.float32),
         "y_m": np.empty(n, np.float32), "yaw_deg": np.empty(n, np.float32), "alt_m": np.empty(n, np.float32),
         "of_rate_x": np.empty(n, np.float32), "of_rate_y": np.empty(n, np.float32), "of_q": np.empty(n, np.uint8),
         "kf_flags": np.empty(n, np.uint8), "grid_raw": np.empty((n, 512), np.uint8)}
    got = L.uqs_scanlog_read(path.encode(), int(keep_nan_pose), n, *(_ptr(d[k]) for k in
                             ("host_ms", "scan_ms", "x_m", "y_m", "yaw_deg", "alt_m", "of_rate_x", "of_rate_y", "of_q", "kf_flags", "grid_raw")))
    if got != n:
        raise UqsError(ERR_BAD_ARG, f"scan log changed while reading ({got} != {n})")
    return d


# ---- multi-GPU (include/uqs_mapping.h, "Multi-GPU") ------------------------------------------------------------
def flight_shard(n_flights: int, rank: int, world: int):
    """``uqs_flight_shard``: [first, count) of the flights ``rank`` replays (host arithmetic, no device needed)."""
    if world <= 0 or not (0 <= rank < world):
        raise ValueError("bad rank/world")
    a, b = C.c_int(0), C.c_int(0)
    lib().uqs_flight_shard(int(n_flights), int(rank), int(world), C.byref(a), C.byref(b))
    return a.value, b.value


def row_band(H: int, rank: int, world: int, align: int = 4):
    """``uqs_row_band``: [row0, rows) of the grid rows ``rank`` owns (host arithmetic, no device needed)."""
    if world <= 0 or not (0 <= rank < world):
        raise ValueError("bad rank/world")
    a, b = C.c_int(0), C.c_int(0)
    lib().uqs_row_band(int(H), int(rank), int(world), int(align), C.byref(a), C.byref(b))
    return a.value, b.value


def comm_unique_id() -> bytes:
    buf = C.create_string_buffer(COMM_ID_BYTES)
    _check(lib().uqs_comm_unique_id(buf))
    return buf.raw


def comm_init_rank(uid: bytes, nranks: int, rank: int):
    if len(uid) != COMM_ID_BYTES:
        raise ValueError("the communicator id is 128 bytes")
    _check(lib().uqs_comm_init_rank(C.create_string_buffer(uid, COMM_ID_BYTES), int(nranks), int(rank)))


def comm_destroy():
    _check(lib().uqs_comm_destroy())


def comm_nranks() -> int:
    return int(lib().uqs_comm_nranks())


def set_band_balance(on: bool = True):
    _check(lib().uqs_set_band_balance(1 if on else 0))


def balanced_row_bands_dev(p: Params, n_frames: int, x_ptr: int, y_ptr: int, world: int):
    """``uqs_balanced_row_bands_dev``: the row cuts a ``world``-rank banded replay of this log would use."""
    e = (C.c_int * (world + 1))()
    _check(lib().uqs_balanced_row_bands_dev(C.byref(p), int(n_frames), C.c_void_p(x_ptr), C.c_void_p(y_ptr), int(world), e))
    return list(e)


def band_edges():
    """Row cuts of the last banded replay: rank r owned rows [e[r], e[r+1])."""
    e = (C.c_int * 17)()
    n = lib().uqs_band_edges(e)
    return list(e[:n + 1])


def nccl_version() -> int:
    return int(lib().uqs_nccl_version())


def replay_banded_dev(p: Params, n_frames: int, x_ptr: int, y_ptr: int, yaw_ptr: int, ranges_ptr: int, grid_ptr: int,
                      gather: bool = True, want_stats: bool = False):
    """``uqs_replay_banded_dev``: this rank's owned row band of one grid, then the all-gather of the bands."""
    st = Stats()
    _check(lib().uqs_replay_banded_dev(C.byref(p), int(n_frames), C.c_void_p(x_ptr), C.c_void_p(y_ptr), C.c_void_p(yaw_ptr),
                                       C.c_void_p(ranges_ptr), C.c_void_p(grid_ptr), 1 if gather else 0,
                                       C.byref(st) if want_stats else None))
    return st.as_dict() if want_stats else None


def replay_banded(p: Params, x, y, yaw_deg, ranges, out: Optional[np.ndarray] = None, want_grid: bool = True):
    """``uqs_replay_banded`` (host buffers, one process per GPU): returns (grid or None, stats)."""
    x, y, yaw_deg = _f32(x).ravel(), _f32(y).ravel(), _f32(yaw_deg).ravel()
    n = x.size
    ranges = _f32(ranges).reshape(n, BEAMS_PER_FRAME)
    grid = (out if out is not None else np.empty((p.H, p.W), np.int8)) if want_grid else None
    st = Stats()
    _check(lib().uqs_replay_banded(C.byref(p), n, _ptr(x), _ptr(y), _ptr(yaw_deg), _ptr(ranges),
                                   _ptr(grid) if grid is not None else None, C.byref(st)))
    return grid, st.as_dict()


def multi_init(n_devices: int, devices=None):
    arr = (C.c_int * n_devices)(*devices) if devices is not None else None
    _check(lib().uqs_multi_init(int(n_devices), arr))


def multi_select(i: int):
    _check(lib().uqs_multi_select(int(i)))


def multi_shutdown():
    lib().uqs_multi_shutdown()


def multi_replay_banded(p: Params, x, y, yaw_deg, ranges, out: Optional[np.ndarray] = None):
    """``uqs_multi_replay_banded``: config 4 on every device of ``multi_init`` from one host thread."""
    x, y, yaw_deg = _f32(x).ravel(), _f32(y).ravel(), _f32(yaw_deg).ravel()
    n = x.size
    ranges = _f32(ranges).reshape(n, BEAMS_PER_FRAME)
    grid = out if out is not None else np.empty((p.H, p.W), np.int8)
    st = Stats()
    _check(lib().uqs_multi_replay_banded(C.byref(p), n, _ptr(x), _ptr(y), _ptr(yaw_deg), _ptr(ranges), _ptr(grid), C.byref(st)))
    return grid, st.as_dict()


def grid_hashes_dev(grids_ptr: int, n_grids: int, cells: int) -> np.ndarray:
    """``uqs_grid_hashes_dev``: 64-bit digest of each device grid (sum of splitmix64(i << 8 | byte)); synchronises."""
    out = np.empty(n_grids, np.uint64)
    _check(lib().uqs_grid_hashes_dev(C.c_void_p(grids_ptr), int(n_grids), int(cells), _ptr(out)))
    return out


def grid_hash(grid: np.ndarray) -> int:
    """``uqs_grid_hash``: the same digest of one host grid (plain host arithmetic in the C library)."""
    g = np.ascontiguousarray(grid, np.int8)
    return int(lib().uqs_grid_hash(_ptr(g), g.size))


def set_copy_only(on: bool):
    _check(lib().uqs_set_copy_only(1 if on else 0))


def measure_atoms_peak() -> float:
    """Shared-memory atomic (ATOMS.ADD) update rate, conflict-free: the price of the north star's atomics sketch."""
    v = C.c_double(0)
    _check(lib().uqs_measure_atoms_peak(C.byref(v)))
    return float(v.value)


def measure_rmw_peak() -> float:
    v = C.c_double(0)
    _check(lib().uqs_measure_rmw_peak(C.byref(v)))
    return float(v.value)


class DropIn:
    """The reference's own symbols (``map_update_from_beams`` & co.) through the C ABI."""

    def __init__(self, p: Params):
        self.L = lib()
        self.p = p.copy()
        _check(self.L.uqs_dropin_configure(C.byref(self.p)))

    def _g(self, ctype, name):
        return ctype.in_dll(self.L, name)

    def hover_init(self, ox: float, oy: float):
        """uav_local_nav.c:2187-2194: origin := pose, clear grid, map_inited = true."""
        self._g(C.c_float, "map_origin_x").value = ox
        self._g(C.c_float, "map_origin_y").value = oy
        self.L.map_reset()
        self._g(C.c_bool, "map_inited").value = True

    def set_inited(self, v: bool):
        self._g(C.c_bool, "map_inited").value = v

    def set_beams(self, beams32):
        arr = (C.c_float * 32).in_dll(self.L, "tof_beams_m")
        b = _f32(beams32).ravel()
        C.memmove(arr, b.ctypes.data, 128)

    def map_update_from_beams(self, x, y, yaw):
        self.L.map_update_from_beams(np.float32(x), np.float32(y), np.float32(yaw))

    def raycast_update(self, x0, y0, x1, y1, hit):
        self.L.raycast_update(np.float32(x0), np.float32(y0), np.float32(x1), np.float32(y1), bool(hit))

    def world_to_grid(self, x, y):
        gx, gy = C.c_int(-1), C.c_int(-1)
        ok = self.L.world_to_grid(np.float32(x), np.float32(y), C.byref(gx), C.byref(gy))
        return bool(ok), gx.value, gy.value

    def map_recentre_if_needed(self, x, y):
        self.L.map_recentre_if_needed(np.float32(x), np.float32(y))

    def frontier_score_dir(self, x, y, yaw, off) -> int:
        return int(self.L.frontier_score_dir(np.float32(x), np.float32(y), np.float32(yaw), np.float32(off)))

    def origin(self):
        return self._g(C.c_float, "map_origin_x").value, self._g(C.c_float, "map_origin_y").value

    def kf_flags(self) -> int:
        return self._g(C.c_uint8, "pending_kf_flags").value

    def grid(self) -> np.ndarray:
        self.L.uqs_dropin_flush()
        ptr = C.POINTER(C.c_int8).in_dll(self.L, "occ_grid")
        return np.ctypeslib.as_array(ptr, shape=(self.p.H, self.p.W)).copy()
