/*
 * uqs_mapping.h -- C ABI of the B200-native post-flight 2D mapping path.
 *
 * This header is the drop-in boundary for ONE path of exie1122/micro-quad-SLAM:
 * poses -> ToF beam ray-cast -> int8 log-odds occupancy grid, i.e. the block
 * uav_local_nav.c:181-306 as driven from log_tick() at uav_local_nav.c:1629-1635.
 * All of it runs as hand-written CUDA for sm_100a inside libuqs_mapping.so; there
 * is no CPU implementation in the library and every entry point fails (returns
 * non-zero / becomes a no-op with uqs_last_error() set) when no CUDA device is
 * usable.
 *
 * Two groups of symbols:
 *
 *  (1) DROP-IN symbols -- same names, types and argument meaning as the
 *      reference's file-static mapping symbols, so uav_local_nav.c can be built
 *      with lines 181-385 removed and this header included instead
 *      (see INTEGRATION.md).  Reference failure behaviour is kept: they are
 *      silent no-ops when !map_inited or when a ray is off-grid.
 *
 *  (2) BATCH symbols (uqs_*) -- what a post-flight replay harness calls: whole
 *      logs, many flights, device-resident or host buffers, explicit errors.
 *
 * Plain C, plain pointers and sizes; no CUDA or torch types appear here.
 */
#ifndef UQS_MAPPING_H
#define UQS_MAPPING_H

#include <stdbool.h>
#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

/* ------------------------------------------------------------------------ */
/* Geometry and sensor constants.  In the reference these are compile-time   */
/* #defines / static consts; here they are one runtime struct.               */
/* ------------------------------------------------------------------------ */
typedef struct uqs_params {
  int32_t W, H;          /* MAP_W, MAP_H                     uav_local_nav.c:185-186 */
  float   res_m;         /* MAP_RES_M                        uav_local_nav.c:182     */
  float   size_m;        /* MAP_SIZE_M (recentering only)    uav_local_nav.c:183     */
  float   origin_x;      /* map_origin_x: world x at cell W/2   uav_local_nav.c:191  */
  float   origin_y;      /* map_origin_y: world y at cell H/2   uav_local_nav.c:192  */
  float   max_range_m;   /* TOF_MAX_RANGE_M = 4.00f          uav_local_nav.c:117     */
  float   fov_deg;       /* TOF_FOV_DEG = 63.0f              uav_local_nav.c:118     */
  float   min_range_m;   /* the 0.05f literal in `dist <= 0.05f`   uav_local_nav.c:290 */
  float   hit_margin_m;  /* the 0.05f literal in `MAX - 0.05f`     uav_local_nav.c:292 */
  int32_t lo_free;       /* LO_FREE_DEC = 1                  uav_local_nav.c:194     */
  int32_t lo_occ;        /* LO_OCC_INC  = 6                  uav_local_nav.c:195     */
  int32_t lo_min;        /* LO_MIN = -80                     uav_local_nav.c:196     */
  int32_t lo_max;        /* LO_MAX = +80                     uav_local_nav.c:197     */
} uqs_params;

/* The reference's own constants (500x500 @ 0.10 m, origin to be set by caller). */
void uqs_params_default(uqs_params* p);

#define UQS_BEAMS_PER_FRAME 32   /* 4 directions x TOF_COLS(8), uav_local_nav.c:105,286-287 */

/* Error codes returned by uqs_* batch calls (0 = ok). */
enum {
  UQS_OK = 0,
  UQS_ERR_NO_DEVICE = 1,     /* no CUDA device / driver: nothing can run          */
  UQS_ERR_CUDA = 2,          /* a CUDA call or kernel failed; see uqs_last_error() */
  UQS_ERR_BAD_ARG = 3,       /* NULL pointer, non-positive size, bad params        */
  UQS_ERR_NOT_INIT = 4,      /* uqs_init() has not succeeded                       */
  UQS_ERR_DOMAIN = 5,        /* internal consistency failure: a ray reached an engine that cannot represent
                                it.  No input raises it since every float angle (glibc's reduce_large branch
                                included) and every ray length is covered -- see uqs_set_engine() */
  UQS_ERR_NOMEM = 6,
  UQS_ERR_NO_NCCL = 7,       /* libnccl.so.2 could not be loaded (multi-GPU entry points only) */
  UQS_ERR_NCCL = 8           /* an NCCL call failed; see uqs_last_error()                       */
};

/* Counters returned by the replay calls.  All exact integers. */
typedef struct uqs_stats {
  uint64_t ray_cell_updates;  /* U = sum over accepted rays of max(|dgx|,|dgy|)+1:
                                 iterations of the while(1) at uav_local_nav.c:254-277 */
  uint64_t rays_accepted;     /* rays that reached raycast_update with both ends on grid */
  uint64_t rays_skipped;      /* NaN / <= min_range (:289-290) or off-grid (:243-244)   */
  uint64_t frames;            /* map_update_from_beams calls replayed                   */
  uint64_t domain_errors;     /* rays dropped because of UQS_ERR_DOMAIN (should be 0)   */
} uqs_stats;

/* ------------------------------------------------------------------------ */
/* (2) Batch API                                                             */
/* ------------------------------------------------------------------------ */

/* Select a CUDA device, create the library's stream and scratch allocator.
 * Returns UQS_ERR_NO_DEVICE if none is available (there is no fallback). */
int  uqs_init(int device);
void uqs_shutdown(void);
const char* uqs_last_error(void);
int  uqs_device_sm_count(void);

/* Run all subsequent work on the caller's CUDA stream (a cudaStream_t passed as
 * void*; NULL is the legacy default stream).  uqs_use_own_stream() goes back to the
 * library's own stream.  Lets a host time the kernels
 * with its own events. */
int  uqs_set_stream(void* cuda_stream);
int  uqs_use_own_stream(void);
/* Number of kernels this library has launched so far (bench.py's gpu_launches). */
unsigned long long uqs_kernel_launches(void);
/* Per-kernel device timing with events on the launching stream.  uqs_profile_collect()
 * returns the summed device time (ms) and launch count per kernel family since the last
 * call -- [0] pose integration, [1] ray set-up, [2] replay -- and synchronises. */
int  uqs_set_profiling(int on);
int  uqs_profile_collect(double ms[3], int counts[3]);
/* Timeline of the spans recorded since the last uqs_profile_collect(): out[3*i] = kind (0 pose,
 * 1 ray set-up, 2 replay, 3 H2D copy, 4 D2H copy of the host-buffer pipeline), out[3*i+1] and
 * out[3*i+2] = start and end in ms after the first span's start.  Returns the number of spans
 * written (<= max_spans, -1 when not initialised); does not clear them; synchronises the device. */
int  uqs_profile_timeline(double* out, int max_spans);
/* Block until everything enqueued so far has finished. */
int  uqs_sync(void);

/* Kernel tuning knobs (0 keeps the built-in choice).  sub-tile = the rectangle of
 * cells one warp owns in shared memory; time_slices > 1 splits a flight's frames
 * into contiguous slices that are replayed concurrently and composed exactly
 * (1 = never slice).  Any setting produces identical bytes. */
int  uqs_set_tuning(int subtile_w, int subtile_h, int time_slices);
/* Replay engine: 0 = automatic (each flight's touched bounding box resident in one CTA's
 * shared memory when it fits and there are at least SMs/4 flights; warp-owned
 * sub-tiles otherwise), 1 = always sub-tiles, 2 = always resident
 * (error if the flights' touched bounding box does not fit), 3 = always the unrestricted
 * kernel.  flight_warps = warps per CTA of the resident engine (0 = automatic, 4, 8, 16
 * or 32).  All engines produce identical bytes.
 * The unrestricted kernel (one warp per flight on the grid in global memory, the
 * reference's loop statement for statement) is what engines 0-2 route to by themselves
 * for the inputs their fast paths do not cover: rays that can exceed 1024 cells
 * (max_range_m / res_m > 1021 on a grid wider than 1025 cells, or raycast_update() on
 * such a grid), a clamp range that excludes 0, and accumulate != 0 onto a grid holding
 * values outside [lo_min, lo_max].  Nothing is refused or approximated. */
int  uqs_set_engine(int engine, int flight_warps);
/* Lane layout of the resident engine's free-space steps: 0 = the 32 beams of a frame x 1 step per warp
 * instruction, 1 = the 8 beams of one sensor x 4 consecutive steps (fewer shared-memory bank conflicts).
 * -1 = the built-in choice.  Identical bytes either way.  uqs_replay_frontier[_dev] ignores this knob. */
int  uqs_set_fan_layout(int on);
/* Resident engine with a dedicated decode warp: 0 = every warp decodes every NW-th frame of its flight, 1 = an
 * extra producer warp per CTA does nothing but decode frames into the shared-memory ring, two frames ahead of the
 * consumer warps (4, 8 or 16 of them).  -1 = the built-in choice.  Identical bytes either way.
 * uqs_replay_frontier[_dev] ignores this knob. */
int  uqs_set_decode_warp(int on);
/* Measurement knob: adds `steps` (0..8) to every frame's collision bound K0, capped at the frame's longest beam
 * (always safe; identical bytes): what one collision-checked step per frame costs the resident engine. */
int  uqs_set_k0_bias(int steps);
/* Experiment knob for the layouts above: row pitch of the resident box in 32-bit words, modulo 32
 * (-1 = the built-in odd pitch).  Identical bytes for any value. */
int  uqs_set_resident_pitch_mod(int words_mod32);

/*
 * P0 -- dead-reckoning pose integration (BUILDER-DEFINED: the reference has no
 * such stage; spec in DESIGN.md section "P0", mirrors uav_local_nav.c:943,1151-1164).
 * Arrays are [n_flights][n_samples], row-major.  x_out/y_out get the pose of
 * every sample; x[0]=y[0]=0.
 *   mode 0: exact -- increments in parallel, summation replayed in sample order
 *           (bit-identical to the CPU statement of the spec)
 *   mode 1: scan  -- decoupled-lookback prefix scan in binary64 (throughput
 *           variant; differs from mode 0 by the fp32 rounding of the serial sum)
 */
int uqs_pose_integrate(int n_flights, int n_samples,
                       const uint32_t* t_ms, const float* of_rate_x, const float* of_rate_y,
                       const float* h_m, const float* yaw_deg, const uint8_t* of_q,
                       float* x_out, float* y_out, int mode);

/*
 * Replay n_flights independent logs of n_frames frames each into n_flights
 * grids of W*H int8 (row-major, k = gy*W + gx, uav_local_nav.c:216), each
 * starting from all-zero (uav_local_nav.c:2190).  For every frame this is
 * exactly map_update_from_beams(x, y, yaw_deg) (uav_local_nav.c:280-306) with
 * tof_beams_m = ranges[frame][0..31] (direction-major F,R,B,L x 8 columns).
 * Host buffers; H2D/D2H copies are part of the call.
 *   x, y, yaw_deg : [n_flights][n_frames]      ranges : [n_flights][n_frames][32]
 *   grids_out     : [n_flights][H][W] int8
 */
int uqs_replay(const uqs_params* p, int n_flights, int n_frames,
               const float* x, const float* y, const float* yaw_deg, const float* ranges,
               int8_t* grids_out, uqs_stats* stats);

/* The host-buffer calls cut the flights into chunks and overlap H2D, kernels and D2H of
 * successive chunks (page-locked host buffers needed for the overlap).  0 = automatic. */
int uqs_set_host_chunk(int flights_per_chunk);

/* Same, with every pointer a DEVICE pointer on the device given to uqs_init().
 * accumulate != 0 continues from the grids' current contents instead of zero
 * (used for chained replays and by the drop-in symbols).  row0/rows restrict
 * the update to grid rows [row0, row0+rows) -- the tile a GPU owns when one
 * large grid is split across GPUs; pass 0, H for the whole grid.  grids_dev
 * always addresses full W*H grids.  Asynchronous on the current stream; stats
 * (host pointer, may be NULL) is filled after an internal sync only if given. */
int uqs_replay_dev(const uqs_params* p, int n_flights, int n_frames,
                   const float* x_dev, const float* y_dev, const float* yaw_dev,
                   const float* ranges_dev, int8_t* grids_dev,
                   int accumulate, int row0, int rows, uqs_stats* stats);

/* P0 followed by the replay, one frame per flow sample (frame i uses pose i and
 * yaw_deg[i]).  Host buffers.  poses_out_x/y may be NULL. */
int uqs_replay_flow(const uqs_params* p, int n_flights, int n_samples,
                    const uint32_t* t_ms, const float* of_rate_x, const float* of_rate_y,
                    const float* h_m, const float* yaw_deg, const uint8_t* of_q,
                    const float* ranges, int8_t* grids_out,
                    float* poses_out_x, float* poses_out_y, uqs_stats* stats);

/* uqs_replay_flow with the ranges as u16 MILLIMETRES (0xFFFF = no return): the unit the ToF sensors deliver and
 * the reference converts with `(float)mm * 0.001f` (uav_local_nav.c:1327-1328); the device applies that same
 * binary32 multiply, so a log given in either form yields identical bytes.  Halves the host-to-device traffic. */
int uqs_replay_flow_mm(const uqs_params* p, int n_flights, int n_samples,
                       const uint32_t* t_ms, const float* of_rate_x, const float* of_rate_y,
                       const float* h_m, const float* yaw_deg, const uint8_t* of_q,
                       const uint16_t* ranges_mm, int8_t* grids_out,
                       float* poses_out_x, float* poses_out_y, uqs_stats* stats);

/* uqs_replay_flow with BOXED output: per flight the bounding box of every cell it touched
 * (boxes_out[f] = {x0, y0, x1, y1}, upper corner exclusive; all zeros for a flight without any accepted ray) and
 * the box's cells, row-major with row pitch x1 - x0, at packed_out + offsets_out[f].  Cells outside the box are 0
 * by construction (uav_local_nav.c:2190 and no update reached them).  Exactly one of ranges (float metres) /
 * ranges_mm (u16 millimetres) is non-NULL.  packed_cap = bytes available at packed_out (n_flights * W * H always
 * suffices); *packed_bytes = bytes used; UQS_ERR_NOMEM when more were needed.  The device-to-host traffic is the
 * touched region only (~28 % of a 400x400 grid for a 60 s flight).  uqs_unpack_boxed() (plain host code) expands
 * the result to dense [n_flights][H][W] grids. */
int uqs_replay_flow_boxed(const uqs_params* p, int n_flights, int n_samples,
                          const uint32_t* t_ms, const float* of_rate_x, const float* of_rate_y,
                          const float* h_m, const float* yaw_deg, const uint8_t* of_q,
                          const float* ranges, const uint16_t* ranges_mm,
                          int32_t* boxes_out, uint64_t* offsets_out, int8_t* packed_out, size_t packed_cap,
                          size_t* packed_bytes, float* poses_out_x, float* poses_out_y, uqs_stats* stats);
int uqs_unpack_boxed(const uqs_params* p, int n_flights, const int32_t* boxes, const uint64_t* offsets,
                     const int8_t* packed, int8_t* grids_out);

/* Device-pointer form of uqs_pose_integrate (asynchronous on the current stream). */
int uqs_pose_integrate_dev(int n_flights, int n_samples,
                           const uint32_t* t_ms, const float* of_rate_x, const float* of_rate_y,
                           const float* h_m, const float* yaw_deg, const uint8_t* of_q,
                           float* x_out, float* y_out, int mode);

/* Batched world_to_grid / beam end-points on the device (host buffers), used by
 * the parity tests to compare cell indices one by one with the reference.
 *   cells_out : [n][32][2] int32 end cell (gx,gy) or (-1,-1) when the ray is skipped
 *   origin_out: [n][2] int32 start cell or (-1,-1) */
int uqs_beam_cells(const uqs_params* p, int n_frames,
                   const float* x, const float* y, const float* yaw_deg, const float* ranges,
                   int32_t* cells_out, int32_t* origin_out);
/* Parity hook for the collision bound of the resident engine: per frame, K0 (two beams of the frame can share
 * a cell only at steps k < K0; -1 when the frame's pose is off the grid) as the resident engine receives it,
 * uqs_set_k0_bias included, and whether the frame's beams were found in circular angular order.  Host pointers. */
int uqs_frame_bounds(const uqs_params* p, int n_frames, const float* x, const float* y, const float* yaw_deg,
                     const float* ranges, int32_t* k0_out, int32_t* sorted_out);

/* Device evaluation of the glibc-2.39 sincosf restatement for n host floats
 * (parity test hook for SURVEY.md Appendix B). */
int uqs_sincosf_batch(size_t n, const float* ang, float* sin_out, float* cos_out);

/* ---- rows either side of the path (SURVEY.md section 8(f)) ------------------------------- */

/* N1: raw ToF scans -> tof_beams_m.  raw = [n][512] bytes, 4 sensors (F,R,B,L) x 64 cells x u16 LE mm
 * (scanrec_t.grid_raw, uav_local_nav.c:1546; wire format tof_esp32.ino:192-211).  Per column the
 * second-smallest valid row (robust_col_dist_m, :1320-1342).  dir_min (may be NULL) = tof_min_m[4]. */
int uqs_beams_from_scans(long long n_frames, const uint8_t* raw, float max_range_m, float* beams_out /* [n][32] */,
                         float* dir_min_out /* [n][4] or NULL */);
int uqs_beams_from_scans_dev(long long n_frames, const uint8_t* raw_dev, float max_range_m, float* beams_dev,
                             float* dir_min_dev);

/* N2: replay ONE log exactly as log_tick() does with recentering enabled (uav_local_nav.c:1629-1635:
 * map_recentre_if_needed(pose) before every update).  origin_out = final map origin; events_out receives
 * up to max_events {frame, sx_cells, sy_cells} triples. */
int uqs_replay_recentering(const uqs_params* p, int n_frames, const float* x, const float* y, const float* yaw_deg,
                           const float* ranges, int8_t* grid_out, float origin_out[2], int* n_events_out,
                           int* events_out, int max_events, uqs_stats* stats);

/* N3: frontier_score_dir() (uav_local_nav.c:356-385) for n queries against one host grid. */
int uqs_frontier_scores(const uqs_params* p, const int8_t* grid, int n, const float* x, const float* y,
                        const float* yaw_deg, const float* offset_deg, int* scores_out);

/* N3 at the frame a decision was taken: one frontier query (24 bytes, no padding).  Its score is what
 * frontier_score_dir(x, y, yaw_deg, offset_deg) returns when occ_grid holds flight `flight`'s grid after its frames
 * 0..frame have been applied -- the map EXPLORE scored against in the control tick of that frame (uav_local_nav.c:
 * 1715-1736, 2225-2253).  The query carries its own pose (the controller's pose at the tick); pass x[f], y[f], yaw[f]
 * for the frame's own pose. */
typedef struct uqs_query {
  int32_t flight, frame;
  float   x, y, yaw_deg, offset_deg;
} uqs_query;

/* uqs_replay_dev plus n_queries frontier queries answered inside the same replay: scores_dev[i] = score of
 * queries_dev[i] (input order; any order of queries, duplicates and many per frame are fine).  Grids and stats are
 * byte-identical to uqs_replay_dev with the same arguments (row0 = 0, rows = H: whole grids only); n_queries == 0 is
 * exactly uqs_replay_dev (scores_dev and queries_dev may then be NULL).  A query with flight outside [0, n_flights) or
 * frame outside [0, n_frames) returns UQS_ERR_BAD_ARG naming the first such index, before any grid is written (the
 * check synchronises).  Queries use the fixed origin of p (no recentering).  The engine, sub-tile geometry and time
 * slicing are chosen as for uqs_replay_dev; the resident engine's probe variant uses the default lane layout, so
 * uqs_set_fan_layout() and uqs_set_decode_warp() do not apply to this call.  Asynchronous on the current stream. */
int uqs_replay_frontier_dev(const uqs_params* p, int n_flights, int n_frames,
                            const float* x_dev, const float* y_dev, const float* yaw_dev, const float* ranges_dev,
                            int8_t* grids_dev, int accumulate,
                            int n_queries, const uqs_query* queries_dev, int32_t* scores_dev, uqs_stats* stats);
/* Host-buffer form (grids start at zero; grids_out may be NULL).  Synchronous. */
int uqs_replay_frontier(const uqs_params* p, int n_flights, int n_frames, const float* x, const float* y,
                        const float* yaw_deg, const float* ranges, int8_t* grids_out,
                        int n_queries, const uqs_query* queries, int32_t* scores_out, uqs_stats* stats);

/* N4: reader of scanlog.bin ("SCLOG2\n" + packed 569-byte scanrec_t records, uav_local_nav.c:1505,1522-1547).
 * Returns the number of qualifying records (> max_records means the buffers were too small), < 0 on error.
 * Records whose pose is NaN (:1559-1561) are skipped unless keep_nan_pose != 0.  Any output may be NULL. */
long uqs_scanlog_read(const char* path, int keep_nan_pose, long max_records, uint32_t* host_ms, uint32_t* scan_ms,
                      float* x_m, float* y_m, float* yaw_deg, float* alt_m, float* of_rate_x, float* of_rate_y,
                      uint8_t* of_q, uint8_t* kf_flags, uint8_t* grid_raw);
long uqs_scanlog_count(const char* path, int keep_nan_pose);

/* N4: reader of navlog.csv (header uav_local_nav.c:1489-1494, rows :1586-1625): 22 text columns per log tick,
 * "nan" for missing values, flights appended without further headers, a truncated last row is dropped.  Fills
 * the columns P0 and the mapper consume; any output may be NULL; t_ms keeps the low 32 bits of the 64-bit
 * millisecond clock.  Returns the number of well-formed rows in the file (call with max_rows = 0 to size the
 * buffers), -1 if the file cannot be opened. */
long uqs_navlog_read(const char* path, long max_rows, uint32_t* t_ms, float* yaw_deg, float* alt_m, float* x_m,
                     float* y_m, float* vx_mps, float* vy_mps, float* rf_m, uint8_t* of_q, float* of_rate_x,
                     float* of_rate_y, float* tof4);

/* ------------------------------------------------------------------------ */
/* Multi-GPU (SURVEY.md section 8(e))                                        */
/* ------------------------------------------------------------------------ */
/* Partitions -- host arithmetic only, usable without a device.
 *   uqs_flight_shard: contiguous block [first, first+count) of n_flights independent flights for `rank`
 *                     (configs 3 and 5: every GPU replays its own flights into its own grids; no collective).
 *   uqs_row_band:     rows [row0, row0+rows) of an H-row grid OWNED by `rank`, edges multiples of `align`
 *                     (config 4: occ_grid, uav_local_nav.c:188, split across GPUs.  The reference clamps after
 *                     every update, :259-260, so partial grids cannot be summed; owned bands are exact). */
void uqs_flight_shard(int n_flights, int rank, int world, int* first, int* count);
void uqs_row_band(int H, int rank, int world, int align, int* row0, int* rows);

/* (i) One process per GPU.  Rank 0 calls uqs_comm_unique_id(), the launcher broadcasts the 128 bytes by its own
 * means, every rank calls uqs_comm_init_rank() after uqs_init(local device) (ncclCommInitRank underneath;
 * NCCL is loaded at run time with dlopen, UQS_ERR_NO_NCCL if absent). */
#define UQS_COMM_ID_BYTES 128
int uqs_comm_unique_id(void* id128);
int uqs_comm_init_rank(const void* id128, int nranks, int rank);
int uqs_comm_destroy(void);
int uqs_comm_nranks(void);
int uqs_comm_rank(void);
int uqs_nccl_version(void);            /* e.g. 22809; 0 if NCCL cannot be loaded */
/* Where the banded replays cut the grid: 1 (default) = so that every rank gets the same share of the LOG -- a
 * histogram of the frames' origin rows widened by the sensor's reach, computed on the device from the log each
 * call (a sweep that covers the middle of a large grid would leave equal outer bands idle); 0 = equal bands
 * (uqs_row_band).  Every rank derives the same cuts from the same log; any cuts give identical bytes.
 * uqs_band_edges: edges_out[0..nranks] of the last banded replay, returns nranks. */
int uqs_set_band_balance(int on);
int uqs_balanced_row_bands_dev(const uqs_params* p, int n_frames, const float* x_dev, const float* y_dev,
                               int world, int* edges_out /* [world + 1] */);
int uqs_band_edges(int* edges_out);
/* Config 4 on this rank: replay this rank's owned row band of ONE W x H grid from a log that every rank holds
 * on its device, then (gather != 0) the path's single exchange: the disjoint bands are all-gathered over NCCL so
 * that every rank holds the whole grid.  grid_dev addresses the full W*H grid.  Asynchronous on the current
 * stream unless stats is given.  Without a communicator this is a whole-grid replay (1 rank). */
int uqs_replay_banded_dev(const uqs_params* p, int n_frames, const float* x_dev, const float* y_dev,
                          const float* yaw_dev, const float* ranges_dev, int8_t* grid_dev, int gather,
                          uqs_stats* stats);
/* Host-buffer form: every rank passes the same log; rank r uploads only slice r over PCIe, the slices are
 * all-gathered over NVLink, then as above with the gather; grid_out (NULL on ranks that do not want it)
 * receives the whole grid.  Synchronous. */
int uqs_replay_banded(const uqs_params* p, int n_frames, const float* x, const float* y, const float* yaw_deg,
                      const float* ranges, int8_t* grid_out, uqs_stats* stats);

/* (ii) One host thread driving N devices (what a plain C harness does; ncclCommInitAll underneath).
 * uqs_multi_init() creates one device context per GPU (devices == NULL: 0..n-1); uqs_multi_select(i) makes
 * context i current, after which EVERY single-device call of this header addresses device i (flight shards:
 * select, enqueue uqs_replay_dev on the shard, next device; then uqs_sync each).  uqs_multi_replay_banded() is
 * config 4 end to end from host buffers: slices up on N PCIe links, log all-gather, owned bands, band
 * all-gather, bands down on N links, nothing blocking between devices. */
int  uqs_multi_init(int n_devices, const int* devices);
int  uqs_multi_count(void);
int  uqs_multi_select(int i);
void uqs_multi_shutdown(void);
int  uqs_multi_replay_banded(const uqs_params* p, int n_frames, const float* x, const float* y,
                             const float* yaw_deg, const float* ranges, int8_t* grid_out, uqs_stats* stats);
const int8_t* uqs_multi_grid_dev(int i);   /* device i's copy of the whole grid after the call above */

/* Order-independent 64-bit digest of a grid: sum over cells i of splitmix64(i << 8 | (uint8)cell) mod 2^64.
 * Lets harnesses compare grids across GPUs / GPU counts without moving them.  _dev: n_grids device grids of
 * `cells` bytes each -> hashes_out[n_grids] (host), synchronises; uqs_grid_hash: one host grid, host arithmetic. */
int      uqs_grid_hashes_dev(const int8_t* grids_dev, int n_grids, size_t cells, uint64_t* hashes_out);
uint64_t uqs_grid_hash(const int8_t* grid, size_t cells);

/* Measurement knob: != 0 makes the host-buffer calls (uqs_replay, uqs_replay_flow[_mm]) run their copies and
 * synchronisation only, no kernels -- the copy floor bench.py reports beside the end-to-end time. */
int uqs_set_copy_only(int on);

/* Measured on-chip read-modify-write ceiling: every warp of a full grid does
 * conflict-free byte RMWs on its shared-memory sub-tile.  Returns updates/s. */
int uqs_measure_rmw_peak(double* updates_per_s);
/* The same pattern with one shared-memory ATOMIC per update (ATOMS.ADD on 32-bit words): what the "integer
 * log-odds atomics" of the original sketch would cost per update, clamp not included.  Returns updates/s. */
int uqs_measure_atoms_peak(double* updates_per_s);

/* ------------------------------------------------------------------------ */
/* (1) Drop-in symbols (replace uav_local_nav.c:188-192, 205-216, 229, 241-306) */
/* ------------------------------------------------------------------------ */

/* Must be called once before the drop-in symbols are used: allocates the
 * device grid and the pinned host mirror `occ_grid` for a W x H map.
 * (The reference's arrays are static; a shared library needs an allocator.) */
int  uqs_dropin_configure(const uqs_params* p);
/* Replaces `memset(occ_grid, 0, sizeof(occ_grid))` at uav_local_nav.c:2190
 * (sizeof of a pointer would silently be 8). */
void map_reset(void);
/* Make every update enqueued so far visible in occ_grid (host).  Called
 * implicitly by frontier_score_dir(); call it before reading occ_grid[]. */
void uqs_dropin_flush(void);
/* Push a caller-edited occ_grid[] back to the device copy (after direct host writes). */
int  uqs_dropin_upload(void);

extern int8_t*  occ_grid;            /* W*H int8, row-major, host-visible mirror   (:188) */
extern bool     map_inited;          /*                                            (:190) */
extern float    map_origin_x;        /*                                            (:191) */
extern float    map_origin_y;        /*                                            (:192) */
extern float    tof_beams_m[4][8];   /* written by the caller before each update   (:108) */
extern uint8_t  pending_kf_flags;    /* |= KF_MAP_RECENTER (1u<<5) on recenter     (:229) */

bool world_to_grid(float x, float y, int* gx, int* gy);                          /* :205 */
void raycast_update(float x0, float y0, float x1, float y1, bool hit_occ);       /* :241 */
void map_update_from_beams(float x_m, float y_m, float yaw_deg);                 /* :280 */
void map_recenter_shift(int sx_cells, int sy_cells);                             /* :308 */
void map_recentre_if_needed(float x_m, float y_m);                               /* :324 */
int  frontier_score_dir(float x_m, float y_m, float yaw_deg, float offset_deg);  /* :356 */

#ifdef __cplusplus
}
#endif
#endif /* UQS_MAPPING_H */
