// uqs_kernels.cuh -- kernel argument blocks and prototypes shared by the host layer.
#pragma once
#include "uqs_device.cuh"

namespace uqs {

constexpr int kReplayThreads = 256;               // 8 warps per CTA, each owning one sub-tile
constexpr int kReplayWarps = kReplayThreads / 32;
constexpr int kReplayQueueBytes = 64 * 12;         // per-warp candidate queue of k_replay_tiles (kQueueBytes)
constexpr int kDecSlotBytes = 32 * 32 + 16;       // one decoded frame in the resident engine's ring
constexpr int kDecSlotsMax = 4;                    // the ring holds min(warps per CTA, 4) frames
constexpr int kJobGroup = 64;                     // flights per scheduling group of the sub-tile engine

struct ReplayArgs {
  const uint4* frames;      // [n_flights][n_frames]
  const uint2* groups;      // [n_flights][groups_per_flight]  bbox of 32 consecutive frames
  const uint2* rays;        // [n_flights][n_frames][32]
  int8_t* grids;            // [n_flights][H][W]
  unsigned long long* job_counter;
  const uint32_t* tile_order;  // [nsx*nsy] sub-tile ids, heaviest first (nullptr = natural order)
  unsigned long long total_jobs;
  int n_flights, n_frames, groups_per_flight;
  int W, H;
  int row0, rows;           // rows of the grid this launch owns
  int sw, sh, nsx, nsy;     // sub-tile size and count per grid
  int pitch, tile_bytes;    // shared-memory row pitch (bytes, odd number of words) and tile size
  int pitch_cells;          // row pitch, in 32-bit cells, of a time-slice MAP tile (odd)
  int slices;               // time slices per log (1 = none); slice s > 0 produces clamp-add maps
  int groups_per_slice;     // 32-frame groups per slice
  uint32_t* maps;           // [n_flights][slices-1][H][W] maps of slices 1..S-1
  int lo_free, lo_occ, lo_min, lo_max, end_nohit;
  int accumulate;
};

// whole-grid-resident engine: one CTA per flight
struct FlightArgs {
  const uint4* frames;
  const uint2* rays;
  int8_t* grids;
  unsigned long long* job_counter;
  int n_flights, n_frames;
  const int4* boxes;        // per flight: resident cell range [x0,x1) x [y0,y1)
  int W, H, pitch;
  int max_rows;             // rows of the resident region (max over the launch's flights)
  int ring_size;            // bytes of collision table per warp (power of two), placed after the grid
  int lo_free, lo_occ, lo_min, lo_max, end_nohit;
  int accumulate;
};

// Frontier probes served inside a replay (uqs_frontier.cu): one cell a query's score reads, at the moment its owner
// has applied exactly the frames <= `frame`.  Sorted by (bucket, frame); bucket b holds [start[b], start[b+1]):
// per flight for the resident and unrestricted engines, per (flight, time slice, sub-tile) for the sub-tile engine.
struct ProbeArgs {
  const int4* probes;       // {frame, cell = gy*W + gx, slot, flight (launch-local)}
  const int* start;         // [n_buckets + 1]
  uint32_t* values;         // [slot]: the cell's value, or its 32-bit map word in a time-slice map tile
  int n_buckets;
};

// Recentering (uqs_next.cu).  One recenter event of a flight: the shift (sx, sy) applied before `frame` is mapped, the
// map origin after it (binary32, as uav_local_nav.c:346-347 leaves it) and S, the sum of every shift applied so far.
// A flight's cells are numbered in its global frame, global = window cell + S; the replay's grids hold global cells
// minus the flight's smallest S (s_min), so that they start at 0.
struct __align__(16) PlanEvent {
  int frame, sx, sy, pad;
  int Sx, Sy;
  float ox, oy;
};
// the index of a flight's last event at a frame <= f among its events [eb, ee) (frame order), eb - 1 when there is none
__device__ __forceinline__ int last_event_at(const PlanEvent* events, int eb, int ee, int f) {
  int lo = eb, hi = ee;                                 // first event of a frame > f
  while (lo < hi) {
    const int mid = (lo + hi) >> 1;
    if (events[mid].frame <= f) lo = mid + 1; else hi = mid;
  }
  return lo - 1;
}
struct RecenterArgs {
  const PlanEvent* events;  // every flight's events in frame order
  const int* ev_start;      // [n_flights + 1] (launch-local flights): flight f's events are [ev_start[f], ev_start[f+1])
  const int2* s_min;        // [n_flights] the flight's smallest S
  int W, H;                 // the window: the map the drone holds
};

struct ScanState;

__global__ void k_pose_increments(long long total, int n_samples, const uint32_t* t_ms,
                                  const float* rate_x, const float* rate_y, const float* h_m,
                                  const float* yaw_deg, const uint8_t* q, float deg2rad, float* inc_n,
                                  float* inc_e, unsigned long long* domain_errors);
__global__ void k_pose_chain(int n_flights, int n_samples, const float* inc_n, const float* inc_e,
                             float* xo, float* yo);
__global__ void k_pose_scan(int n_flights, int n_samples, int parts_per_flight, const float* inc_n,
                            const float* inc_e, float* xo, float* yo, volatile ScanState* state,
                            unsigned int* ticket);
int pose_scan_tile();
size_t pose_scan_state_bytes();
cudaError_t zero_async(void* p, size_t bytes, cudaStream_t st);   // zero fill by a kernel (never a copy engine)
int pose_scan_threads();

// k_ray_setup: the ray and frame records of a chunk of flights (grid = (groups per flight, flights))
cudaError_t ray_setup_launch(dim3 grid, cudaStream_t st, const DevParams& p, int n_frames, const float* x, const float* y,
                             const float* yaw_deg, const float* ranges, const uint8_t* kind, int want_k0,
                             const uint32_t* inv_table, uint4* frames, uint2* groups, uint2* rays, unsigned long long* stats);
// the same records from 256-thread blocks (8 warps x 4 frames), which fit beside the resident replay's CTAs on an SM
cudaError_t ray_setup256_launch(dim3 grid, cudaStream_t st, const DevParams& p, int n_frames, const float* x, const float* y,
                                const float* yaw_deg, const float* ranges, const uint8_t* kind, int want_k0,
                                const uint32_t* inv_table, uint4* frames, uint2* groups, uint2* rays, unsigned long long* stats);
// whether one k_ray_setup256 block fits on an SM beside `ctas` CTAs of the resident replay (nw, fan, prod) with `smem`
// dynamic bytes each: registers, shared memory, threads and block slots
cudaError_t setup256_fits_beside(int nw, int fan, int prod, size_t smem, int ctas, bool* fits);
// the same for recentred flights: each frame is set up against its flight's origin at that frame, and its records are
// in the flight's global frame (events, ev_start and s_min as in RecenterArgs)
cudaError_t ray_setup_recenter_launch(dim3 grid, cudaStream_t st, const DevParams& p, int n_frames, const float* x,
                                      const float* y, const float* yaw_deg, const float* ranges, const uint32_t* inv_table,
                                      uint4* frames, uint2* groups, uint2* rays, unsigned long long* stats,
                                      const PlanEvent* events, const int* ev_start, const int2* s_min);
__global__ void k_records_to_cells(long long n_frames, const uint4* frames, const uint2* rays,
                                   int32_t* cells, int32_t* origin);
__global__ void k_sincosf(size_t n, const float* a, float* s, float* c);
__global__ void k_world_to_grid_one(DevParams p, float wx, float wy, int* out);
// the sub-tile engine (k_replay_tiles), plain or serving probes
cudaError_t tiles_prepare(bool probe, size_t smem, int* ctas_per_sm);
cudaError_t tiles_launch(bool probe, unsigned grid, size_t smem, cudaStream_t st, const ReplayArgs& A, const ProbeArgs& Q);
// the sub-tile engine replaying recentred flights: tiles cover the flights' global frames (no time slices), plain or
// serving probes whose cells are in those global frames
cudaError_t tiles_recenter_prepare(bool probe, size_t smem, int* ctas_per_sm);
cudaError_t tiles_recenter_launch(bool probe, unsigned grid, size_t smem, cudaStream_t st, const ReplayArgs& A,
                                  const ProbeArgs& Q, const RecenterArgs& R);
__global__ void k_compose_slices(int8_t* grids, const uint32_t* maps, int n_flights, int W, int H, int S, int row0,
                                 int rows);
cudaError_t flights_probe_prepare(int nw, size_t smem, int* ctas_per_sm);
cudaError_t flights_probe_launch(int nw, unsigned grid, size_t smem, cudaStream_t st, const FlightArgs& A, const ProbeArgs& Q);
cudaError_t flight_boxes_launch(int n_flights, int groups_per_flight, const uint2* groups, int W, int H, int4* boxes,
                                int* dims, int* host_dims_dev, cudaStream_t st);
cudaError_t flights_prepare(int nw, int fan, int prod, size_t smem, int* ctas_per_sm);
cudaError_t flights_launch(int nw, int fan, int prod, unsigned grid, size_t smem, cudaStream_t st, const FlightArgs& A);
__global__ void k_rmw_peak(int tile_bytes, int iters, int lo_min, int* sink);
__global__ void k_atoms_peak(int tile_bytes, int iters, int* sink);
// uqs_next.cu
__global__ void k_recenter_decide_one(float res, float size_m, float ox, float oy, float x, float y, int* out);
__global__ void k_recenter_shift(const int8_t* src, int8_t* dst, int W, int H, int sx, int sy);
__global__ void k_frontier_scores(DevParams p, const int8_t* grid, int n, const float* x, const float* y,
                                  const float* yaw_deg, const float* offset_deg, int* scores,
                                  unsigned long long* domain_errors);

}  // namespace uqs
