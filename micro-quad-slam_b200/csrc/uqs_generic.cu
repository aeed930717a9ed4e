// uqs_generic.cu -- the unrestricted replay: map_update_from_beams()/raycast_update() (uav_local_nav.c:241-306)
// for the inputs the fast engines do not cover.
//
// The two fast engines (uqs_kernels.cu) rest on three assumptions: rays of at most kMaxRayCells cells (their
// divide-free Bresenham step), 0 inside [lo_min, lo_max] (untouched cells stay 0 and free-space steps need only the
// lower clamp), and -- when accumulating -- a start grid whose values already lie in [lo_min, lo_max].  The ABI
// accepts inputs outside all three (a 3 mm grid, an exotic clamp range, a caller-edited occ_grid).  Such calls are
// replayed here: one warp per flight walks frames, beams and cells in reference order on the grid in global memory
// (L2), lanes along the ray, integer division for the minor axis, both clamps after every update -- the reference's
// loop statement for statement, with no restriction on ray length or values.  It is slow by design (no shared-memory
// residency, one warp per flight); nothing on the benchmarked path takes it.
#include "uqs_host.h"

namespace uqs {

// PROBE: after the rays of frame f, the warp reads the flight's frontier probes of frame f from the grid.
template <bool PROBE>
__global__ void __launch_bounds__(128)
k_replay_generic(const __grid_constant__ DevParams p, int n_flights, int n_frames, const float* __restrict__ x,
                 const float* __restrict__ y, const float* __restrict__ yaw_deg, const float* __restrict__ ranges,
                 const uint8_t* __restrict__ kind, int8_t* __restrict__ grids, int row0, int rows,
                 unsigned long long* __restrict__ stats /* [4]: U, accepted, skipped, domain */, ProbeArgs Q) {
  const int flight = (int)((blockIdx.x * (long long)blockDim.x + threadIdx.x) >> 5);
  const int lane = threadIdx.x & 31;
  if (flight >= n_flights) return;
  int8_t* grid = grids + (size_t)flight * p.W * p.H;
  const size_t fbase = (size_t)flight * n_frames;
  unsigned long long cells = 0;
  unsigned accepted = 0, skipped = 0;
  int pb = 0, pe = 0, next_pf = 0x7fffffff;            // this flight's probes [pb, pe), frame of the next one
  if (PROBE) {
    pb = Q.start[flight];
    pe = Q.start[flight + 1];
    if (pb < pe) next_pf = Q.probes[pb].x;
  }
  for (int f = 0; f < n_frames; f++) {
    const size_t fi = fbase + f;
    const float px = x[fi], py = y[fi], third = yaw_deg[fi];
    const bool raw = kind != nullptr && kind[fi] == 1;              // one raycast_update(x0,y0,x1,y1,hit) (drop-in symbol)
    float ex = 0.f, ey = 0.f;
    bool hit = false;
    int st;
    if (!raw) {
      const float dist = p.ranges_u16 ? range_from_mm(reinterpret_cast<const uint16_t*>(ranges)[fi * 32 + lane]) : ranges[fi * 32 + lane];
      st = beam_endpoint(p, px, py, third, dist, lane, ex, ey, hit);
    } else {
      st = lane == 0 ? 1 : 0;
      ex = third;
      ey = ranges[fi * 32];
      hit = ranges[fi * 32 + 1] != 0.0f;
    }
    int gx0, gy0, gx1 = 0, gy1 = 0;
    const bool have_o = world_to_grid(p, px, py, gx0, gy0);                          // :243
    const bool ok = st > 0 && have_o && world_to_grid(p, ex, ey, gx1, gy1);          // :244
    if (ok) accepted++;
    else if (!(raw && lane != 0)) skipped++;
    unsigned todo = __ballot_sync(0xffffffffu, ok);
    while (todo) {                                                  // beams in (d, c) order, :286-287
      const int b = __ffs(todo) - 1;
      todo &= todo - 1;
      const int ax = __shfl_sync(0xffffffffu, gx1, b), ay = __shfl_sync(0xffffffffu, gy1, b);
      const bool bhit = __shfl_sync(0xffffffffu, hit ? 1 : 0, b) != 0;
      const int dx = ax - gx0, dy = ay - gy0;
      const int adx = abs(dx), ady = abs(dy);
      const bool xmaj = adx >= ady;
      const int m = xmaj ? adx : ady, n = xmaj ? ady : adx, h = m >> 1;
      const int sxs = dx >= 0 ? 1 : -1, sys = dy >= 0 ? 1 : -1;
      // cell k of the walk at :254-277 is (major0 + k, minor0 + floor((k*n + m/2)/m)) (DESIGN.md section 2;
      // k*n < 2^30 for grids up to 32766 cells, so 32-bit integer division is exact)
      for (int k = lane; k <= m; k += 32) {
        const int q = m ? (k * n + h) / m : 0;
        const int cx = gx0 + (xmaj ? k : q) * sxs, cy = gy0 + (xmaj ? q : k) * sys;
        if (cy >= row0 && cy < row0 + rows) {
          const size_t at = (size_t)cy * p.W + cx;
          const int delta = (k == m) ? (bhit ? p.lo_occ : p.end_nohit) : -p.lo_free;   // :258-268
          int v = (int)grid[at] + delta;
          v = v < p.lo_min ? p.lo_min : (v > p.lo_max ? p.lo_max : v);                 // clamp_lo, :199-203
          grid[at] = (int8_t)v;
        }
      }
      if (lane == 0) cells += (unsigned long long)m + 1ull;
      __syncwarp();                                                 // the next ray may revisit these cells
    }
    if (PROBE) {
      while (next_pf == f) {                                        // the taken probes are a prefix (frame order)
        const int i = pb + lane;
        const int4 pr = i < pe ? Q.probes[i] : make_int4(-1, 0, 0, 0);
        const bool take = pr.x == f;
        if (take) Q.values[pr.z] = (uint32_t)(int)grid[pr.y];
        pb += __popc(__ballot_sync(0xffffffffu, take));
        next_pf = pb < pe ? Q.probes[pb].x : 0x7fffffff;
      }
      __syncwarp();                                                 // frame f + 1 may write the cells just read
    }
  }
  const unsigned acc = __reduce_add_sync(0xffffffffu, accepted), skp = __reduce_add_sync(0xffffffffu, skipped);
  if (lane == 0) {
    atomicAdd(&stats[0], cells);
    atomicAdd(&stats[1], (unsigned long long)acc);
    atomicAdd(&stats[2], (unsigned long long)skp);
  }
}

// rows [row0, row0+rows) of every grid := 0
__global__ void k_zero_rows(int8_t* __restrict__ grids, int n_flights, int W, int H, int row0, int rows) {
  const size_t per = (size_t)W * rows;
  const size_t nth = (size_t)gridDim.x * blockDim.x;
  for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < per * n_flights; i += nth) {
    const size_t fl = i / per;
    grids[fl * W * H + (size_t)row0 * W + (i - fl * per)] = 0;
  }
}

// counts cells outside [lo_min, lo_max] in rows [row0, row0+rows) of every grid
__global__ void k_range_check(const int8_t* __restrict__ grids, int n_flights, int W, int H, int row0, int rows, int lo_min,
                              int lo_max, unsigned long long* __restrict__ bad) {
  const size_t per = (size_t)W * rows;
  const size_t nth = (size_t)gridDim.x * blockDim.x;
  unsigned mine = 0;
  for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < per * n_flights; i += nth) {
    const size_t fl = i / per;
    const int v = grids[fl * W * H + (size_t)row0 * W + (i - fl * per)];
    mine += (v < lo_min || v > lo_max) ? 1u : 0u;
  }
  mine = __reduce_add_sync(0xffffffffu, mine);
  if ((threadIdx.x & 31) == 0 && mine) atomicAdd(bad, (unsigned long long)mine);
}

// Order-independent 64-bit digest of a grid: sum over cells of splitmix64(index << 8 | byte).  Position-sensitive
// (a zero cell still contributes), trivially parallel, and the same formula in plain C (uqs_grid_hash) and numpy
// (tests): used to compare grids across GPUs / GPU counts without moving them.
__host__ __device__ inline unsigned long long mix64(unsigned long long z) {
  z += 0x9E3779B97F4A7C15ull;
  z = (z ^ (z >> 30)) * 0xBF58476D1CE4E5B9ull;
  z = (z ^ (z >> 27)) * 0x94D049BB133111EBull;
  return z ^ (z >> 31);
}

__global__ void __launch_bounds__(256)
k_grid_hash(const int8_t* __restrict__ grids, size_t cells, unsigned long long* __restrict__ out) {
  const int8_t* g = grids + (size_t)blockIdx.y * cells;
  unsigned long long h = 0;
  for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < cells; i += (size_t)gridDim.x * blockDim.x)
    h += mix64(((unsigned long long)i << 8) | (unsigned long long)(uint8_t)g[i]);
  for (int o = 16; o; o >>= 1) h += __shfl_xor_sync(0xffffffffu, h, o);
  if ((threadIdx.x & 31) == 0 && h) atomicAdd(&out[blockIdx.y], h);
}

cudaError_t grid_hash_launch(const int8_t* grids, int n_grids, size_t cells, unsigned long long* out, cudaStream_t st) {
  const unsigned bx = (unsigned)std::min<size_t>(std::max<size_t>((cells + 256 * 16 - 1) / (256 * 16), 1), 1024);
  for (int g0 = 0; g0 < n_grids; g0 += 65535) {
    const int ng = std::min(65535, n_grids - g0);
    k_grid_hash<<<dim3(bx, (unsigned)ng), 256, 0, st>>>(grids + (size_t)g0 * cells, cells, out + g0);
  }
  return cudaGetLastError();
}

static unsigned sweep_blocks(size_t items) {
  return (unsigned)std::min<size_t>(std::max<size_t>((items + 255) / 256, 1), (size_t)148 * 16);
}

cudaError_t generic_launch(const DevParams& dp, int n_flights, int n_frames, const float* x, const float* y, const float* yaw,
                           const float* ranges, const uint8_t* kind, int8_t* grids, int accumulate, int row0, int rows,
                           unsigned long long* stats, cudaStream_t st, const ProbeArgs* Q) {
  if (!accumulate) k_zero_rows<<<sweep_blocks((size_t)dp.W * rows * n_flights), 256, 0, st>>>(grids, n_flights, dp.W, dp.H, row0, rows);
  if (Q)
    k_replay_generic<true><<<(unsigned)((n_flights + 3) / 4), 128, 0, st>>>(dp, n_flights, n_frames, x, y, yaw, ranges, kind, grids,
                                                                           row0, rows, stats, *Q);
  else
    k_replay_generic<false><<<(unsigned)((n_flights + 3) / 4), 128, 0, st>>>(dp, n_flights, n_frames, x, y, yaw, ranges, kind, grids,
                                                                            row0, rows, stats, ProbeArgs{});
  return cudaGetLastError();
}

cudaError_t range_check_launch(const int8_t* grids, int n_flights, int W, int H, int row0, int rows, int lo_min, int lo_max,
                               unsigned long long* bad, cudaStream_t st) {
  k_range_check<<<sweep_blocks((size_t)W * rows * n_flights), 256, 0, st>>>(grids, n_flights, W, H, row0, rows, lo_min, lo_max, bad);
  return cudaGetLastError();
}

}  // namespace uqs

using namespace uqs;

extern "C" {

/* 64-bit digest of each of n_grids device grids of `cells` bytes -> hashes_out (host).  Synchronises. */
int uqs_grid_hashes_dev(const int8_t* grids_dev, int n_grids, size_t cells, uint64_t* hashes_out) {
  int rc = check_ready();
  if (rc) return rc;
  if (!grids_dev || n_grids <= 0 || !cells || !hashes_out) { set_error("uqs_grid_hashes_dev: bad argument"); return UQS_ERR_BAD_ARG; }
  cudaStream_t st = g_ctx.stream();
  if ((rc = g_ctx.in_kind.ensure((size_t)n_grids * 8))) return rc;
  cudaError_t e = zero_async(g_ctx.in_kind.p, (size_t)n_grids * 8, st);
  if (e == cudaSuccess) e = grid_hash_launch(grids_dev, n_grids, cells, (unsigned long long*)g_ctx.in_kind.p, st);
  if (e == cudaSuccess) e = cudaMemcpyAsync(hashes_out, g_ctx.in_kind.p, (size_t)n_grids * 8, cudaMemcpyDeviceToHost, st);
  if (e == cudaSuccess) e = cudaStreamSynchronize(st);
  if (e != cudaSuccess) return cuda_fail(e, "uqs_grid_hashes_dev");
  g_ctx.launches += 2 + (n_grids - 1) / 65535;
  return UQS_OK;
}

/* the same digest of a host grid, in plain host arithmetic (for harnesses that hold the grid in RAM) */
uint64_t uqs_grid_hash(const int8_t* grid, size_t cells) {
  unsigned long long h = 0;
  for (size_t i = 0; i < cells; i++) h += mix64(((unsigned long long)i << 8) | (unsigned long long)(uint8_t)grid[i]);
  return h;
}

}  // extern "C"
