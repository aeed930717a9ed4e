// uqs_api.cu -- host side of the C ABI declared in include/uqs_mapping.h (batch symbols).
//
// Plain C-callable functions; the library owns its CUDA stream and scratch buffers,
// callers own every buffer they pass.  No CPU implementation of the path exists in
// this library: without a usable CUDA device every call returns UQS_ERR_NO_DEVICE /
// UQS_ERR_NOT_INIT.
#include <algorithm>
#include <cmath>
#include <cstdarg>
#include <cstdio>
#include <cstring>
#include <vector>

#include "../../include/uqs_mapping.h"
#include "uqs_host.h"

namespace uqs {

static Context g_single;            // the context of uqs_init(); uqs_multi.cu owns the others
Context* g_cur = &g_single;

static char g_err[512] = "";

void set_error(const char* fmt, ...) {
  va_list ap;
  va_start(ap, fmt);
  vsnprintf(g_err, sizeof(g_err), fmt, ap);
  va_end(ap);
}

int cuda_fail(cudaError_t e, const char* what) {
  set_error("CUDA error in %s: %s", what, cudaGetErrorString(e));
  return UQS_ERR_CUDA;
}

int DevBuf::ensure(size_t bytes) {
  if (bytes <= cap) return UQS_OK;
  if (p) cudaFree(p);
  p = nullptr;
  cap = 0;
  size_t want = bytes + bytes / 8 + 256;
  cudaError_t e = cudaMalloc(&p, want);
  if (e != cudaSuccess) {
    cudaGetLastError();
    want = bytes;
    e = cudaMalloc(&p, want);
  }
  if (e != cudaSuccess) {
    p = nullptr;
    set_error("cudaMalloc(%zu) failed: %s", want, cudaGetErrorString(e));
    return UQS_ERR_NOMEM;
  }
  cap = want;
  return UQS_OK;
}

void DevBuf::release() {
  if (p) cudaFree(p);
  p = nullptr;
  cap = 0;
}

int check_ready() {
  if (!g_ctx.ready) {
    if (!g_err[0]) set_error("uqs_init() has not been called or failed");
    return UQS_ERR_NOT_INIT;
  }
  return UQS_OK;
}

int make_dev_params(const uqs_params* p, DevParams* d) {
  if (!p) { set_error("params is NULL"); return UQS_ERR_BAD_ARG; }
  if (p->W < 2 || p->H < 2 || p->W > 32766 || p->H > 32766) {
    set_error("grid size %dx%d outside [2, 32766]", p->W, p->H);
    return UQS_ERR_BAD_ARG;
  }
  if (!(p->res_m > 0.0f) || !std::isfinite(p->origin_x) || !std::isfinite(p->origin_y)) {
    set_error("res_m must be > 0 and the origin finite");
    return UQS_ERR_BAD_ARG;
  }
  if (p->lo_min < -128 || p->lo_max > 127 || p->lo_min > p->lo_max) {
    set_error("log-odds clamp [%d,%d] does not fit int8", p->lo_min, p->lo_max);
    return UQS_ERR_BAD_ARG;
  }
  if (p->lo_free < 0 || p->lo_free > 127 || p->lo_occ < 0 || p->lo_occ > 127) {
    set_error("log-odds steps must be in [0,127]");
    return UQS_ERR_BAD_ARG;
  }
  d->W = p->W; d->H = p->H; d->halfW = p->W / 2; d->halfH = p->H / 2;
  d->res = p->res_m; d->ox = p->origin_x; d->oy = p->origin_y;
  d->max_range = p->max_range_m; d->min_range = p->min_range_m;
  // the same binary32 operations the reference's compiler folds (uav_local_nav.c:284,292,299)
  volatile float mr = p->max_range_m, hm = p->hit_margin_m, fov = p->fov_deg;
  volatile float pi_f = (float)M_PI;
  d->hit_below = mr - hm;
  d->half_fov = fov * 0.5f;
  d->deg2rad = pi_f / 180.0f;
  for (int c = 0; c < 8; c++) {                       // (:295-296) one rounding per operator, like the reference
    volatile float cf = (float)c;
    volatile float u = (cf - 3.5f) / 3.5f;
    volatile float hf = d->half_fov;
    d->col_off[c] = u * hf;
  }
  d->lo_free = p->lo_free; d->lo_occ = p->lo_occ; d->lo_min = p->lo_min; d->lo_max = p->lo_max;
  d->end_nohit = -(p->lo_free / 2);
  d->ranges_u16 = 0;
  return UQS_OK;
}

// magic reciprocals of the closed-form Bresenham, built once per device (uqs_device.cuh: minor_steps)
int ensure_inv_table() {
  if (g_ctx.inv_table.p) return UQS_OK;
  std::vector<uint32_t> t(kMaxRayCells + 1);
  t[0] = 0;
  for (uint32_t m = 1; m <= (uint32_t)kMaxRayCells; m++) t[m] = (uint32_t)(((1ull << 31) + m - 1) / m);
  int rc = g_ctx.inv_table.ensure(t.size() * sizeof(uint32_t));
  if (rc) return rc;
  // on the stream the kernels run on (non-blocking streams are not ordered against the legacy stream), and
  // complete before the pageable source goes out of scope
  cudaError_t e = cudaMemcpyAsync(g_ctx.inv_table.p, t.data(), t.size() * sizeof(uint32_t), cudaMemcpyHostToDevice, g_ctx.stream());
  if (e == cudaSuccess) e = cudaStreamSynchronize(g_ctx.stream());
  if (e == cudaSuccess) e = cudaDeviceSynchronize();     // visible to every stream of the library (pipeline, caller's)
  if (e != cudaSuccess) { g_ctx.inv_table.release(); return cuda_fail(e, "inv table upload"); }
  return UQS_OK;
}

// sub-tile geometry for a grid of W columns and `rows` owned rows, aiming at `target`-cell sub-tiles
static void choose_tiles(int W, int rows, int target, int* sw, int* sh, int* nsx, int* nsy) {
  auto pick = [](int extent, int forced, int target, int* size, int* count) {
    if (forced > 0) {
      *size = std::min(forced, extent);
    } else {
      int n = std::max(1, (extent + target / 2) / target);
      int s = (extent + n - 1) / n;
      s = (s + 3) & ~3;
      *size = std::min(s, extent);
    }
    *count = (extent + *size - 1) / *size;
  };
  // measured on the 400x400 ensemble: 80 wide x 100 high beats 80x80 by ~4 % (fewer row crossings per ray
  // for the same number of resident warps); small (time-sliced) tiles stay square
  pick(W, g_ctx.tune_sw, target, sw, nsx);
  pick(rows, g_ctx.tune_sh, target >= 80 ? target + target / 4 : target, sh, nsy);
}

// zero fill by a kernel of ours (counted like every other launch)
static cudaError_t zero_counted(void* p, size_t bytes, cudaStream_t st) {
  g_ctx.launches += bytes ? 1 : 0;
  return zero_async(p, bytes, st);
}

// Sub-tile engine geometry and time slices of a replay of n_flights x n_frames over `rows` rows (replay_device; the
// recentering call asks it whether a call would be time-sliced)
void tile_geometry(const DevParams& dp, int n_flights, int n_frames, int rows, int* psw, int* psh, int* pnsx, int* pnsy,
                   int* pslices) {
  const int gpf = (n_frames + 31) / 32;
  // Sub-tile engine geometry.  With plenty of (flight, tile) jobs, ~80-cell tiles and no time slicing.
  // With few (one long log, one small flight) the chip would idle: cut the log into S time slices,
  // replayed concurrently as clamp-add maps on 40-cell tiles and composed afterwards (exact).
  int sw, sh, nsx, nsy, slices = 1;
  choose_tiles(dp.W, rows, 80, &sw, &sh, &nsx, &nsy);
  {
    const long long warp_slots = (long long)g_ctx.sm_count * 32;
    const long long jobs80 = (long long)n_flights * nsx * nsy;
    int want = g_ctx.tune_slices;
    int slice_tile = 40;
    const bool band = rows < dp.H;          // an owned row band of a grid shared between GPUs
    if (want == 0 && band && g_ctx.tune_sw == 0 && g_ctx.tune_sh == 0 && jobs80 < 2 * warp_slots) {
      // A band holds too few 80x100 tiles to balance the persistent warps, but time slices do not pay here: the band's
      // hot tiles already bound the launch (one warp per tile job, ~6 ms for a tile the sweep passes twice), and map
      // tiles cost 3x the instructions per update.  Measured per band of the 16384^2 sweep cut 8 / 4 / 2 ways
      // (tools/c4_band_tuning.py, profiles/r2_c4_band_tuning.log): 56-cell value tiles, no slices.
      choose_tiles(dp.W, rows, 56, &sw, &sh, &nsx, &nsy);
      want = 1;
    }
    if (want == 0 && jobs80 < 2 * warp_slots) {
      // largest map tile that still yields >= 8 jobs per warp slot at the finest admissible slicing (>= 256
      // frames per slice, <= 64 slices).  Measured: 56-cell tiles win for long rays (>= 200 cells: the one-hour
      // log at 1 cm), 40 for short ones (two more CTAs per SM matter more), smaller only when jobs are scarce.
      const int s_max = std::max(1, std::min(64, gpf / 8));
      const bool long_rays = dp.max_range >= 200.0f * dp.res;
      long long jobs_t = 1;
      for (int t : { 56, 40, 24, 16 }) {
        if (t == 56 && !long_rays) continue;
        int a, b, nx, ny;
        choose_tiles(dp.W, rows, t, &a, &b, &nx, &ny);
        slice_tile = t;
        jobs_t = (long long)n_flights * nx * ny;
        if (jobs_t * s_max >= 8 * warp_slots) break;
      }
      want = (int)std::min<long long>(s_max, std::max<long long>(1, (16 * warp_slots + jobs_t - 1) / jobs_t));
    }
    if (want > 1) {
      const size_t map_bytes = (size_t)dp.W * dp.H * 4;
      const size_t cap = ((size_t)6 << 30) / map_bytes;              // bound the map scratch
      want = (int)std::min<size_t>((size_t)want, std::max<size_t>(cap, 1) + 1);
    }
    if (want > 1) {
      slices = want;
      choose_tiles(dp.W, rows, slice_tile, &sw, &sh, &nsx, &nsy);
    }
  }
  const int pitch_cells = sw | 1;
  if (slices > 1 && g_ctx.tune_slices == 0 && ((size_t)pitch_cells * sh * 4 + kReplayQueueBytes) * kReplayWarps > 227u * 1024u)
    slices = 1;                                        // a forced large sub-tile leaves no room for 32-bit map cells
  *psw = sw; *psh = sh; *pnsx = nsx; *pnsy = nsy; *pslices = slices;
}

int replay_device(const DevParams& dp, int n_flights, int n_frames, const float* x, const float* y,
                  const float* yaw, const float* ranges, const uint8_t* kind, int8_t* grids,
                  int accumulate, int row0, int rows, bool reset_stats, const ProbeSet* probes) {
  cudaStream_t st = g_ctx.stream();
  const int gpf = (n_frames + 31) / 32;
  g_ctx.w->boxes_valid = false;                  // set again below once this call's touched boxes exist
  {
    const int rc0 = ensure_inv_table();
    if (rc0) return rc0;
  }
  // Inputs outside what the fast engines assume go to the unrestricted kernel (uqs_generic.cu): rays that can be
  // longer than kMaxRayCells cells, a clamp range that excludes 0, or -- when accumulating -- a start grid with
  // values outside [lo_min, lo_max] (checked on the device; the reference clamps such a cell on its next update).
  {
    const int side = std::max(dp.W, dp.H);
    const bool long_rays = side > kMaxRayCells + 1 && (kind != nullptr || !(dp.max_range / dp.res + 3.0f <= (float)kMaxRayCells));
    bool generic = g_ctx.engine == 3 || long_rays || dp.lo_min > 0 || dp.lo_max < 0;
    int rcg;
    if ((rcg = g_ctx.w->counters.ensure(64 * sizeof(unsigned long long)))) return rcg;
    unsigned long long* cnt = (unsigned long long*)g_ctx.w->counters.p;
    cudaError_t eg = cudaSuccess;
    if (!generic && accumulate) {
      unsigned long long bad = 0;
      eg = zero_counted(cnt + 40, sizeof(unsigned long long), st);
      if (eg == cudaSuccess) eg = range_check_launch(grids, n_flights, dp.W, dp.H, row0, rows, dp.lo_min, dp.lo_max, cnt + 40, st);
      if (eg == cudaSuccess) eg = cudaMemcpyAsync(&bad, cnt + 40, sizeof(bad), cudaMemcpyDeviceToHost, st);
      if (eg == cudaSuccess) eg = cudaStreamSynchronize(st);
      if (eg != cudaSuccess) return cuda_fail(eg, "start-grid range check");
      g_ctx.launches += 1;
      generic = bad != 0;
    }
    if (generic) {
      if (reset_stats) eg = zero_counted(cnt, 8 * sizeof(unsigned long long), st);
      if (eg != cudaSuccess) return cuda_fail(eg, "memset stats");
      ProbeArgs PA;
      if (probes && (rcg = probe_buckets(*probes, 0, n_flights, n_frames, dp.W, 0, 0, 0, 0, 0, 0, &PA))) return rcg;
      KernelTimer t_rep(2);
      eg = generic_launch(dp, n_flights, n_frames, x, y, yaw, ranges, kind, grids, accumulate, row0, rows, cnt, st, probes ? &PA : nullptr);
      t_rep.stop();
      if (eg != cudaSuccess) return cuda_fail(eg, "k_replay_generic launch");
      g_ctx.launches += accumulate ? 1 : 2;
      return UQS_OK;
    }
  }
  int sw, sh, nsx, nsy, slices;
  tile_geometry(dp, n_flights, n_frames, rows, &sw, &sh, &nsx, &nsy, &slices);
  int pitch = (sw + 3) & ~3;
  if (((pitch >> 2) & 1) == 0) pitch += 4;            // odd word pitch: column walks hit 32 banks
  const int pitch_cells = sw | 1;
  const int gps = (gpf + slices - 1) / slices;          // 32-frame groups per slice
  const int tile_bytes = slices > 1 ? std::max(pitch * sh, pitch_cells * sh * 4) : pitch * sh;
  size_t smem = (size_t)tile_bytes * kReplayWarps + (size_t)kReplayQueueBytes * kReplayWarps;   // tiles + candidate queues

  // Engine 2 keeps, per CTA, the bounding box of the cells one flight can touch resident in shared memory
  // (frame-synchronous, DESIGN.md section 3).  Whether it fits -- and how many CTAs share an SM -- is only known
  // after the ray set-up of a chunk (k_flight_boxes), so the choice is made per chunk below.
  // warps per resident CTA (measured): 4 when there are flights for every CTA slot of every SM -- per-frame
  // bookkeeping is paid per warp -- more warps per CTA when flights are scarce
  // (chunks of the host-buffer pipeline overlap on two streams and fill the chip together: 4 as well)
  const int nw = g_ctx.flight_warps ? g_ctx.flight_warps
                 : ((n_flights >= 4 * g_ctx.sm_count || g_ctx.chip_shared) ? 4 : (n_flights >= 2 * g_ctx.sm_count ? 8 : 16));
  const bool may_reside = g_ctx.engine != 1 && row0 == 0 && rows == dp.H;
  if (g_ctx.engine == 2 && !may_reside) {
    set_error("engine 2 (resident) cannot replay a row band");
    return UQS_ERR_BAD_ARG;
  }
  if (smem > 227u * 1024u) {
    set_error("sub-tile %dx%d needs %zu B of shared memory per CTA (> 227 KB)", sw, sh, smem);
    return UQS_ERR_BAD_ARG;
  }

  // scratch is bounded: flights are processed in chunks of at most `chunk` flights
  const size_t per_flight = (size_t)n_frames * (32 * sizeof(uint2) + sizeof(uint4)) + (size_t)gpf * sizeof(uint2);
  const size_t budget = g_ctx.scratch_budget;
  int chunk = (int)std::max<size_t>(1, std::min<size_t>((size_t)n_flights, budget / std::max<size_t>(per_flight, 1)));
  chunk = std::min(chunk, 65535);                       // flights are gridDim.y of the ray set-up
  int rc;
  if ((rc = g_ctx.w->rays.ensure((size_t)chunk * n_frames * 32 * sizeof(uint2)))) return rc;
  if ((rc = g_ctx.w->frames.ensure((size_t)chunk * n_frames * sizeof(uint4)))) return rc;
  if ((rc = g_ctx.w->groups.ensure((size_t)chunk * gpf * sizeof(uint2)))) return rc;
  if ((rc = g_ctx.w->counters.ensure(64 * sizeof(unsigned long long)))) return rc;
  unsigned long long* counters = (unsigned long long*)g_ctx.w->counters.p;   // [0..3] stats, [8], [9] job counters
  uint4* const frames = (uint4*)g_ctx.w->frames.p;
  uint2* const groups = (uint2*)g_ctx.w->groups.p;
  uint2* const rays = (uint2*)g_ctx.w->rays.p;
  cudaError_t e;
  if (reset_stats) {
    e = zero_counted(counters, 8 * sizeof(unsigned long long), st);
    if (e != cudaSuccess) return cuda_fail(e, "memset stats");
  }
  g_ctx.overlap_chunks = 0;

  int ctas_per_sm = 0;
  e = tiles_prepare(probes != nullptr, smem, &ctas_per_sm);
  if (e != cudaSuccess) return cuda_fail(e, "occupancy(k_replay_tiles)");
  if (ctas_per_sm < 1) { set_error("replay kernel does not fit on an SM (smem %zu)", smem); return UQS_ERR_CUDA; }
  if (may_reside && (rc = g_ctx.w->boxes.ensure((size_t)chunk * sizeof(int4)))) return rc;

  // The records of flight f0 + i of a chunk starting at flight f0 sit at record flight i: frames[i * n_frames ...],
  // groups[i * gpf ...], rays[i * n_frames * 32 ...], boxes[i].  Each lambda below takes the chunk-relative first
  // flight `lo` of the n flights it serves and the chunk's first flight f0.
  auto setup = [&](int f0, int lo, int n, cudaStream_t s, bool small) -> int {
    const size_t fo = (size_t)(f0 + lo) * n_frames, ro = (size_t)lo * n_frames;
    const float* r = dp.ranges_u16 ? reinterpret_cast<const float*>(reinterpret_cast<const uint16_t*>(ranges) + fo * 32) : ranges + fo * 32;
    KernelTimer t_setup(1, s);
    e = (small ? ray_setup256_launch : ray_setup_launch)(
        dim3((unsigned)gpf, (unsigned)n), s, dp, n_frames, x + fo, y + fo, yaw + fo, r, kind ? kind + fo : nullptr,
        may_reside ? 1 + g_ctx.k0_bias : 0, (const uint32_t*)g_ctx.inv_table.p, frames + ro, groups + (size_t)lo * gpf,
        rays + ro * 32, counters);
    t_setup.stop();
    if (e != cudaSuccess) return cuda_fail(e, "k_ray_setup launch");
    return UQS_OK;
  };

  // touched bounding box per flight -> shared memory per CTA -> CTAs per SM -> engine choice (after the set-up of
  // flights [lo, lo + n), which ran on s: synchronises s, the launch geometry of the replay depends on the boxes)
  struct Resident {
    int fnw = 0, ring_size = 256, f_ctas = 0, fpitch = 0, bh = 0;
    size_t fsmem = 0;
    bool resident = false;
  };
  auto configure = [&](int lo, int n, cudaStream_t s, Resident* R) -> int {
    int* d_dims = (int*)(counters + 32);
    if (!g_ctx.w->h_dims) {
      e = cudaHostAlloc((void**)&g_ctx.w->h_dims, 16, cudaHostAllocMapped);
      if (e != cudaSuccess) { g_ctx.w->h_dims = nullptr; return cuda_fail(e, "cudaHostAlloc(dims)"); }
    }
    int* h_dims_dev = nullptr;
    e = cudaHostGetDevicePointer((void**)&h_dims_dev, g_ctx.w->h_dims, 0);
    if (e == cudaSuccess) e = zero_counted(d_dims, 2 * sizeof(int), s);
    if (e == cudaSuccess)
      e = flight_boxes_launch(n, gpf, groups + (size_t)lo * gpf, dp.W, dp.H, (int4*)g_ctx.w->boxes.p + lo, d_dims, h_dims_dev, s);
    if (e == cudaSuccess) e = cudaStreamSynchronize(s);
    if (e != cudaSuccess) return cuda_fail(e, "k_flight_boxes");
    const int dims[2] = { g_ctx.w->h_dims[0], g_ctx.w->h_dims[1] };
    g_ctx.launches += 2;                                     // boxes, publish
    g_ctx.w->boxes_valid = n == n_flights;                   // one internal chunk: the boxes describe the whole call
    g_ctx.w->boxes_n = n; g_ctx.w->box_w = dims[0]; g_ctx.w->box_h = dims[1];
    const int bw = std::max(dims[0], 4), bh = std::max(dims[1], 1);
    int fpitch = (bw + 3) & ~3;
    if (((fpitch >> 2) & 1) == 0) fpitch += 4;
    if (g_ctx.pitch_mod >= 0)                                 // experiment knob: row pitch in words == pitch_mod (mod 32)
      while (((fpitch >> 2) & 31) != g_ctx.pitch_mod) fpitch += 4;
    const size_t region = (size_t)fpitch * bh;
    // Warps per resident CTA.  Measured over box sizes from 17 KB (8 CTAs per SM) to 173 KB (one): the kernel wants
    // >= 24 resident warps per SM from as few warps per CTA as possible (per-frame work is paid per warp), and never
    // more than 16 per CTA (a frame has ~80-400 steps to share out).  Few flights: more warps per CTA (nw_min).
    int ring_size = 256, f_ctas = 0, fnw = nw;
    size_t fsmem = 0;
    auto fit = [&](int w, int* ring, size_t* bytes, int* ctas) -> cudaError_t {
      *ring = 256;                                        // per-warp collision table (power of two)
      const size_t dec_bytes = (size_t)std::min(w, kDecSlotsMax) * kDecSlotBytes + 16;      // ring of decoded frames (+ alignment)
      while (*ring > 32 && region + (size_t)(*ring + 4) * w + dec_bytes > kFlightSmemMax) *ring >>= 1;
      *bytes = region + (size_t)(*ring + 4) * w + dec_bytes;         // + one spare word per warp
      *ctas = 0;
      return *bytes <= kFlightSmemMax ? flights_prepare(w, g_ctx.flight_fan, g_ctx.flight_prod, *bytes, ctas) : cudaSuccess;
    };
    if (g_ctx.flight_warps) {
      e = fit(fnw, &ring_size, &fsmem, &f_ctas);
    } else {
      e = cudaSuccess;
      for (int w : { 4, 8, 16 }) {
        if (w < nw) continue;                             // nw: the minimum the flight count asks for
        int r, c;
        size_t bts;
        if ((e = fit(w, &r, &bts, &c)) != cudaSuccess) break;
        if (c < 1) break;                                 // more warps only need more shared memory
        fnw = w; ring_size = r; fsmem = bts; f_ctas = c;
        if (c * w >= 24) break;
      }
    }
    if (e != cudaSuccess) return cuda_fail(e, "k_replay_flights attributes");
    if (g_ctx.engine == 2 && f_ctas < 1) {
      set_error("engine 2: the touched region %dx%d of a flight does not fit %zu B of shared memory", bw, bh, kFlightSmemMax);
      return UQS_ERR_BAD_ARG;
    }
    // auto: resident when the box fits and there are at least SMs/4 flights (measured crossover; with one CTA of
    // 16 warps per SM it still beats the sub-tile engine by 1.6x on the 668^2 and 800^2 grids of config 5);
    // otherwise the sub-tile engine (time-sliced when flights are few)
    // (a chunk of the host-buffer pipeline shares the chip with its neighbours: no flight-count condition there)
    // (round 2, tools/c5_shard_engines.py: with 128 flights -- a 1/8 shard of a config-5 resolution -- the resident engine
    // at 16 warps per CTA needs 1.8-2.8 ms against 3.3-6.9 ms for time-sliced sub-tiles on every geometry that fits; one
    // resident flight takes ~2 ms whatever the count, the sub-tile engine ~0.9 ms + 0.04 ms per flight: crossover ~30)
    const bool pipelined = g_ctx.chip_shared;               // other chunks of a host-buffer call share the chip
    R->resident = f_ctas >= 1 && (g_ctx.engine == 2 || n * 4 >= g_ctx.sm_count || pipelined);
    R->fnw = fnw; R->ring_size = ring_size; R->f_ctas = f_ctas; R->fpitch = fpitch; R->bh = bh; R->fsmem = fsmem;
    return UQS_OK;
  };

  // the resident replay of flights [lo, lo + n) on stream s with job counter jc
  auto replay_resident = [&](const Resident& R, int f0, int lo, int n, cudaStream_t s, unsigned long long* jc) -> int {
    FlightArgs FA;
    FA.frames = frames + (size_t)lo * n_frames;
    FA.rays = rays + (size_t)lo * n_frames * 32;
    FA.boxes = (const int4*)g_ctx.w->boxes.p + lo;
    FA.grids = grids + (size_t)(f0 + lo) * dp.W * dp.H;
    FA.job_counter = jc;
    FA.n_flights = n; FA.n_frames = n_frames;
    FA.W = dp.W; FA.H = dp.H; FA.pitch = R.fpitch; FA.max_rows = R.bh; FA.ring_size = R.ring_size;
    FA.lo_free = dp.lo_free; FA.lo_occ = dp.lo_occ; FA.lo_min = dp.lo_min; FA.lo_max = dp.lo_max;
    FA.end_nohit = dp.end_nohit;
    FA.accumulate = accumulate;
    e = zero_counted(FA.job_counter, sizeof(unsigned long long), s);
    // cells outside a flight's box are never touched: they are zero in a fresh replay
    if (e == cudaSuccess && !accumulate) e = zero_counted(FA.grids, (size_t)n * dp.W * dp.H, s);
    if (e != cudaSuccess) return cuda_fail(e, "memset before k_replay_flights");
    if (probes) {
      int p_ctas = 0;
      ProbeArgs PA;
      if ((rc = probe_buckets(*probes, f0 + lo, n, n_frames, dp.W, 0, 0, 0, 0, 0, 0, &PA))) return rc;
      if ((e = flights_probe_prepare(R.fnw, R.fsmem, &p_ctas)) != cudaSuccess) return cuda_fail(e, "k_replay_flights (probes) attributes");
      if (p_ctas < 1) { set_error("resident engine (probes): %zu B of shared memory do not fit an SM", R.fsmem); return UQS_ERR_CUDA; }
      KernelTimer t_rep(2, s);
      e = flights_probe_launch(R.fnw, (unsigned)std::min<long long>(n, (long long)p_ctas * g_ctx.sm_count), R.fsmem, s, FA, PA);
      t_rep.stop();
      if (e != cudaSuccess) return cuda_fail(e, "k_replay_flights (probes) launch");
      g_ctx.launches += 2;
      return UQS_OK;
    }
    const unsigned fgrid = (unsigned)std::min<long long>(n, (long long)R.f_ctas * g_ctx.sm_count);
    KernelTimer t_rep(2, s);
    e = flights_launch(R.fnw, g_ctx.flight_fan, g_ctx.flight_prod, fgrid, R.fsmem, s, FA);
    t_rep.stop();
    if (e != cudaSuccess) return cuda_fail(e, "k_replay_flights launch");
    g_ctx.launches += 2;
    return UQS_OK;
  };

  // the sub-tile replay of flights [lo, lo + n) on the library stream
  auto replay_tiles = [&](int f0, int lo, int n) -> int {
    // sub-tiles nearest the grid centre first (trajectories stay within 60 % of the half-extent,
    // so those are the heavy ones); cached per geometry
    if (g_ctx.w->order_nsx != nsx || g_ctx.w->order_nsy != nsy) {
      std::vector<uint32_t> ord((size_t)nsx * nsy);
      for (uint32_t i = 0; i < ord.size(); i++) ord[i] = i;
      auto dist2 = [&](uint32_t t) {
        const double cx = ((t % nsx) + 0.5) * sw - dp.W * 0.5, cy = ((t / nsx) + 0.5) * sh + row0 - dp.H * 0.5;
        return cx * cx + cy * cy;
      };
      std::stable_sort(ord.begin(), ord.end(), [&](uint32_t a, uint32_t b) { return dist2(a) < dist2(b); });
      if ((rc = g_ctx.w->order.ensure(ord.size() * sizeof(uint32_t)))) return rc;
      e = cudaMemcpyAsync(g_ctx.w->order.p, ord.data(), ord.size() * sizeof(uint32_t), cudaMemcpyHostToDevice, st);
      if (e == cudaSuccess) e = cudaStreamSynchronize(st);       // ord is a local
      if (e != cudaSuccess) return cuda_fail(e, "tile order upload");
      g_ctx.w->order_nsx = nsx;
      g_ctx.w->order_nsy = nsy;
    }
    ReplayArgs A;
    A.tile_order = (const uint32_t*)g_ctx.w->order.p;
    A.n_flights = n;
    A.frames = frames + (size_t)lo * n_frames;
    A.groups = groups + (size_t)lo * gpf;
    A.rays = rays + (size_t)lo * n_frames * 32;
    A.grids = grids + (size_t)(f0 + lo) * dp.W * dp.H;
    A.job_counter = counters + 8;
    A.total_jobs = (unsigned long long)n * nsx * nsy * slices;
    A.slices = slices; A.groups_per_slice = gps; A.pitch_cells = pitch_cells;
    A.maps = nullptr;
    if (slices > 1) {
      if ((rc = g_ctx.w->maps.ensure((size_t)n * (slices - 1) * dp.W * dp.H * sizeof(uint32_t)))) return rc;
      A.maps = (uint32_t*)g_ctx.w->maps.p;
    }
    A.n_frames = n_frames; A.groups_per_flight = gpf;
    A.W = dp.W; A.H = dp.H; A.row0 = row0; A.rows = rows;
    A.sw = sw; A.sh = sh; A.nsx = nsx; A.nsy = nsy;
    A.pitch = pitch; A.tile_bytes = tile_bytes;
    A.lo_free = dp.lo_free; A.lo_occ = dp.lo_occ; A.lo_min = dp.lo_min; A.lo_max = dp.lo_max;
    A.end_nohit = dp.end_nohit;
    A.accumulate = accumulate;
    e = zero_counted(A.job_counter, sizeof(unsigned long long), st);
    if (e != cudaSuccess) return cuda_fail(e, "memset job counter");
    unsigned long long want = (A.total_jobs + kReplayWarps - 1) / kReplayWarps;
    unsigned grid = (unsigned)std::min<unsigned long long>(want, (unsigned long long)ctas_per_sm * g_ctx.sm_count);
    ProbeArgs PA;
    if (probes && (rc = probe_buckets(*probes, f0 + lo, n, n_frames, dp.W, slices, gps, sw, sh, nsx, nsy, &PA))) return rc;
    KernelTimer t_rep(2);
    e = tiles_launch(probes != nullptr, grid, smem, st, A, probes ? PA : ProbeArgs{});
    if (e == cudaSuccess && probes && slices > 1 &&     // before slice 0's values are overwritten
        (rc = probe_resolve_slices(PA, (int)probes->slots(), A.grids, A.maps, dp.W, dp.H, slices, gps)))
      return rc;
    if (e == cudaSuccess && slices > 1) {
      const size_t cells = (size_t)dp.W * rows * n;
      k_compose_slices<<<(unsigned)((cells + 255) / 256), 256, 0, st>>>(A.grids, A.maps, n, dp.W, dp.H, slices, row0, rows);
      e = cudaGetLastError();
      g_ctx.launches += 1;
    }
    t_rep.stop();
    if (e != cudaSuccess) return cuda_fail(e, "k_replay_tiles launch");
    g_ctx.launches += 2;
    return UQS_OK;
  };

  // Overlapped schedule (resident engine, no probes): the set-up of chunk k + 1 runs, in 256-thread blocks on a
  // low-priority stream, in the SM resources and issue slots the replay of chunk k leaves over; the replays alternate
  // between two high-priority streams, so that the next one fills the SMs as the previous one's CTAs drain.  The first
  // chunk is about one wave of resident CTAs (its set-up is the only one exposed), the later ones `setup_overlap` waves
  // (the last one up to twice that: a fraction of a wave replayed on its own would end on a ragged tail).  Measured on
  // a B200 (profiles/r3_setup_overlap_ab.log): calls with less than one such later chunk lose more than they hide.
  const bool overlap = g_ctx.setup_overlap > 0 && may_reside && !probes && !g_ctx.chip_shared;
  // four CTAs per SM, before any box is known: the wave of config 3's resident replay (4 CTAs of 8 warps)
  const int wave0 = g_ctx.sm_count * 4;

  for (int f0 = 0; f0 < n_flights; f0 += chunk) {
    const int nf = std::min(chunk, n_flights - f0);
    int done = 0;                                            // flights of this chunk set up so far
    if (overlap && nf > wave0) {
      Resident R;
      if ((rc = setup(f0, 0, wave0, st, false)) || (rc = configure(0, wave0, st, &R))) return rc;
      done = wave0;
      bool fits = false;
      if (R.resident && (e = setup256_fits_beside(R.fnw, g_ctx.flight_fan, g_ctx.flight_prod, R.fsmem, R.f_ctas, &fits)) != cudaSuccess)
        return cuda_fail(e, "k_ray_setup256 attributes");
      const long long later = (long long)g_ctx.setup_overlap * R.f_ctas * g_ctx.sm_count;
      if (fits && nf - wave0 >= later) {
        if (!g_ctx.aux_setup) {
          int lo_pri = 0, hi_pri = 0;
          e = cudaDeviceGetStreamPriorityRange(&lo_pri, &hi_pri);
          if (e == cudaSuccess) e = cudaStreamCreateWithPriority(&g_ctx.aux_setup, cudaStreamNonBlocking, lo_pri);
          if (e == cudaSuccess) e = cudaStreamCreateWithPriority(&g_ctx.aux_replay[0], cudaStreamNonBlocking, hi_pri);
          if (e == cudaSuccess) e = cudaStreamCreateWithPriority(&g_ctx.aux_replay[1], cudaStreamNonBlocking, hi_pri);
          if (e == cudaSuccess) e = cudaEventCreateWithFlags(&g_ctx.aux_ev, cudaEventDisableTiming);
          if (e != cudaSuccess) return cuda_fail(e, "set-up overlap streams");
        }
        cudaStream_t ss = g_ctx.aux_setup, *rs = g_ctx.aux_replay;
        // every internal stream starts after the library stream's work so far (inputs, zeroed stats)
        e = cudaEventRecord(g_ctx.aux_ev, st);
        for (cudaStream_t s : { ss, rs[0], rs[1] })
          if (e == cudaSuccess) e = cudaStreamWaitEvent(s, g_ctx.aux_ev, 0);
        if (e != cudaSuccess) return cuda_fail(e, "set-up overlap join");
        if ((rc = replay_resident(R, f0, 0, wave0, rs[0], counters + 8))) return rc;
        int box_w = g_ctx.w->box_w, box_h = g_ctx.w->box_h;       // the boxes of the chunk's flights, all of them
        for (int lo = wave0, k = 1, n = 0; lo < nf; lo += n, k++) {
          n = nf - lo < 2 * later ? nf - lo : (int)later;
          if ((rc = setup(f0, lo, n, ss, true)) || (rc = configure(lo, n, ss, &R))) return rc;
          box_w = std::max(box_w, g_ctx.w->box_w); box_h = std::max(box_h, g_ctx.w->box_h);
          g_ctx.overlap_chunks += 1;
          if (R.resident) {
            if ((rc = replay_resident(R, f0, lo, n, rs[k & 1], counters + 8 + (k & 1)))) return rc;
          } else {
            // a chunk whose boxes do not fit: the sub-tile engine, after both replay streams
            for (int i = 0; i < 2 && e == cudaSuccess; i++)
              if ((e = cudaEventRecord(g_ctx.aux_ev, rs[i])) == cudaSuccess) e = cudaStreamWaitEvent(st, g_ctx.aux_ev, 0);
            if (e != cudaSuccess) return cuda_fail(e, "set-up overlap join");
            if ((rc = replay_tiles(f0, lo, n))) return rc;
            for (int i = 0; i < 2 && e == cudaSuccess; i++)
              if ((e = cudaEventRecord(g_ctx.aux_ev, st)) == cudaSuccess) e = cudaStreamWaitEvent(rs[i], g_ctx.aux_ev, 0);
            if (e != cudaSuccess) return cuda_fail(e, "set-up overlap join");
          }
        }
        // the library stream (and so any event the caller records on it) covers all of the call's work
        for (cudaStream_t s : { ss, rs[0], rs[1] })
          if (e == cudaSuccess && (e = cudaEventRecord(g_ctx.aux_ev, s)) == cudaSuccess) e = cudaStreamWaitEvent(st, g_ctx.aux_ev, 0);
        if (e != cudaSuccess) return cuda_fail(e, "set-up overlap join");
        g_ctx.w->boxes_valid = nf == n_flights;
        g_ctx.w->boxes_n = nf; g_ctx.w->box_w = box_w; g_ctx.w->box_h = box_h;
        continue;
      }
      // no room beside the replay's CTAs: the serial schedule, the rest of the chunk set up behind the first wave
    }
    if ((rc = setup(f0, done, nf - done, st, false))) return rc;
    if (may_reside) {
      Resident R;
      if ((rc = configure(0, nf, st, &R))) return rc;
      if (R.resident) {
        if ((rc = replay_resident(R, f0, 0, nf, st, counters + 8))) return rc;
        continue;
      }
    }
    if ((rc = replay_tiles(f0, 0, nf))) return rc;
  }
  return UQS_OK;
}

// Recentred flights through the sub-tile engine (uqs_replay_recentering_dev, route A): the ray set-up places every
// frame's records in its flight's global frame, and the sub-tiles cover the largest global extent gw x gh of the call.
// Grids start at zero; stats are reset.  The caller has checked that the inputs suit the sub-tile engine.  probes: cells
// in each flight's global frame (gw wide), served by the (flight, sub-tile) that owns them.
int replay_device_recentering(const DevParams& dp, int n_flights, int n_frames, const float* x, const float* y,
                              const float* yaw, const float* ranges, int8_t* grids, const PlanEvent* events,
                              const int* ev_start, const int2* s_min, int gw, int gh, const ProbeSet* probes) {
  cudaStream_t st = g_ctx.stream();
  const int gpf = (n_frames + 31) / 32;
  g_ctx.w->boxes_valid = false;
  int rc;
  if ((rc = ensure_inv_table())) return rc;
  int sw, sh, nsx, nsy;
  choose_tiles(gw, gh, 80, &sw, &sh, &nsx, &nsy);
  int pitch = (sw + 3) & ~3;
  if (((pitch >> 2) & 1) == 0) pitch += 4;
  const size_t smem = ((size_t)pitch * sh + kReplayQueueBytes) * kReplayWarps;
  if (smem > 227u * 1024u) {
    set_error("sub-tile %dx%d needs %zu B of shared memory per CTA (> 227 KB)", sw, sh, smem);
    return UQS_ERR_BAD_ARG;
  }
  const size_t per_flight = (size_t)n_frames * (32 * sizeof(uint2) + sizeof(uint4)) + (size_t)gpf * sizeof(uint2);
  int chunk = (int)std::max<size_t>(1, std::min<size_t>((size_t)n_flights, g_ctx.scratch_budget / std::max<size_t>(per_flight, 1)));
  chunk = std::min(chunk, 65535);                       // flights are gridDim.y of the ray set-up
  if ((rc = g_ctx.w->rays.ensure((size_t)chunk * n_frames * 32 * sizeof(uint2))) ||
      (rc = g_ctx.w->frames.ensure((size_t)chunk * n_frames * sizeof(uint4))) ||
      (rc = g_ctx.w->groups.ensure((size_t)chunk * gpf * sizeof(uint2))) ||
      (rc = g_ctx.w->counters.ensure(64 * sizeof(unsigned long long))))
    return rc;
  unsigned long long* counters = (unsigned long long*)g_ctx.w->counters.p;
  cudaError_t e = zero_counted(counters, 8 * sizeof(unsigned long long), st);
  if (e == cudaSuccess) e = zero_counted(grids, (size_t)n_flights * dp.W * dp.H, st);   // cells no sub-tile writes read 0
  if (e != cudaSuccess) return cuda_fail(e, "memset before the recentering replay");
  int ctas_per_sm = 0;
  if ((e = tiles_recenter_prepare(probes != nullptr, smem, &ctas_per_sm)) != cudaSuccess) return cuda_fail(e, "occupancy(k_replay_tiles)");
  if (ctas_per_sm < 1) { set_error("replay kernel does not fit on an SM (smem %zu)", smem); return UQS_ERR_CUDA; }
  for (int f0 = 0; f0 < n_flights; f0 += chunk) {
    const int nf = std::min(chunk, n_flights - f0);
    const size_t fo = (size_t)f0 * n_frames;
    KernelTimer t_setup(1);
    e = ray_setup_recenter_launch(dim3((unsigned)gpf, (unsigned)nf), st, dp, n_frames, x + fo, y + fo, yaw + fo, ranges + fo * 32,
                                  (const uint32_t*)g_ctx.inv_table.p, (uint4*)g_ctx.w->frames.p, (uint2*)g_ctx.w->groups.p,
                                  (uint2*)g_ctx.w->rays.p, counters, events, ev_start + f0, s_min + f0);
    t_setup.stop();
    if (e != cudaSuccess) return cuda_fail(e, "k_ray_setup launch");
    ReplayArgs A = {};
    A.tile_order = nullptr;
    A.n_flights = nf;
    A.frames = (const uint4*)g_ctx.w->frames.p;
    A.groups = (const uint2*)g_ctx.w->groups.p;
    A.rays = (const uint2*)g_ctx.w->rays.p;
    A.grids = grids + (size_t)f0 * dp.W * dp.H;
    A.job_counter = counters + 8;
    A.total_jobs = (unsigned long long)nf * nsx * nsy;
    A.slices = 1; A.groups_per_slice = gpf; A.pitch_cells = sw | 1;
    A.maps = nullptr;
    A.n_frames = n_frames; A.groups_per_flight = gpf;
    A.W = gw; A.H = gh; A.row0 = 0; A.rows = gh;
    A.sw = sw; A.sh = sh; A.nsx = nsx; A.nsy = nsy;
    A.pitch = pitch; A.tile_bytes = pitch * sh;
    A.lo_free = dp.lo_free; A.lo_occ = dp.lo_occ; A.lo_min = dp.lo_min; A.lo_max = dp.lo_max;
    A.end_nohit = dp.end_nohit;
    A.accumulate = 0;
    RecenterArgs R;
    R.events = events; R.ev_start = ev_start + f0; R.s_min = s_min + f0;
    R.W = dp.W; R.H = dp.H;
    e = zero_counted(A.job_counter, sizeof(unsigned long long), st);
    if (e != cudaSuccess) return cuda_fail(e, "memset job counter");
    const unsigned long long want = (A.total_jobs + kReplayWarps - 1) / kReplayWarps;
    const unsigned grid = (unsigned)std::min<unsigned long long>(want, (unsigned long long)ctas_per_sm * g_ctx.sm_count);
    ProbeArgs PA;
    if (probes && (rc = probe_buckets(*probes, f0, nf, n_frames, gw, 1, gpf, sw, sh, nsx, nsy, &PA))) return rc;
    KernelTimer t_rep(2);
    e = tiles_recenter_launch(probes != nullptr, grid, smem, st, A, probes ? PA : ProbeArgs{}, R);
    t_rep.stop();
    if (e != cudaSuccess) return cuda_fail(e, "k_replay_tiles launch");
    g_ctx.launches += 2;
  }
  return UQS_OK;
}

// counters of every Work in `mask` (bit i = works[i]) summed; synchronises their streams
int fetch_stats_mask(uqs_stats* stats, uint64_t frames, unsigned mask) {
  if (!stats) return UQS_OK;
  unsigned long long tot[4] = { 0, 0, 0, 0 };
  for (int i = 0; i < 3; i++) {
    if (!(mask & (1u << i)) || !g_ctx.works[i].counters.p) continue;
    Work* saved = g_ctx.w;
    g_ctx.w = &g_ctx.works[i];
    cudaStream_t st = g_ctx.stream();
    g_ctx.w = saved;
    unsigned long long h[4];
    cudaError_t e = cudaMemcpyAsync(h, g_ctx.works[i].counters.p, sizeof(h), cudaMemcpyDeviceToHost, st);
    if (e != cudaSuccess) return cuda_fail(e, "stats D2H");
    e = cudaStreamSynchronize(st);
    if (e != cudaSuccess) return cuda_fail(e, "stats sync");
    for (int k = 0; k < 4; k++) tot[k] += h[k];
  }
  stats->ray_cell_updates = tot[0];
  stats->rays_accepted = tot[1];
  stats->rays_skipped = tot[2];
  stats->domain_errors = tot[3];
  stats->frames = frames;
  if (tot[3]) {
    set_error("%llu rays longer than %d cells reached a fast engine (internal routing error)", tot[3], kMaxRayCells);
    return UQS_ERR_DOMAIN;
  }
  return UQS_OK;
}

int fetch_stats(uqs_stats* stats, uint64_t frames) { return fetch_stats_mask(stats, frames, 1u); }

int pose_device(int n_flights, int n_samples, const uint32_t* t_ms, const float* rx, const float* ry,
                const float* h, const float* yaw, const uint8_t* q, float* xo, float* yo, int mode) {
  cudaStream_t st = g_ctx.stream();
  const long long total = (long long)n_flights * n_samples;
  int rc;
  if ((rc = g_ctx.w->inc.ensure((size_t)total * 2 * sizeof(float)))) return rc;
  if ((rc = g_ctx.w->counters.ensure(64 * sizeof(unsigned long long)))) return rc;
  float* inc_n = (float*)g_ctx.w->inc.p;
  float* inc_e = inc_n + total;
  unsigned long long* dom = nullptr;        // no input is out of P0's domain any more (sincosf covers every float)
  cudaError_t e = cudaSuccess;
  volatile float pi_f = (float)M_PI;
  const float deg2rad = pi_f / 180.0f;
  KernelTimer t_pose(0);
  k_pose_increments<<<(unsigned)((total + 255) / 256), 256, 0, st>>>(total, n_samples, t_ms, rx, ry, h, yaw, q,
                                                                     deg2rad, inc_n, inc_e, dom);
  e = cudaGetLastError();
  if (e != cudaSuccess) return cuda_fail(e, "k_pose_increments launch");
  if (mode == 0) {
    const int warps_per_block = 4;               // kChainWarps of k_pose_chain
    k_pose_chain<<<(unsigned)((n_flights + warps_per_block - 1) / warps_per_block), warps_per_block * 32, 0, st>>>(
        n_flights, n_samples, inc_n, inc_e, xo, yo);
  } else {
    const int tile = pose_scan_tile();
    const int ppf = (n_samples + tile - 1) / tile;
    const size_t nparts = (size_t)n_flights * ppf;
    if ((rc = g_ctx.w->scan.ensure(nparts * pose_scan_state_bytes() + 64))) return rc;
    e = cudaMemsetAsync(g_ctx.w->scan.p, 0, nparts * pose_scan_state_bytes() + 64, st);
    if (e != cudaSuccess) return cuda_fail(e, "memset scan state");
    unsigned int* ticket = (unsigned int*)((char*)g_ctx.w->scan.p + nparts * pose_scan_state_bytes());
    k_pose_scan<<<(unsigned)nparts, pose_scan_threads(), 0, st>>>(n_flights, n_samples, ppf, inc_n, inc_e, xo, yo,
                                                                  (volatile ScanState*)g_ctx.w->scan.p, ticket);
  }
  e = cudaGetLastError();
  t_pose.stop();
  if (e != cudaSuccess) return cuda_fail(e, "pose kernel launch");
  g_ctx.launches += 2;
  return UQS_OK;
}

void context_select_single() {
  g_cur = &g_single;
  if (g_single.ready) cudaSetDevice(g_single.device);
}

int context_init(Context& c, int device) {
  int n = 0;
  cudaError_t e = cudaGetDeviceCount(&n);
  if (e != cudaSuccess || n <= 0) {
    cudaGetLastError();
    set_error("no CUDA device available (%s); this library has no CPU fallback",
              e != cudaSuccess ? cudaGetErrorString(e) : "device count is 0");
    c.ready = false;
    return UQS_ERR_NO_DEVICE;
  }
  if (device < 0 || device >= n) { set_error("device %d out of range (0..%d)", device, n - 1); return UQS_ERR_BAD_ARG; }
  if ((e = cudaSetDevice(device)) != cudaSuccess) return cuda_fail(e, "cudaSetDevice");
  cudaDeviceProp prop;
  if ((e = cudaGetDeviceProperties(&prop, device)) != cudaSuccess) return cuda_fail(e, "cudaGetDeviceProperties");
  if (prop.major < 10) {
    set_error("device %d is sm_%d%d; this library is built for sm_100a only", device, prop.major, prop.minor);
    return UQS_ERR_NO_DEVICE;
  }
  if ((e = cudaStreamCreateWithFlags(&c.own_stream, cudaStreamNonBlocking)) != cudaSuccess)
    return cuda_fail(e, "cudaStreamCreate");
  c.device = device;
  c.sm_count = prop.multiProcessorCount;
  c.ext_stream = nullptr;
  c.use_ext = false;
  c.ready = true;
  g_err[0] = 0;
  return UQS_OK;
}

// the caller makes `c` current first (the release helpers act on the current context)
void context_shutdown(Context& c) {
  if (!c.ready) return;
  cudaSetDevice(c.device);
  cudaDeviceSynchronize();
  comm_release();
  dropin_release();
  pipeline_release();
  c.release_all();
  if (c.own_stream) cudaStreamDestroy(c.own_stream);
  c.own_stream = nullptr;
  for (cudaStream_t* s : { &c.aux_setup, &c.aux_replay[0], &c.aux_replay[1] }) {
    if (*s) cudaStreamDestroy(*s);
    *s = nullptr;
  }
  if (c.aux_ev) cudaEventDestroy(c.aux_ev);
  c.aux_ev = nullptr;
  c.ready = false;
}

}  // namespace uqs

using namespace uqs;

extern "C" {

void uqs_params_default(uqs_params* p) {
  if (!p) return;
  p->W = 500; p->H = 500; p->res_m = 0.10f; p->size_m = 50.0f;      /* uav_local_nav.c:182-186 */
  p->origin_x = 0.0f; p->origin_y = 0.0f;
  p->max_range_m = 4.00f; p->fov_deg = 63.0f;                        /* :117-118 */
  p->min_range_m = 0.05f; p->hit_margin_m = 0.05f;                   /* :290, :292 */
  p->lo_free = 1; p->lo_occ = 6; p->lo_min = -80; p->lo_max = 80;    /* :194-197 */
}

const char* uqs_last_error(void) { return g_err; }

int uqs_init(int device) {
  g_cur = &g_single;
  if (g_single.ready && g_single.device == device) {
    cudaSetDevice(device);
    return UQS_OK;
  }
  if (g_single.ready) uqs_shutdown();
  return context_init(g_single, device);
}

void uqs_shutdown(void) {
  Context* saved = g_cur;
  g_cur = &g_single;
  context_shutdown(g_single);
  g_cur = (saved == &g_single) ? &g_single : saved;
}

int uqs_device_sm_count(void) { return g_ctx.ready ? g_ctx.sm_count : 0; }

int uqs_set_stream(void* s) {
  int rc = check_ready();
  if (rc) return rc;
  g_ctx.ext_stream = (cudaStream_t)s;
  g_ctx.use_ext = true;      /* NULL = the legacy default stream, which torch uses unless told otherwise */
  return UQS_OK;
}

int uqs_use_own_stream(void) {
  int rc = check_ready();
  if (rc) return rc;
  g_ctx.use_ext = false;
  return UQS_OK;
}

int uqs_sync(void) {
  int rc = check_ready();
  if (rc) return rc;
  cudaError_t e = cudaStreamSynchronize(g_ctx.stream());
  if (e != cudaSuccess) return cuda_fail(e, "cudaStreamSynchronize");
  return UQS_OK;
}

int uqs_set_tuning(int sw, int sh, int time_slices) {
  if (sw < 0 || sh < 0 || time_slices < 0) { set_error("negative tuning value"); return UQS_ERR_BAD_ARG; }
  g_ctx.tune_sw = sw;
  g_ctx.tune_sh = sh;
  g_ctx.tune_slices = time_slices;
  return UQS_OK;
}

int uqs_set_engine(int engine, int flight_warps) {
  if (engine < 0 || engine > 3 || (flight_warps != 0 && flight_warps != 4 && flight_warps != 8 && flight_warps != 16 && flight_warps != 32)) {
    set_error("engine must be 0 (auto), 1 (sub-tiles), 2 (grid resident) or 3 (unrestricted); warps 0, 4, 8, 16 or 32");
    return UQS_ERR_BAD_ARG;
  }
  g_ctx.engine = engine;
  g_ctx.flight_warps = flight_warps;
  return UQS_OK;
}

/* Lane layout of the resident engine's free-space steps: 0 = 32 beams x 1 step, 1 = 8 beams of one sensor x 4
 * consecutive steps (see k_replay_flights).  Identical bytes. */
/* Experiment knob: row pitch of the resident box in 32-bit words, modulo 32 (-1 = the built-in odd pitch). */
int uqs_set_resident_pitch_mod(int words_mod32) {
  g_ctx.pitch_mod = words_mod32 < 0 ? -1 : (words_mod32 & 31);
  return UQS_OK;
}

/* Resident engine with a dedicated decode warp (0 = every warp decodes every NW-th frame, 1 = an extra producer warp;
 * -1 = the built-in choice).  Identical bytes. */
int uqs_set_decode_warp(int on) {
  g_ctx.flight_prod = on < 0 ? kDefaultDecodeWarp : (on ? 1 : 0);
  return UQS_OK;
}

/* Measurement knob: adds `steps` (0..8) to every frame's collision bound K0 (a larger K0 is always safe: more steps
 * take the collision-checked path).  Prices one collision-checked step per frame in the resident engine. */
int uqs_set_k0_bias(int steps) {
  g_ctx.k0_bias = steps < 0 ? 0 : (steps > 8 ? 8 : steps);
  return UQS_OK;
}

/* Schedule of the resident engine's device calls: n > 0 = the ray set-up of each chunk of n resident waves runs beside
 * the previous chunk's replay, 0 = set-up and replay in turn, -1 = the built-in choice.  Identical bytes. */
int uqs_set_setup_overlap(int waves) {
  g_ctx.setup_overlap = waves < 0 ? kDefaultSetupOverlap : std::min(waves, 64);
  return UQS_OK;
}

int uqs_setup_overlap_chunks(void) { return g_ctx.overlap_chunks; }

int uqs_set_fan_layout(int on) {
  g_ctx.flight_fan = on < 0 ? kDefaultFanLayout : (on ? 1 : 0);
  return UQS_OK;
}

unsigned long long uqs_kernel_launches(void) { return g_ctx.launches; }

int uqs_set_profiling(int on) {
  int rc = check_ready();
  if (rc) return rc;
  g_ctx.profiling = on != 0;
  return UQS_OK;
}

/* Sum of device time per kernel family since the last call (ms): [0] pose, [1] ray set-up,
 * [2] replay; counts[] = launches of each.  Synchronises the stream. */
int uqs_profile_collect(double ms[3], int counts[3]) {
  int rc = check_ready();
  if (rc) return rc;
  cudaError_t e = cudaStreamSynchronize(g_ctx.stream());
  if (e != cudaSuccess) return cuda_fail(e, "profile sync");
  for (int i = 0; i < 3; i++) { ms[i] = 0.0; counts[i] = 0; }
  for (auto& s : g_ctx.spans) {
    float t = 0.f;
    if (s.kind < 3 && cudaEventElapsedTime(&t, s.a, s.b) == cudaSuccess) { ms[s.kind] += t; counts[s.kind]++; }
    cudaEventDestroy(s.a);
    cudaEventDestroy(s.b);
  }
  g_ctx.spans.clear();
  return UQS_OK;
}

/* Timeline of the spans recorded since the last uqs_profile_collect(): out[3*i] = kind (0 pose, 1 ray set-up,
 * 2 replay, 3 H2D, 4 D2H), out[3*i+1], out[3*i+2] = start, end in ms after the first span's start.  Returns the
 * number of spans written (at most max_spans); does not clear them.  Synchronises the device. */
int uqs_profile_timeline(double* out, int max_spans) {
  int rc = check_ready();
  if (rc) return -1;
  if (cudaDeviceSynchronize() != cudaSuccess || g_ctx.spans.empty() || !out) return 0;
  int n = 0;
  const cudaEvent_t ref = g_ctx.spans[0].a;
  for (auto& s : g_ctx.spans) {
    if (n >= max_spans) break;
    float t0 = 0.f, t1 = 0.f;
    if (cudaEventElapsedTime(&t0, ref, s.a) != cudaSuccess || cudaEventElapsedTime(&t1, ref, s.b) != cudaSuccess) continue;
    out[3 * n] = s.kind; out[3 * n + 1] = t0; out[3 * n + 2] = t1;
    n++;
  }
  return n;
}

int uqs_replay_dev(const uqs_params* p, int n_flights, int n_frames, const float* x, const float* y,
                   const float* yaw, const float* ranges, int8_t* grids, int accumulate, int row0,
                   int rows, uqs_stats* stats) {
  int rc = check_ready();
  if (rc) return rc;
  DevParams dp;
  if ((rc = make_dev_params(p, &dp))) return rc;
  if (n_flights <= 0 || n_frames <= 0 || !x || !y || !yaw || !ranges || !grids) {
    set_error("uqs_replay_dev: NULL pointer or non-positive size");
    return UQS_ERR_BAD_ARG;
  }
  if (row0 < 0 || rows <= 0 || row0 + rows > p->H) { set_error("row range [%d,%d) outside the grid", row0, row0 + rows); return UQS_ERR_BAD_ARG; }
  if ((rc = replay_device(dp, n_flights, n_frames, x, y, yaw, ranges, nullptr, grids, accumulate, row0, rows, true)))
    return rc;
  return fetch_stats(stats, (uint64_t)n_flights * n_frames);
}

int uqs_pose_integrate_dev(int n_flights, int n_samples, const uint32_t* t_ms, const float* rx,
                           const float* ry, const float* h, const float* yaw, const uint8_t* q,
                           float* xo, float* yo, int mode) {
  int rc = check_ready();
  if (rc) return rc;
  if (n_flights <= 0 || n_samples <= 0 || !t_ms || !rx || !ry || !h || !yaw || !q || !xo || !yo || (mode != 0 && mode != 1)) {
    set_error("uqs_pose_integrate_dev: bad argument");
    return UQS_ERR_BAD_ARG;
  }
  return pose_device(n_flights, n_samples, t_ms, rx, ry, h, yaw, q, xo, yo, mode);
}

/* ---- host-buffer forms: stage through library-owned device buffers --------------------- */

static int h2d(DevBuf& b, const void* src, size_t bytes, const char* what) {
  int rc = b.ensure(bytes);
  if (rc) return rc;
  cudaError_t e = cudaMemcpyAsync(b.p, src, bytes, cudaMemcpyHostToDevice, g_ctx.stream());
  if (e != cudaSuccess) return cuda_fail(e, what);
  return UQS_OK;
}

int uqs_pose_integrate(int n_flights, int n_samples, const uint32_t* t_ms, const float* rx,
                       const float* ry, const float* h, const float* yaw, const uint8_t* q,
                       float* xo, float* yo, int mode) {
  int rc = check_ready();
  if (rc) return rc;
  if (n_flights <= 0 || n_samples <= 0 || !t_ms || !rx || !ry || !h || !yaw || !q || !xo || !yo || (mode != 0 && mode != 1)) {
    set_error("uqs_pose_integrate: bad argument");
    return UQS_ERR_BAD_ARG;
  }
  const size_t n = (size_t)n_flights * n_samples;
  if ((rc = h2d(g_ctx.in_t, t_ms, n * 4, "t_ms H2D"))) return rc;
  if ((rc = h2d(g_ctx.in_rx, rx, n * 4, "of_rate_x H2D"))) return rc;
  if ((rc = h2d(g_ctx.in_ry, ry, n * 4, "of_rate_y H2D"))) return rc;
  if ((rc = h2d(g_ctx.in_h, h, n * 4, "h_m H2D"))) return rc;
  if ((rc = h2d(g_ctx.in_yaw, yaw, n * 4, "yaw H2D"))) return rc;
  if ((rc = h2d(g_ctx.in_q, q, n, "of_q H2D"))) return rc;
  if ((rc = g_ctx.in_x.ensure(n * 4)) || (rc = g_ctx.in_y.ensure(n * 4))) return rc;
  if ((rc = pose_device(n_flights, n_samples, (uint32_t*)g_ctx.in_t.p, (float*)g_ctx.in_rx.p, (float*)g_ctx.in_ry.p,
                        (float*)g_ctx.in_h.p, (float*)g_ctx.in_yaw.p, (uint8_t*)g_ctx.in_q.p, (float*)g_ctx.in_x.p,
                        (float*)g_ctx.in_y.p, mode)))
    return rc;
  cudaError_t e = cudaMemcpyAsync(xo, g_ctx.in_x.p, n * 4, cudaMemcpyDeviceToHost, g_ctx.stream());
  if (e == cudaSuccess) e = cudaMemcpyAsync(yo, g_ctx.in_y.p, n * 4, cudaMemcpyDeviceToHost, g_ctx.stream());
  if (e == cudaSuccess) e = cudaStreamSynchronize(g_ctx.stream());
  if (e != cudaSuccess) return cuda_fail(e, "pose D2H");
  return UQS_OK;
}

int uqs_beam_cells(const uqs_params* p, int n_frames, const float* x, const float* y, const float* yaw,
                   const float* ranges, int32_t* cells_out, int32_t* origin_out) {
  int rc = check_ready();
  if (rc) return rc;
  DevParams dp;
  if ((rc = make_dev_params(p, &dp))) return rc;
  if (n_frames <= 0 || !x || !y || !yaw || !ranges || !cells_out || !origin_out) { set_error("uqs_beam_cells: bad argument"); return UQS_ERR_BAD_ARG; }
  if ((rc = ensure_inv_table())) return rc;
  cudaStream_t st = g_ctx.stream();
  const size_t n = (size_t)n_frames;
  const int gpf = (n_frames + 31) / 32;
  if ((rc = h2d(g_ctx.in_x, x, n * 4, "x H2D")) || (rc = h2d(g_ctx.in_y, y, n * 4, "y H2D")) ||
      (rc = h2d(g_ctx.in_yaw, yaw, n * 4, "yaw H2D")) || (rc = h2d(g_ctx.in_ranges, ranges, n * 128, "ranges H2D")))
    return rc;
  if ((rc = g_ctx.w->rays.ensure(n * 32 * sizeof(uint2))) || (rc = g_ctx.w->frames.ensure(n * sizeof(uint4))) ||
      (rc = g_ctx.w->groups.ensure((size_t)gpf * sizeof(uint2))) || (rc = g_ctx.w->counters.ensure(64 * 8)) ||
      (rc = g_ctx.out_grids.ensure(n * 32 * 2 * 4 + n * 2 * 4)))
    return rc;
  cudaError_t e = cudaMemsetAsync(g_ctx.w->counters.p, 0, 64, st);
  if (e != cudaSuccess) return cuda_fail(e, "memset");
  e = ray_setup_launch(dim3((unsigned)gpf), st, dp, n_frames, (float*)g_ctx.in_x.p, (float*)g_ctx.in_y.p, (float*)g_ctx.in_yaw.p,
                       (float*)g_ctx.in_ranges.p, nullptr, 0, (const uint32_t*)g_ctx.inv_table.p, (uint4*)g_ctx.w->frames.p,
                       (uint2*)g_ctx.w->groups.p, (uint2*)g_ctx.w->rays.p, (unsigned long long*)g_ctx.w->counters.p);
  if (e != cudaSuccess) return cuda_fail(e, "k_ray_setup launch");
  int32_t* d_cells = (int32_t*)g_ctx.out_grids.p;
  int32_t* d_origin = d_cells + n * 64;
  k_records_to_cells<<<(unsigned)((n * 32 + 255) / 256), 256, 0, st>>>((long long)n, (uint4*)g_ctx.w->frames.p,
                                                                       (uint2*)g_ctx.w->rays.p, d_cells, d_origin);
  e = cudaGetLastError();
  if (e != cudaSuccess) return cuda_fail(e, "beam_cells kernels");
  e = cudaMemcpyAsync(cells_out, d_cells, n * 64 * 4, cudaMemcpyDeviceToHost, st);
  if (e == cudaSuccess) e = cudaMemcpyAsync(origin_out, d_origin, n * 2 * 4, cudaMemcpyDeviceToHost, st);
  if (e == cudaSuccess) e = cudaStreamSynchronize(st);
  if (e != cudaSuccess) return cuda_fail(e, "beam_cells D2H");
  g_ctx.launches += 2;
  return UQS_OK;
}

/* Parity hook for the collision bound: K0 and the angular-order flag of every frame, as k_ray_setup writes
 * them for the resident engine, K0 including the bias of uqs_set_k0_bias.  tests/ verify by brute force that no two
 * beams of a frame share a cell at any step >= K0 and that flagged frames really are in circular angular order. */
int uqs_frame_bounds(const uqs_params* p, int n_frames, const float* x, const float* y, const float* yaw,
                     const float* ranges, int32_t* k0_out, int32_t* sorted_out) {
  int rc = check_ready();
  if (rc) return rc;
  DevParams dp;
  if ((rc = make_dev_params(p, &dp))) return rc;
  if (n_frames <= 0 || !x || !y || !yaw || !ranges || !k0_out || !sorted_out) { set_error("uqs_frame_bounds: bad argument"); return UQS_ERR_BAD_ARG; }
  if ((rc = ensure_inv_table())) return rc;
  cudaStream_t st = g_ctx.stream();
  const size_t n = (size_t)n_frames;
  const int gpf = (n_frames + 31) / 32;
  if ((rc = h2d(g_ctx.in_x, x, n * 4, "x H2D")) || (rc = h2d(g_ctx.in_y, y, n * 4, "y H2D")) ||
      (rc = h2d(g_ctx.in_yaw, yaw, n * 4, "yaw H2D")) || (rc = h2d(g_ctx.in_ranges, ranges, n * 128, "ranges H2D")))
    return rc;
  if ((rc = g_ctx.w->rays.ensure(n * 32 * sizeof(uint2))) || (rc = g_ctx.w->frames.ensure(n * sizeof(uint4))) ||
      (rc = g_ctx.w->groups.ensure((size_t)gpf * sizeof(uint2))) || (rc = g_ctx.w->counters.ensure(64 * 8)))
    return rc;
  cudaError_t e = cudaMemsetAsync(g_ctx.w->counters.p, 0, 64, st);
  if (e != cudaSuccess) return cuda_fail(e, "memset");
  e = ray_setup_launch(dim3((unsigned)gpf), st, dp, n_frames, (float*)g_ctx.in_x.p, (float*)g_ctx.in_y.p, (float*)g_ctx.in_yaw.p,
                       (float*)g_ctx.in_ranges.p, nullptr, 1 + g_ctx.k0_bias, (const uint32_t*)g_ctx.inv_table.p,
                       (uint4*)g_ctx.w->frames.p, (uint2*)g_ctx.w->groups.p, (uint2*)g_ctx.w->rays.p,
                       (unsigned long long*)g_ctx.w->counters.p);
  if (e != cudaSuccess) return cuda_fail(e, "k_ray_setup launch");
  std::vector<uint4> fr(n);
  e = cudaMemcpyAsync(fr.data(), g_ctx.w->frames.p, n * sizeof(uint4), cudaMemcpyDeviceToHost, st);
  if (e == cudaSuccess) e = cudaStreamSynchronize(st);
  if (e != cudaSuccess) return cuda_fail(e, "frame_bounds D2H");
  for (size_t i = 0; i < n; i++) {
    k0_out[i] = (fr[i].y & kFrameHasOrigin) ? (int32_t)(fr[i].x >> 16) : -1;       // -1: the frame's pose is off the grid
    sorted_out[i] = (fr[i].y & kFrameSorted) ? 1 : 0;
  }
  g_ctx.launches += 1;
  return UQS_OK;
}

int uqs_sincosf_batch(size_t n, const float* ang, float* s, float* c) {
  int rc = check_ready();
  if (rc) return rc;
  if (!n || !ang || !s || !c) { set_error("uqs_sincosf_batch: bad argument"); return UQS_ERR_BAD_ARG; }
  cudaStream_t st = g_ctx.stream();
  if ((rc = h2d(g_ctx.in_x, ang, n * 4, "ang H2D")) || (rc = g_ctx.in_y.ensure(n * 4)) || (rc = g_ctx.in_yaw.ensure(n * 4)))
    return rc;
  k_sincosf<<<(unsigned)((n + 255) / 256), 256, 0, st>>>(n, (float*)g_ctx.in_x.p, (float*)g_ctx.in_y.p, (float*)g_ctx.in_yaw.p);
  cudaError_t e = cudaGetLastError();
  if (e == cudaSuccess) e = cudaMemcpyAsync(s, g_ctx.in_y.p, n * 4, cudaMemcpyDeviceToHost, st);
  if (e == cudaSuccess) e = cudaMemcpyAsync(c, g_ctx.in_yaw.p, n * 4, cudaMemcpyDeviceToHost, st);
  if (e == cudaSuccess) e = cudaStreamSynchronize(st);
  if (e != cudaSuccess) return cuda_fail(e, "sincosf batch");
  g_ctx.launches += 1;
  return UQS_OK;
}

int uqs_measure_rmw_peak(double* updates_per_s) {
  int rc = check_ready();
  if (rc) return rc;
  if (!updates_per_s) { set_error("NULL output"); return UQS_ERR_BAD_ARG; }
  cudaStream_t st = g_ctx.stream();
  const int tile_bytes = 4096, iters = 8192;
  const size_t smem = (size_t)tile_bytes * kReplayWarps;
  cudaError_t e = cudaFuncSetAttribute(k_rmw_peak, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
  if (e != cudaSuccess) return cuda_fail(e, "cudaFuncSetAttribute(k_rmw_peak)");
  int per_sm = 0;
  e = cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, k_rmw_peak, kReplayThreads, smem);
  if (e != cudaSuccess || per_sm < 1) return cuda_fail(e, "occupancy(k_rmw_peak)");
  if ((rc = g_ctx.w->counters.ensure(64 * 8))) return rc;
  const unsigned grid = (unsigned)(per_sm * g_ctx.sm_count);
  cudaEvent_t a, b;
  cudaEventCreate(&a);
  cudaEventCreate(&b);
  k_rmw_peak<<<grid, kReplayThreads, smem, st>>>(tile_bytes, 64, -80, (int*)g_ctx.w->counters.p + 96);
  cudaEventRecord(a, st);
  k_rmw_peak<<<grid, kReplayThreads, smem, st>>>(tile_bytes, iters, -80, (int*)g_ctx.w->counters.p + 96);
  cudaEventRecord(b, st);
  e = cudaEventSynchronize(b);
  float ms = 0.f;
  cudaEventElapsedTime(&ms, a, b);
  cudaEventDestroy(a);
  cudaEventDestroy(b);
  if (e != cudaSuccess) return cuda_fail(e, "k_rmw_peak");
  const double updates = (double)grid * kReplayThreads * (double)iters * 8.0;
  *updates_per_s = updates / (ms * 1e-3);
  g_ctx.launches += 2;
  return UQS_OK;
}

/* Shared-memory ATOMIC update rate (ATOMS.ADD, conflict-free addresses, eight in flight per warp): the price of the
 * north star's "integer log-odds atomics", reported by bench.py next to uqs_measure_rmw_peak(). */
int uqs_measure_atoms_peak(double* updates_per_s) {
  int rc = check_ready();
  if (rc) return rc;
  if (!updates_per_s) { set_error("NULL output"); return UQS_ERR_BAD_ARG; }
  cudaStream_t st = g_ctx.stream();
  const int tile_bytes = 4096, iters = 2048;
  const size_t smem = (size_t)tile_bytes * kReplayWarps;
  cudaError_t e = cudaFuncSetAttribute(k_atoms_peak, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
  if (e != cudaSuccess) return cuda_fail(e, "cudaFuncSetAttribute(k_atoms_peak)");
  int per_sm = 0;
  e = cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, k_atoms_peak, kReplayThreads, smem);
  if (e != cudaSuccess || per_sm < 1) return cuda_fail(e, "occupancy(k_atoms_peak)");
  if ((rc = g_ctx.w->counters.ensure(64 * 8))) return rc;
  const unsigned grid = (unsigned)(per_sm * g_ctx.sm_count);
  cudaEvent_t a, b;
  cudaEventCreate(&a);
  cudaEventCreate(&b);
  k_atoms_peak<<<grid, kReplayThreads, smem, st>>>(tile_bytes, 64, (int*)g_ctx.w->counters.p + 96);
  cudaEventRecord(a, st);
  k_atoms_peak<<<grid, kReplayThreads, smem, st>>>(tile_bytes, iters, (int*)g_ctx.w->counters.p + 96);
  cudaEventRecord(b, st);
  e = cudaEventSynchronize(b);
  float ms = 0.f;
  cudaEventElapsedTime(&ms, a, b);
  cudaEventDestroy(a);
  cudaEventDestroy(b);
  if (e != cudaSuccess) return cuda_fail(e, "k_atoms_peak");
  *updates_per_s = (double)grid * kReplayThreads * (double)iters * 8.0 / (ms * 1e-3);
  g_ctx.launches += 2;
  return UQS_OK;
}

}  // extern "C"
