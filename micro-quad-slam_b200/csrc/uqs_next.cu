// uqs_next.cu -- the rows either side of the hot path (SURVEY.md section 8(f)):
//   N1  raw 8x8 ToF scans -> 32 beams        compute_beams_and_minima / robust_col_dist_m, uav_local_nav.c:1320-1359
//   N2  map recentering                      map_recenter_shift / map_recentre_if_needed,  uav_local_nav.c:308-353
//   N3  frontier scoring (grid consumer)     frontier_score_dir,                           uav_local_nav.c:356-385
// Same rules as the hot path: one rounding per C operator, glibc sincosf restated, no host arithmetic.
#include <cmath>
#include <cstdio>
#include <vector>

#include "uqs_host.h"

namespace uqs {

// ---------------------------------------------------------------------------------------------
// N1: per column, the second-smallest valid range over the 8 rows (smallest if only one is valid)
// ---------------------------------------------------------------------------------------------
// raw: [n][512] bytes = 4 sensors (F,R,B,L) x 64 cells x u16 little-endian millimetres (tof_esp32.ino:192-211)
__global__ void k_scans_to_beams(long long n, const uint8_t* __restrict__ raw, float max_range,
                                 float* __restrict__ beams, float* __restrict__ dir_min) {
  const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;     // (frame, d, c)
  if (i >= n * 32) return;
  const long long f = i >> 5;
  const int d = (int)(i >> 3) & 3, c = (int)i & 7;
  const uint8_t* g = raw + f * 512 + d * 128;
  const float qnan = __int_as_float(0x7fc00000);
  float best = qnan, second = qnan;
#pragma unroll
  for (int row = 0; row < 8; row++) {
    const int k = (row * 8 + c) * 2;
    const unsigned mm = (unsigned)g[k] | ((unsigned)g[k + 1] << 8);
    if (mm == 0xFFFFu || mm == 0u) continue;                       // :1327
    float m = __fmul_rn((float)mm, 0.001f);                        // :1328
    if (m <= 0.02f) continue;                                      // :1329
    if (m > max_range) m = max_range;                              // :1330
    if (isnan(best) || m < best) { second = best; best = m; }      // :1332-1334
    else if (isnan(second) || m < second) second = m;              // :1335-1337
  }
  const float out = !isnan(second) ? second : best;                // :1340-1341
  beams[i] = out;
  if (dir_min) {                                                   // tof_min_m, :1354-1357
    float mn = out;
    for (int o = 1; o < 8; o <<= 1) {
      const float other = __shfl_xor_sync(0xffffffffu, mn, o);
      if (isnan(mn) || (!isnan(other) && other < mn)) mn = other;
    }
    if (c == 0) dir_min[f * 4 + d] = mn;
  }
}

// ---------------------------------------------------------------------------------------------
// N2: recentering
// ---------------------------------------------------------------------------------------------
struct RecenterEvent { int frame, sx, sy; float ox, oy; };     // shift applied BEFORE `frame` is mapped

// map_recentre_if_needed(), :324-349, decision only: returns true and the shift when one is due
__device__ __forceinline__ bool recenter_decide(float res, float size_m, float ox, float oy, float x, float y,
                                                int& sx, int& sy) {
  const float half = __fmul_rn(size_m, 0.5f);
  const float thresh = __fmul_rn(half, 0.60f);
  const float dx = __fsub_rn(x, ox), dy = __fsub_rn(y, oy);
  if (fabsf(dx) < thresh && fabsf(dy) < thresh) return false;
  sx = lrintf_as_int(__fdiv_rn(dx, res));
  sy = lrintf_as_int(__fdiv_rn(dy, res));
  const int max_shift = (int)__fmul_rn(__fdiv_rn(half, res), 0.5f);     // C truncation, :337
  sx = min(max(sx, -max_shift), max_shift);
  sy = min(max(sy, -max_shift), max_shift);
  return !(sx == 0 && sy == 0);
}

// one thread walks one log in order (the decision depends on poses and the running origin only)
__global__ void k_recenter_plan(int n_frames, const float* __restrict__ x, const float* __restrict__ y, float res,
                                float size_m, float ox, float oy, RecenterEvent* events, int max_events, int* n_events) {
  if (blockIdx.x != 0 || threadIdx.x != 0) return;
  int n = 0;
  for (int f = 0; f < n_frames; f++) {
    int sx, sy;
    if (recenter_decide(res, size_m, ox, oy, x[f], y[f], sx, sy)) {
      ox = __fadd_rn(ox, __fmul_rn((float)sx, res));                     // :346-347
      oy = __fadd_rn(oy, __fmul_rn((float)sy, res));
      if (n < max_events) events[n] = { f, sx, sy, ox, oy };
      n++;
    }
  }
  *n_events = n;
}

__global__ void k_recenter_decide_one(float res, float size_m, float ox, float oy, float x, float y, int* out) {
  int sx = 0, sy = 0;
  const bool go = recenter_decide(res, size_m, ox, oy, x, y, sx, sy);
  out[0] = go ? 1 : 0;
  out[1] = sx;
  out[2] = sy;
  reinterpret_cast<float*>(out)[3] = go ? __fadd_rn(ox, __fmul_rn((float)sx, res)) : ox;
  reinterpret_cast<float*>(out)[4] = go ? __fadd_rn(oy, __fmul_rn((float)sy, res)) : oy;
}

// map_recenter_shift(), :308-322: dst(x,y) = src(x+sx, y+sy) inside the grid, else 0
__global__ void k_recenter_shift(const int8_t* __restrict__ src, int8_t* __restrict__ dst, int W, int H, int sx, int sy) {
  const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= (long long)W * H) return;
  const int yy = (int)(i / W), xx = (int)(i - (long long)yy * W);
  const int u = xx + sx, v = yy + sy;
  dst[i] = (u >= 0 && u < W && v >= 0 && v < H) ? src[(size_t)v * W + u] : (int8_t)0;
}

// ---------------------------------------------------------------------------------------------
// N3: frontier scoring
// ---------------------------------------------------------------------------------------------
__global__ void k_frontier_scores(DevParams p, const int8_t* __restrict__ grid, int n, const float* __restrict__ x,
                                  const float* __restrict__ y, const float* __restrict__ yaw_deg,
                                  const float* __restrict__ offset_deg, int* __restrict__ scores,
                                  unsigned long long* __restrict__ domain_errors) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  const float step = frontier_step(p);
  int score = 0;
  for (int r = 0; r < 3; r++) {
    float sa, ca;
    if (!sincosf_glibc(frontier_ray_angle(p, yaw_deg[i], offset_deg[i], r), sa, ca)) { atomicAdd(domain_errors, 1ull); continue; }
    for (float d = step; d <= kFrontierRange; d = __fadd_rn(d, step)) {   // :371
      int gx, gy;
      if (!frontier_point(p, x[i], y[i], d, ca, sa, gx, gy)) break;
      score += frontier_weight((int)grid[(size_t)gy * p.W + gx]);
    }
  }
  scores[i] = score;                                               // unknown*3 + free - occ*4, :383
}

}  // namespace uqs

using namespace uqs;

namespace {
int stage(DevBuf& b, const void* src, size_t bytes) {
  int rc = b.ensure(bytes);
  if (rc) return rc;
  cudaError_t e = cudaMemcpyAsync(b.p, src, bytes, cudaMemcpyHostToDevice, g_ctx.stream());
  return e == cudaSuccess ? UQS_OK : cuda_fail(e, "H2D");
}
}  // namespace

extern "C" {

/* N1 */
int uqs_beams_from_scans_dev(long long n_frames, const uint8_t* raw_dev, float max_range_m, float* beams_dev,
                             float* dir_min_dev) {
  int rc = check_ready();
  if (rc) return rc;
  if (n_frames <= 0 || !raw_dev || !beams_dev) { set_error("uqs_beams_from_scans_dev: bad argument"); return UQS_ERR_BAD_ARG; }
  k_scans_to_beams<<<(unsigned)((n_frames * 32 + 255) / 256), 256, 0, g_ctx.stream()>>>(n_frames, raw_dev, max_range_m,
                                                                                      beams_dev, dir_min_dev);
  cudaError_t e = cudaGetLastError();
  if (e != cudaSuccess) return cuda_fail(e, "k_scans_to_beams");
  g_ctx.launches += 1;
  return UQS_OK;
}

int uqs_beams_from_scans(long long n_frames, const uint8_t* raw, float max_range_m, float* beams_out, float* dir_min_out) {
  int rc = check_ready();
  if (rc) return rc;
  if (n_frames <= 0 || !raw || !beams_out) { set_error("uqs_beams_from_scans: bad argument"); return UQS_ERR_BAD_ARG; }
  if ((rc = stage(g_ctx.in_ranges, raw, (size_t)n_frames * 512)) || (rc = g_ctx.in_x.ensure((size_t)n_frames * 128)) ||
      (rc = g_ctx.in_y.ensure((size_t)n_frames * 16)))
    return rc;
  if ((rc = uqs_beams_from_scans_dev(n_frames, (uint8_t*)g_ctx.in_ranges.p, max_range_m, (float*)g_ctx.in_x.p,
                                     dir_min_out ? (float*)g_ctx.in_y.p : nullptr)))
    return rc;
  cudaError_t e = cudaMemcpyAsync(beams_out, g_ctx.in_x.p, (size_t)n_frames * 128, cudaMemcpyDeviceToHost, g_ctx.stream());
  if (e == cudaSuccess && dir_min_out)
    e = cudaMemcpyAsync(dir_min_out, g_ctx.in_y.p, (size_t)n_frames * 16, cudaMemcpyDeviceToHost, g_ctx.stream());
  if (e == cudaSuccess) e = cudaStreamSynchronize(g_ctx.stream());
  return e == cudaSuccess ? UQS_OK : cuda_fail(e, "beams D2H");
}

/* N3 */
int uqs_frontier_scores(const uqs_params* p, const int8_t* grid /* host, [H][W] */, int n, const float* x, const float* y,
                        const float* yaw_deg, const float* offset_deg, int* scores_out) {
  int rc = check_ready();
  if (rc) return rc;
  DevParams dp;
  if ((rc = make_dev_params(p, &dp))) return rc;
  if (!grid || n <= 0 || !x || !y || !yaw_deg || !offset_deg || !scores_out) { set_error("uqs_frontier_scores: bad argument"); return UQS_ERR_BAD_ARG; }
  cudaStream_t st = g_ctx.stream();
  if ((rc = stage(g_ctx.out_grids, grid, (size_t)p->W * p->H)) || (rc = stage(g_ctx.in_x, x, (size_t)n * 4)) ||
      (rc = stage(g_ctx.in_y, y, (size_t)n * 4)) || (rc = stage(g_ctx.in_yaw, yaw_deg, (size_t)n * 4)) ||
      (rc = stage(g_ctx.in_h, offset_deg, (size_t)n * 4)) || (rc = g_ctx.in_t.ensure((size_t)n * 4)) ||
      (rc = g_ctx.w->counters.ensure(64 * 8)))
    return rc;
  unsigned long long* dom = (unsigned long long*)g_ctx.w->counters.p + 24;
  cudaError_t e = cudaMemsetAsync(dom, 0, 8, st);
  if (e != cudaSuccess) return cuda_fail(e, "memset");
  k_frontier_scores<<<(unsigned)((n + 127) / 128), 128, 0, st>>>(dp, (int8_t*)g_ctx.out_grids.p, n, (float*)g_ctx.in_x.p,
                                                                (float*)g_ctx.in_y.p, (float*)g_ctx.in_yaw.p,
                                                                (float*)g_ctx.in_h.p, (int*)g_ctx.in_t.p, dom);
  unsigned long long hdom = 0;
  e = cudaGetLastError();
  if (e == cudaSuccess) e = cudaMemcpyAsync(scores_out, g_ctx.in_t.p, (size_t)n * 4, cudaMemcpyDeviceToHost, st);
  if (e == cudaSuccess) e = cudaMemcpyAsync(&hdom, dom, 8, cudaMemcpyDeviceToHost, st);
  if (e == cudaSuccess) e = cudaStreamSynchronize(st);
  if (e != cudaSuccess) return cuda_fail(e, "k_frontier_scores");
  g_ctx.launches += 1;
  if (hdom) { set_error("%llu frontier rays outside the restated sincosf domain", hdom); return UQS_ERR_DOMAIN; }
  return UQS_OK;
}

/* N2: one log replayed with the reference's recentering honoured (log_tick order, :1629-1635:
 * recentre check first, then the update).  origin_out = final map origin; events_out (may be NULL, capacity
 * max_events) gets {frame, sx, sy} triples. */
int uqs_replay_recentering(const uqs_params* p, int n_frames, const float* x, const float* y, const float* yaw_deg,
                           const float* ranges, int8_t* grid_out, float origin_out[2], int* n_events_out,
                           int* events_out, int max_events, uqs_stats* stats) {
  int rc = check_ready();
  if (rc) return rc;
  DevParams dp;
  if ((rc = make_dev_params(p, &dp))) return rc;
  if (n_frames <= 0 || !x || !y || !yaw_deg || !ranges || !grid_out) { set_error("uqs_replay_recentering: bad argument"); return UQS_ERR_BAD_ARG; }
  cudaStream_t st = g_ctx.stream();
  const size_t cells = (size_t)p->W * p->H, n = (size_t)n_frames;
  const int cap = 4096;
  if ((rc = stage(g_ctx.in_x, x, n * 4)) || (rc = stage(g_ctx.in_y, y, n * 4)) || (rc = stage(g_ctx.in_yaw, yaw_deg, n * 4)) ||
      (rc = stage(g_ctx.in_ranges, ranges, n * 128)) || (rc = g_ctx.out_grids.ensure(2 * cells)) ||
      (rc = g_ctx.in_t.ensure(cap * sizeof(RecenterEvent) + 16)))
    return rc;
  RecenterEvent* d_ev = (RecenterEvent*)g_ctx.in_t.p;
  int* d_n = (int*)((char*)g_ctx.in_t.p + cap * sizeof(RecenterEvent));
  k_recenter_plan<<<1, 1, 0, st>>>(n_frames, (float*)g_ctx.in_x.p, (float*)g_ctx.in_y.p, p->res_m, p->size_m, p->origin_x,
                                   p->origin_y, d_ev, cap, d_n);
  int n_ev = 0;
  cudaError_t e = cudaGetLastError();
  if (e == cudaSuccess) e = cudaMemcpyAsync(&n_ev, d_n, 4, cudaMemcpyDeviceToHost, st);
  if (e == cudaSuccess) e = cudaStreamSynchronize(st);
  if (e != cudaSuccess) return cuda_fail(e, "k_recenter_plan");
  if (n_ev > cap) { set_error("%d recenter events exceed the supported %d", n_ev, cap); return UQS_ERR_BAD_ARG; }
  std::vector<RecenterEvent> ev((size_t)n_ev);
  if (n_ev) {
    e = cudaMemcpy(ev.data(), d_ev, (size_t)n_ev * sizeof(RecenterEvent), cudaMemcpyDeviceToHost);
    if (e != cudaSuccess) return cuda_fail(e, "events D2H");
  }
  int8_t* g0 = (int8_t*)g_ctx.out_grids.p;
  int8_t* g1 = g0 + cells;
  if ((e = cudaMemsetAsync(g0, 0, cells, st)) != cudaSuccess) return cuda_fail(e, "memset grid");
  uqs_params q = *p;
  uqs_stats total = { 0, 0, 0, 0, 0 }, part;
  int f0 = 0;
  for (int k = 0; k <= n_ev; k++) {
    const int f1 = (k < n_ev) ? ev[k].frame : n_frames;
    if (f1 > f0) {
      DevParams dq;
      if ((rc = make_dev_params(&q, &dq))) return rc;
      if ((rc = replay_device(dq, 1, f1 - f0, (float*)g_ctx.in_x.p + f0, (float*)g_ctx.in_y.p + f0, (float*)g_ctx.in_yaw.p + f0,
                              (float*)g_ctx.in_ranges.p + (size_t)f0 * 32, nullptr, g0, 1, 0, p->H, true)))
        return rc;
      rc = fetch_stats(&part, (uint64_t)(f1 - f0));
      if (rc) return rc;
      total.ray_cell_updates += part.ray_cell_updates; total.rays_accepted += part.rays_accepted;
      total.rays_skipped += part.rays_skipped; total.frames += part.frames;
    }
    if (k < n_ev) {
      k_recenter_shift<<<(unsigned)((cells + 255) / 256), 256, 0, st>>>(g0, g1, p->W, p->H, ev[k].sx, ev[k].sy);
      if ((e = cudaGetLastError()) != cudaSuccess) return cuda_fail(e, "k_recenter_shift");
      std::swap(g0, g1);
      q.origin_x = ev[k].ox;
      q.origin_y = ev[k].oy;
      g_ctx.launches += 1;
    }
    f0 = f1;
  }
  e = cudaMemcpyAsync(grid_out, g0, cells, cudaMemcpyDeviceToHost, st);
  if (e == cudaSuccess) e = cudaStreamSynchronize(st);
  if (e != cudaSuccess) return cuda_fail(e, "grid D2H");
  if (origin_out) { origin_out[0] = q.origin_x; origin_out[1] = q.origin_y; }
  if (n_events_out) *n_events_out = n_ev;
  if (events_out)
    for (int k = 0; k < n_ev && k < max_events; k++) { events_out[3 * k] = ev[k].frame; events_out[3 * k + 1] = ev[k].sx; events_out[3 * k + 2] = ev[k].sy; }
  if (stats) *stats = total;
  return UQS_OK;
}

}  // extern "C"
