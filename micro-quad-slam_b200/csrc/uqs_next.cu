// uqs_next.cu -- the rows either side of the hot path (SURVEY.md section 8(f)):
//   N1  raw 8x8 ToF scans -> 32 beams        compute_beams_and_minima / robust_col_dist_m, uav_local_nav.c:1320-1359
//   N2  map recentering                      map_recenter_shift / map_recentre_if_needed,  uav_local_nav.c:308-353
//   N3  frontier scoring (grid consumer)     frontier_score_dir,                           uav_local_nav.c:356-385
// Same rules as the hot path: one rounding per C operator, glibc sincosf restated, no host arithmetic.
#include <algorithm>
#include <climits>
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

// One thread per flight walks its poses in order: the decision depends on the poses and the running origin only, so
// the whole plan exists before any replay.  Pass 1 (WRITE = false): info[f] = {events, min Sx, min Sy, max Sx, max Sy}
// (S = 0 included: the first window) and s_min[f].  Pass 2: the events, at ev_start[f].  S is summed in 64 bits and
// its extremes saturate at +-2^30 (such a flight cannot take the sub-tile route anyway).
constexpr int kPlanInfo = 5;
template <bool WRITE>
__global__ void k_recenter_plan(int n_flights, int n_frames, const float* __restrict__ x, const float* __restrict__ y,
                                float res, float size_m, float ox, float oy, int* __restrict__ info, int2* __restrict__ s_min,
                                const int* __restrict__ ev_start, PlanEvent* __restrict__ events) {
  const int f = blockIdx.x * blockDim.x + threadIdx.x;
  if (f >= n_flights) return;
  const float* xf = x + (size_t)f * n_frames;
  const float* yf = y + (size_t)f * n_frames;
  PlanEvent* out = WRITE ? events + ev_start[f] : nullptr;
  long long Sx = 0, Sy = 0, lo_x = 0, lo_y = 0, hi_x = 0, hi_y = 0;
  int n = 0;
  for (int i = 0; i < n_frames; i++) {
    int sx, sy;
    if (recenter_decide(res, size_m, ox, oy, __ldg(&xf[i]), __ldg(&yf[i]), sx, sy)) {
      ox = __fadd_rn(ox, __fmul_rn((float)sx, res));                     // :346-347
      oy = __fadd_rn(oy, __fmul_rn((float)sy, res));
      Sx += sx;
      Sy += sy;
      if (WRITE) {
        out[n] = { i, sx, sy, 0, (int)Sx, (int)Sy, ox, oy };
      } else {
        lo_x = min(lo_x, Sx); lo_y = min(lo_y, Sy);
        hi_x = max(hi_x, Sx); hi_y = max(hi_y, Sy);
      }
      n++;
    }
  }
  if (!WRITE) {
    const long long cap = 1ll << 30;
    int* o = info + (size_t)f * kPlanInfo;
    o[0] = n;
    o[1] = (int)max(lo_x, -cap); o[2] = (int)max(lo_y, -cap);
    o[3] = (int)min(hi_x, cap);  o[4] = (int)min(hi_y, cap);
    s_min[f] = make_int2(o[1], o[2]);
  }
}

// per flight: the final origin, the event count and the first max_events {frame, sx, sy}
__global__ void k_recenter_outputs(int n_flights, const int* __restrict__ ev_start, const PlanEvent* __restrict__ events,
                                   float ox, float oy, float* __restrict__ origins, int32_t* __restrict__ n_events,
                                   int32_t* __restrict__ events_out, int max_events) {
  const int f = blockIdx.x * blockDim.x + threadIdx.x;
  if (f >= n_flights) return;
  const int eb = ev_start[f], n = ev_start[f + 1] - eb;
  origins[2 * f] = n ? events[eb + n - 1].ox : ox;
  origins[2 * f + 1] = n ? events[eb + n - 1].oy : oy;
  n_events[f] = n;
  for (int k = 0; k < n && k < max_events; k++) {
    int32_t* e = events_out + ((size_t)f * max_events + k) * 3;
    e[0] = events[eb + k].frame;
    e[1] = events[eb + k].sx;
    e[2] = events[eb + k].sy;
  }
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
      if (!frontier_point(p, p.ox, p.oy, x[i], y[i], d, ca, sa, gx, gy)) break;
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

/* N2 for many flights.  Route A, the sub-tile engine in each flight's global frame, when the inputs suit it: rays of
 * at most kMaxRayCells cells, 0 inside the clamp range, no time slices for this call, global extents that fit the
 * records' 16-bit cells, engine 0 or 1.  Route B otherwise: per flight, the log between two events through
 * replay_device at that segment's origin, then the shift, with the stats summed on the device.  Q (or nullptr): frontier
 * queries whose flights, frames and probe count were checked (frontier_queries_begin), answered at their frame; on
 * route A their probes are in the flights' global frames, on route B each segment's replay serves its own queries. */
static int replay_recentering(const uqs_params* p, const DevParams& dp, int n_flights, int n_frames, const float* x,
                              const float* y, const float* yaw, const float* ranges, int8_t* grids, float* origins,
                              int32_t* n_events, int32_t* events, int max_events, const ProbeSet* Q, unsigned long long* dom,
                              int32_t* scores, uqs_stats* stats) {
  int rc;
  cudaStream_t st = g_ctx.stream();
  Work& W = *g_ctx.w;
  const size_t info_bytes = ((size_t)n_flights * kPlanInfo * sizeof(int) + 15) & ~(size_t)15;
  if ((rc = W.plan_info.ensure(info_bytes + (size_t)n_flights * sizeof(int2))) ||
      (rc = W.plan_start.ensure(((size_t)n_flights + 1) * sizeof(int))))
    return rc;
  int* d_info = (int*)W.plan_info.p;
  int2* d_smin = (int2*)((char*)W.plan_info.p + info_bytes);
  int* d_start = (int*)W.plan_start.p;
  const unsigned blocks = (unsigned)((n_flights + 127) / 128);
  k_recenter_plan<false><<<blocks, 128, 0, st>>>(n_flights, n_frames, x, y, p->res_m, p->size_m, p->origin_x, p->origin_y,
                                                 d_info, d_smin, nullptr, nullptr);
  std::vector<int> info((size_t)n_flights * kPlanInfo);
  cudaError_t e = cudaGetLastError();
  if (e == cudaSuccess) e = cudaMemcpyAsync(info.data(), d_info, info.size() * sizeof(int), cudaMemcpyDeviceToHost, st);
  if (e == cudaSuccess) e = cudaStreamSynchronize(st);
  if (e != cudaSuccess) return cuda_fail(e, "k_recenter_plan");
  g_ctx.launches += 1;
  std::vector<int> start((size_t)n_flights + 1);
  long long total = 0, span_x = 0, span_y = 0;
  for (int f = 0; f < n_flights; f++) {
    const int* o = &info[(size_t)f * kPlanInfo];
    start[f] = (int)total;
    total += o[0];
    span_x = std::max(span_x, (long long)o[3] - o[1]);
    span_y = std::max(span_y, (long long)o[4] - o[2]);
    if (total > INT_MAX) { set_error("more than %d recenter events in one call", INT_MAX); return UQS_ERR_BAD_ARG; }
  }
  start[n_flights] = (int)total;
  if ((rc = W.plan_events.ensure(std::max<size_t>(1, (size_t)total) * sizeof(PlanEvent)))) return rc;
  PlanEvent* d_ev = (PlanEvent*)W.plan_events.p;
  e = cudaMemcpyAsync(d_start, start.data(), start.size() * sizeof(int), cudaMemcpyHostToDevice, st);
  if (e != cudaSuccess) return cuda_fail(e, "plan H2D");
  k_recenter_plan<true><<<blocks, 128, 0, st>>>(n_flights, n_frames, x, y, p->res_m, p->size_m, p->origin_x, p->origin_y,
                                                nullptr, nullptr, d_start, d_ev);
  k_recenter_outputs<<<blocks, 128, 0, st>>>(n_flights, d_start, d_ev, p->origin_x, p->origin_y, origins, n_events, events,
                                             max_events);
  if ((e = cudaGetLastError()) != cudaSuccess) return cuda_fail(e, "k_recenter_plan");
  g_ctx.launches += 2;

  const int side = std::max(dp.W, dp.H);
  const bool long_rays = side > kMaxRayCells + 1 && !(dp.max_range / dp.res + 3.0f <= (float)kMaxRayCells);
  int sw, sh, nsx, nsy, slices;
  tile_geometry(dp, n_flights, n_frames, dp.H, &sw, &sh, &nsx, &nsy, &slices);
  const long long gw = span_x + dp.W, gh = span_y + dp.H;
  const bool route_a = !long_rays && dp.lo_min <= 0 && dp.lo_max >= 0 && slices == 1 && gw <= 0x7fff && gh <= 0x7fff &&
                       (g_ctx.engine == 0 || g_ctx.engine == 1);
  const bool probes = Q && Q->s_max > 0;             // (a step longer than 2.5 m samples nothing: every score is 0)
  const int* order = nullptr;                        // route B: slot j of the probes holds query order[j]
  if (route_a) {
    if (probes && (rc = frontier_probes_recentered(dp, *Q, Q->queries, nullptr, d_ev, d_start, d_smin, (int)gw, dom)))
      return rc;
    if ((rc = replay_device_recentering(dp, n_flights, n_frames, x, y, yaw, ranges, grids, d_ev, d_start, d_smin, (int)gw,
                                        (int)gh, probes ? Q : nullptr)))
      return rc;
  } else {
    std::vector<PlanEvent> ev((size_t)total);
    if (total) {
      e = cudaMemcpyAsync(ev.data(), d_ev, (size_t)total * sizeof(PlanEvent), cudaMemcpyDeviceToHost, st);
      if (e == cudaSuccess) e = cudaStreamSynchronize(st);
      if (e != cudaSuccess) return cuda_fail(e, "events D2H");
    }
    // queries grouped by segment, each segment's probes in its window
    uqs_query* local = nullptr;
    std::vector<int> seg_start;
    if (probes) {
      const long long n_segments = (long long)n_flights + total;
      if (n_segments >= INT_MAX) { set_error("more than %d recentering segments in one call", INT_MAX - 1); return UQS_ERR_BAD_ARG; }
      if ((rc = W.probe_local.ensure((size_t)Q->n_queries * (sizeof(uqs_query) + sizeof(int))))) return rc;
      local = (uqs_query*)W.probe_local.p;
      order = (const int*)(local + Q->n_queries);
      if ((rc = frontier_queries_by_segment(Q->n_queries, Q->queries, d_ev, d_start, (int)n_segments, local, (int*)order,
                                            &seg_start)) ||
          (rc = frontier_probes_recentered(dp, *Q, Q->queries, order, d_ev, d_start, nullptr, dp.W, dom)))
        return rc;
    }
    const size_t cells = (size_t)p->W * p->H;
    if ((rc = W.plan_tmp.ensure(cells)) || (rc = W.counters.ensure(64 * sizeof(unsigned long long)))) return rc;
    int8_t* tmp = (int8_t*)W.plan_tmp.p;
    e = zero_async(W.counters.p, 8 * sizeof(unsigned long long), st);
    if (e == cudaSuccess) e = zero_async(grids, (size_t)n_flights * cells, st);
    if (e != cudaSuccess) return cuda_fail(e, "memset before the segment replay");
    g_ctx.launches += 2;
    for (int f = 0; f < n_flights; f++) {
      uqs_params q = *p;
      int8_t* g = grids + (size_t)f * cells;
      const size_t base = (size_t)f * n_frames;
      int f0 = 0;
      for (int k = start[f]; k <= start[f + 1]; k++) {
        const int f1 = k < start[f + 1] ? ev[k].frame : n_frames;
        if (f1 > f0) {
          DevParams dq;
          if ((rc = make_dev_params(&q, &dq))) return rc;
          ProbeSet S;                                        // the queries of segment k + f
          if (probes) {
            const int j0 = seg_start[(size_t)k + f], nq = seg_start[(size_t)k + f + 1] - j0;
            const size_t s0 = (size_t)j0 * 3 * Q->s_max;
            S.n_queries = nq;
            S.s_max = Q->s_max;
            S.queries = local + j0;
            S.cells = Q->cells + s0;
            S.values = Q->values + s0;
          }
          if ((rc = replay_device(dq, 1, f1 - f0, x + base + f0, y + base + f0, yaw + base + f0, ranges + (base + f0) * 32,
                                  nullptr, g, 1, 0, p->H, false, S.n_queries ? &S : nullptr)))
            return rc;
        }
        if (k < start[f + 1]) {
          k_recenter_shift<<<(unsigned)((cells + 255) / 256), 256, 0, st>>>(g, tmp, p->W, p->H, ev[k].sx, ev[k].sy);
          e = cudaGetLastError();
          if (e == cudaSuccess) e = cudaMemcpyAsync(g, tmp, cells, cudaMemcpyDeviceToDevice, st);
          if (e != cudaSuccess) return cuda_fail(e, "k_recenter_shift");
          q.origin_x = ev[k].ox;
          q.origin_y = ev[k].oy;
          g_ctx.launches += 1;
        }
        f0 = f1;
      }
    }
  }
  if (Q) return frontier_queries_end(*Q, order, scores, dom, stats, (uint64_t)n_flights * n_frames);
  return fetch_stats(stats, (uint64_t)n_flights * n_frames);
}

int uqs_replay_recentering_dev(const uqs_params* p, int n_flights, int n_frames, const float* x, const float* y,
                               const float* yaw, const float* ranges, int8_t* grids, float* origins, int32_t* n_events,
                               int32_t* events, int max_events, uqs_stats* stats) {
  int rc = check_ready();
  if (rc) return rc;
  DevParams dp;
  if ((rc = make_dev_params(p, &dp))) return rc;
  if (n_flights <= 0 || n_frames <= 0 || !x || !y || !yaw || !ranges || !grids || !origins || !n_events || max_events < 0 ||
      (max_events > 0 && !events)) {
    set_error("uqs_replay_recentering_dev: NULL pointer or bad size");
    return UQS_ERR_BAD_ARG;
  }
  if (g_ctx.engine == 2) {
    set_error("uqs_replay_recentering_dev: engine 2 (resident) has no recentering variant; use 0, 1 or 3");
    return UQS_ERR_BAD_ARG;
  }
  return replay_recentering(p, dp, n_flights, n_frames, x, y, yaw, ranges, grids, origins, n_events, events, max_events,
                            nullptr, nullptr, nullptr, stats);
}

/* N2 + N3: uqs_replay_recentering_dev plus frontier queries, each answered against its flight's recentred map at its
 * frame (after that frame's recentering and update), in the window of the origin the flight had then. */
int uqs_replay_recentering_frontier_dev(const uqs_params* p, int n_flights, int n_frames, const float* x, const float* y,
                                        const float* yaw, const float* ranges, int8_t* grids, float* origins,
                                        int32_t* n_events, int32_t* events, int max_events, int n_queries,
                                        const uqs_query* queries, int32_t* scores, uqs_stats* stats) {
  if (n_queries == 0)
    return uqs_replay_recentering_dev(p, n_flights, n_frames, x, y, yaw, ranges, grids, origins, n_events, events, max_events,
                                      stats);
  int rc = check_ready();
  if (rc) return rc;
  DevParams dp;
  if ((rc = make_dev_params(p, &dp))) return rc;
  if (n_flights <= 0 || n_frames <= 0 || !x || !y || !yaw || !ranges || !grids || !origins || !n_events || max_events < 0 ||
      (max_events > 0 && !events) || n_queries < 0 || !queries || !scores) {
    set_error("uqs_replay_recentering_frontier_dev: NULL pointer or bad size");
    return UQS_ERR_BAD_ARG;
  }
  if (g_ctx.engine == 2) {
    set_error("uqs_replay_recentering_frontier_dev: engine 2 (resident) has no recentering variant; use 0, 1 or 3");
    return UQS_ERR_BAD_ARG;
  }
  ProbeSet Q;
  unsigned long long* dom = nullptr;
  if ((rc = frontier_queries_begin("uqs_replay_recentering_frontier_dev", p, n_flights, n_frames, n_queries, queries, &Q, &dom)))
    return rc;
  return replay_recentering(p, dp, n_flights, n_frames, x, y, yaw, ranges, grids, origins, n_events, events, max_events, &Q,
                            dom, scores, stats);
}

/* N2, one log from host buffers: uqs_replay_recentering_dev with one flight. */
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
  const int cap = events_out ? std::max(max_events, 0) : 0;
  if ((rc = stage(g_ctx.in_x, x, n * 4)) || (rc = stage(g_ctx.in_y, y, n * 4)) || (rc = stage(g_ctx.in_yaw, yaw_deg, n * 4)) ||
      (rc = stage(g_ctx.in_ranges, ranges, n * 128)) || (rc = g_ctx.out_grids.ensure(cells + 16)) ||
      (rc = g_ctx.in_t.ensure((size_t)std::max(cap, 1) * 12)))
    return rc;
  int8_t* d_grid = (int8_t*)g_ctx.out_grids.p;
  float* d_origin = (float*)(d_grid + ((cells + 3) & ~(size_t)3));
  int32_t* d_n = (int32_t*)(d_origin + 2);
  uqs_stats local;
  if ((rc = uqs_replay_recentering_dev(p, 1, n_frames, (float*)g_ctx.in_x.p, (float*)g_ctx.in_y.p, (float*)g_ctx.in_yaw.p,
                                       (float*)g_ctx.in_ranges.p, d_grid, d_origin, d_n, cap ? (int32_t*)g_ctx.in_t.p : nullptr,
                                       cap, stats ? stats : &local)))
    return rc;
  float origin[2];
  int n_ev = 0;
  cudaError_t e = cudaMemcpyAsync(grid_out, d_grid, cells, cudaMemcpyDeviceToHost, st);
  if (e == cudaSuccess) e = cudaMemcpyAsync(origin, d_origin, sizeof(origin), cudaMemcpyDeviceToHost, st);
  if (e == cudaSuccess) e = cudaMemcpyAsync(&n_ev, d_n, sizeof(int), cudaMemcpyDeviceToHost, st);
  if (e == cudaSuccess) e = cudaStreamSynchronize(st);
  if (e == cudaSuccess && cap) {
    e = cudaMemcpyAsync(events_out, g_ctx.in_t.p, (size_t)std::min(n_ev, cap) * 12, cudaMemcpyDeviceToHost, st);
    if (e == cudaSuccess) e = cudaStreamSynchronize(st);
  }
  if (e != cudaSuccess) return cuda_fail(e, "uqs_replay_recentering D2H");
  if (origin_out) { origin_out[0] = origin[0]; origin_out[1] = origin[1]; }
  if (n_events_out) *n_events_out = n_ev;
  return UQS_OK;
}

/* N2 + N3 from host buffers: uqs_replay_recentering_frontier_dev staged through the library's buffers. */
int uqs_replay_recentering_frontier(const uqs_params* p, int n_flights, int n_frames, const float* x, const float* y,
                                    const float* yaw_deg, const float* ranges, int8_t* grids_out, float* origins_out,
                                    int n_queries, const uqs_query* queries, int32_t* scores_out, uqs_stats* stats) {
  int rc = check_ready();
  if (rc) return rc;
  if (!p || n_flights <= 0 || n_frames <= 0 || !x || !y || !yaw_deg || !ranges || n_queries < 0 ||
      (n_queries > 0 && (!queries || !scores_out))) {
    set_error("uqs_replay_recentering_frontier: NULL pointer or bad size");
    return UQS_ERR_BAD_ARG;
  }
  cudaStream_t st = g_ctx.stream();
  const size_t n = (size_t)n_flights * n_frames, cells = (size_t)n_flights * p->W * p->H;
  const size_t origins_at = (cells + 15) & ~(size_t)15, n_ev_at = origins_at + (size_t)n_flights * 8;
  if ((rc = stage(g_ctx.in_x, x, n * 4)) || (rc = stage(g_ctx.in_y, y, n * 4)) || (rc = stage(g_ctx.in_yaw, yaw_deg, n * 4)) ||
      (rc = stage(g_ctx.in_ranges, ranges, n * 128)) || (rc = g_ctx.out_grids.ensure(n_ev_at + (size_t)n_flights * 4)) ||
      (n_queries && ((rc = stage(g_ctx.in_kind, queries, (size_t)n_queries * sizeof(uqs_query))) ||
                     (rc = g_ctx.in_t.ensure((size_t)n_queries * 4)))))
    return rc;
  char* out = (char*)g_ctx.out_grids.p;
  uqs_stats local;
  if ((rc = uqs_replay_recentering_frontier_dev(p, n_flights, n_frames, (float*)g_ctx.in_x.p, (float*)g_ctx.in_y.p,
                                                (float*)g_ctx.in_yaw.p, (float*)g_ctx.in_ranges.p, (int8_t*)out,
                                                (float*)(out + origins_at), (int32_t*)(out + n_ev_at), nullptr, 0, n_queries,
                                                n_queries ? (const uqs_query*)g_ctx.in_kind.p : nullptr,
                                                n_queries ? (int32_t*)g_ctx.in_t.p : nullptr, stats ? stats : &local)))
    return rc;
  cudaError_t e = cudaSuccess;
  if (grids_out) e = cudaMemcpyAsync(grids_out, out, cells, cudaMemcpyDeviceToHost, st);
  if (e == cudaSuccess && origins_out) e = cudaMemcpyAsync(origins_out, out + origins_at, (size_t)n_flights * 8, cudaMemcpyDeviceToHost, st);
  if (e == cudaSuccess && n_queries) e = cudaMemcpyAsync(scores_out, g_ctx.in_t.p, (size_t)n_queries * 4, cudaMemcpyDeviceToHost, st);
  if (e == cudaSuccess) e = cudaStreamSynchronize(st);
  if (e != cudaSuccess) return cuda_fail(e, "uqs_replay_recentering_frontier D2H");
  return UQS_OK;
}

}  // extern "C"
