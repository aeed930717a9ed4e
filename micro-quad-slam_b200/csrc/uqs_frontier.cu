// uqs_frontier.cu -- N3 at the frame of each decision: frontier_score_dir() (uav_local_nav.c:356-385) for queries
// (flight, frame, pose), each answered against its flight's grid as it stood after that frame, inside the batch
// replay that builds the grids (uqs_replay_frontier_dev).
//
//   k_frontier_probes    query -> probes: the cells its three rays sample (same arithmetic as k_frontier_scores)
//   k_probe_keys         probe -> (bucket, frame) key for the replay engine and geometry replay_device chose
//   (CUB radix sort)     probes in bucket order, frame order inside a bucket
//   k_probe_gather       sorted probe records + bucket starts
//   (replay engines)     each probe's value read by the cell's owner between frame `frame` and the next (PROBE = true)
//   k_probe_slices       time-sliced sub-tile replays: map words -> values, before k_compose_slices
//   k_frontier_reduce    one thread per query: unknown*3 + free - occ*4 over its probes
// Recentred flights (uqs_replay_recentering_frontier_dev, uqs_next.cu): k_frontier_probes<true> samples each query at its
// flight's origin at the query's frame; k_segment_keys / k_segment_gather group the queries by segment between events
// for the segment route.
#include <climits>
#include <cmath>
#include <vector>

#include <cub/device/device_radix_sort.cuh>

#include "uqs_host.h"

namespace uqs {

// One thread per (query, ray): the cell of every sample d = step, 2 step, ... <= 2.5 (binary32 accumulation of d, :371)
// until the first off-window point (:375); the ray's remaining slots are empty (-1).  RECENTER: slot j holds query
// O.order[j] (or j), sampled in the window of its flight's last event at a frame <= its own (world_to_grid at that
// origin, off-window test included) and, with O.s_min, then moved into the flight's global frame, O.gw wide.
struct ProbeOrigins {
  const PlanEvent* events;
  const int* ev_start;
  const int2* s_min;
  const int* order;
  int gw;
};
template <bool RECENTER>
__global__ void k_frontier_probes(DevParams p, int n_queries, int s_max, const uqs_query* __restrict__ queries,
                                  int* __restrict__ cells, unsigned long long* __restrict__ domain_errors, ProbeOrigins O) {
  const long long t = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (t >= (long long)n_queries * 3) return;
  const int j = (int)(t / 3);
  const uqs_query q = queries[RECENTER && O.order ? O.order[j] : j];
  float ox = p.ox, oy = p.oy;
  int offx = 0, offy = 0, width = p.W;
  if (RECENTER) {
    const int eb = O.ev_start[q.flight];
    const int e = last_event_at(O.events, eb, O.ev_start[q.flight + 1], q.frame);
    if (e >= eb) { ox = O.events[e].ox; oy = O.events[e].oy; }
    if (O.s_min) {
      const int2 sm = O.s_min[q.flight];
      offx = (e >= eb ? O.events[e].Sx : 0) - sm.x;
      offy = (e >= eb ? O.events[e].Sy : 0) - sm.y;
      width = O.gw;
    }
  }
  int* out = cells + t * s_max;
  int k = 0;
  float sa, ca;
  if (!sincosf_glibc(frontier_ray_angle(p, q.yaw_deg, q.offset_deg, (int)(t % 3)), sa, ca)) {
    atomicAdd(domain_errors, 1ull);
  } else {
    const float step = frontier_step(p);
    for (float d = step; d <= kFrontierRange && k < s_max; d = __fadd_rn(d, step)) {
      int gx, gy;
      if (!frontier_point(p, ox, oy, q.x, q.y, d, ca, sa, gx, gy)) break;
      out[k++] = (gy + offy) * width + gx + offx;
    }
  }
  for (; k < s_max; k++) out[k] = -1;
}

// index of the first query whose flight or frame is out of range (INT_MAX: none)
__global__ void k_query_check(int n_queries, const uqs_query* __restrict__ queries, int n_flights, int n_frames, int* first_bad) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n_queries) return;
  const uqs_query q = queries[i];
  if (q.flight < 0 || q.flight >= n_flights || q.frame < 0 || q.frame >= n_frames) atomicMin(first_bad, i);
}

// key = bucket * n_frames + frame for the probes of flights [f0, f0 + nf); n_buckets * n_frames for the others
// (empty slots, other chunks), which sort behind every bucket
__global__ void k_probe_keys(int n_slots, int s_max, const uqs_query* __restrict__ queries, const int* __restrict__ cells,
                             int f0, int nf, int n_frames, int W, int slices, int gps, int sw, int sh, int nsx, int nsub,
                             unsigned long long sentinel, unsigned long long* __restrict__ keys, int* __restrict__ idx) {
  const int s = blockIdx.x * blockDim.x + threadIdx.x;
  if (s >= n_slots) return;
  const int cell = cells[s];
  const uqs_query q = queries[s / (3 * s_max)];
  const int fl = q.flight - f0;
  unsigned long long key = sentinel;
  if (cell >= 0 && fl >= 0 && fl < nf) {
    long long b = fl;
    if (slices > 0) {
      const int gy = cell / W, gx = cell - gy * W;
      b = ((long long)fl * slices + (q.frame >> 5) / gps) * nsub + (gy / sh) * nsx + gx / sw;
    }
    key = (unsigned long long)b * (unsigned long long)n_frames + (unsigned long long)q.frame;
  }
  keys[s] = key;
  idx[s] = s;
}

// sorted keys -> probe records and bucket starts (start[b] = first probe of bucket b, start[n_buckets] = probes kept)
__global__ void k_probe_gather(int n, const unsigned long long* __restrict__ keys, const int* __restrict__ idx,
                               const int* __restrict__ cells, int n_frames, int n_buckets, int per_flight,
                               int4* __restrict__ probes, int* __restrict__ start) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  const unsigned long long key = keys[i];
  const int b = (int)(key / (unsigned long long)n_frames);
  if (b < n_buckets) {
    const int slot = idx[i];
    probes[i] = make_int4((int)(key - (unsigned long long)b * n_frames), cells[slot], slot, b / per_flight);
  }
  const int bp = i ? (int)(keys[i - 1] / (unsigned long long)n_frames) : -1;
  for (int bb = bp + 1; bb <= b; bb++) start[bb] = i;
  if (i == n - 1)
    for (int bb = b + 1; bb <= n_buckets; bb++) start[bb] = n;
}

// A probe of time slice s >= 1 holds the map word of slice s up to its frame.  Its value is that map applied after
// slice 0's value (still in the grid) and the maps of slices 1..s-1, each step min(max(v + a, flo), fhi) as in
// k_compose_slices.
__global__ void k_probe_slices(ProbeArgs Q, int n_max, const int8_t* __restrict__ grids, const uint32_t* __restrict__ maps,
                               int W, int H, int S, int gps) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n_max || i >= Q.start[Q.n_buckets]) return;
  const int4 pr = Q.probes[i];
  const int s = (pr.x >> 5) / gps;
  if (s == 0) return;
  const size_t plane = (size_t)W * H;
  int v = (int)grids[(size_t)pr.w * plane + pr.y];
  const uint32_t* m = maps + (size_t)pr.w * (S - 1) * plane + pr.y;
  for (int t = 1; t <= s; t++, m += plane) {
    const uint32_t w = (t < s) ? __ldg(m) : Q.values[pr.z];
    const int flo = (int)(int8_t)(w & 0xffu), fhi = (int)(int8_t)((w >> 8) & 0xffu), a = (int)w >> 16;
    v = min(max(v + a, flo), fhi);
  }
  Q.values[pr.z] = (uint32_t)v;
}

__global__ void k_frontier_reduce(int n_queries, int s_max, const int* __restrict__ cells, const uint32_t* __restrict__ values,
                                  const int* __restrict__ order, int32_t* __restrict__ scores) {
  const int q = blockIdx.x * blockDim.x + threadIdx.x;
  if (q >= n_queries) return;
  const size_t s0 = (size_t)q * 3 * s_max;
  int score = 0;
  for (int k = 0; k < 3 * s_max; k++)
    if (cells[s0 + k] >= 0) score += frontier_weight((int)values[s0 + k]);
  scores[order ? order[q] : q] = score;
}

// query i -> (segment of its frame, i): segment e + 1 + flight follows the flight's last event e at a frame <= its own
__global__ void k_segment_keys(int n, const uqs_query* __restrict__ queries, const PlanEvent* __restrict__ events,
                               const int* __restrict__ ev_start, unsigned long long* __restrict__ keys, int* __restrict__ idx) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  const uqs_query q = queries[i];
  const int e = last_event_at(events, ev_start[q.flight], ev_start[q.flight + 1], q.frame);
  keys[i] = (unsigned long long)(e + 1 + q.flight);
  idx[i] = i;
}

// sorted (segment, query) -> the segment-local queries, their input indices and the segment starts
__global__ void k_segment_gather(int n, const unsigned long long* __restrict__ keys, const int* __restrict__ idx,
                                 const uqs_query* __restrict__ queries, const PlanEvent* __restrict__ events,
                                 const int* __restrict__ ev_start, int n_segments, uqs_query* __restrict__ local,
                                 int* __restrict__ order, int* __restrict__ start) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  const int seg = (int)keys[i];
  uqs_query q = queries[idx[i]];
  const int e = seg - 1 - q.flight;
  q.frame -= e >= ev_start[q.flight] ? events[e].frame : 0;
  q.flight = 0;
  local[i] = q;
  order[i] = idx[i];
  const int bp = i ? (int)keys[i - 1] : -1;
  for (int b = bp + 1; b <= seg; b++) start[b] = i;
  if (i == n - 1)
    for (int b = seg + 1; b <= n_segments; b++) start[b] = n;
}

static unsigned blocks_for(long long n, int threads) { return (unsigned)((n + threads - 1) / threads); }

int probe_buckets(const ProbeSet& Q, int f0, int nf, int n_frames, int W, int slices, int gps, int sw, int sh, int nsx,
                  int nsy, ProbeArgs* out) {
  cudaStream_t st = g_ctx.stream();
  Work& w = *g_ctx.w;
  const int n = (int)Q.slots();
  const int nsub = nsx * nsy;
  const long long n_buckets = slices > 0 ? (long long)nf * slices * nsub : nf;
  if (n_buckets >= INT_MAX) { set_error("%lld frontier probe buckets exceed the supported %d", n_buckets, INT_MAX - 1); return UQS_ERR_BAD_ARG; }
  const unsigned long long sentinel = (unsigned long long)n_buckets * (unsigned long long)n_frames;
  int end_bit = 1;
  while (end_bit < 64 && (sentinel >> end_bit) != 0) end_bit++;
  size_t tmp_bytes = 0;
  unsigned long long *k_in = nullptr, *k_out = nullptr;
  int *i_in = nullptr, *i_out = nullptr;
  cudaError_t e = cub::DeviceRadixSort::SortPairs(nullptr, tmp_bytes, k_in, k_out, i_in, i_out, n, 0, end_bit, st);
  if (e != cudaSuccess) return cuda_fail(e, "probe sort sizing");
  int rc;
  if ((rc = w.probe_keys.ensure((size_t)n * 24)) || (rc = w.probe_sorted.ensure((size_t)n * sizeof(int4))) ||
      (rc = w.probe_start.ensure((size_t)(n_buckets + 1) * sizeof(int))) || (rc = w.probe_tmp.ensure(tmp_bytes)))
    return rc;
  k_in = (unsigned long long*)w.probe_keys.p;
  k_out = k_in + n;
  i_in = (int*)(k_out + n);
  i_out = i_in + n;
  k_probe_keys<<<blocks_for(n, 256), 256, 0, st>>>(n, Q.s_max, Q.queries, Q.cells, f0, nf, n_frames, W, slices, gps, sw, sh, nsx,
                                                   nsub, sentinel, k_in, i_in);
  e = cudaGetLastError();
  if (e == cudaSuccess) e = cub::DeviceRadixSort::SortPairs(w.probe_tmp.p, tmp_bytes, k_in, k_out, i_in, i_out, n, 0, end_bit, st);
  if (e == cudaSuccess) {
    k_probe_gather<<<blocks_for(n, 256), 256, 0, st>>>(n, k_out, i_out, Q.cells, n_frames, (int)n_buckets,
                                                       slices > 0 ? slices * nsub : 1, (int4*)w.probe_sorted.p, (int*)w.probe_start.p);
    e = cudaGetLastError();
  }
  if (e != cudaSuccess) return cuda_fail(e, "frontier probe buckets");
  g_ctx.launches += 3;                                  // keys, gather, and (at least) one sort pass
  out->probes = (const int4*)w.probe_sorted.p;
  out->start = (const int*)w.probe_start.p;
  out->values = Q.values;
  out->n_buckets = (int)n_buckets;
  return UQS_OK;
}

int probe_resolve_slices(const ProbeArgs& A, int n_probes_max, const int8_t* grids, const uint32_t* maps, int W, int H,
                         int slices, int gps) {
  k_probe_slices<<<blocks_for(n_probes_max, 256), 256, 0, g_ctx.stream()>>>(A, n_probes_max, grids, maps, W, H, slices, gps);
  const cudaError_t e = cudaGetLastError();
  if (e != cudaSuccess) return cuda_fail(e, "k_probe_slices");
  g_ctx.launches += 1;
  return UQS_OK;
}

// Samples per frontier ray: the reference's loop (:371) run in binary32 on the host.  Every query's ray has at most
// this many, whatever its pose, so query q owns 3 * s_max fixed slots.  -1 when d stops growing or the count is absurd.
static int frontier_samples(float res) {
  volatile float step = res;
  step = step * 2.0f;
  int n = 0;
  for (volatile float d = step; d <= 2.5f; ) {
    const float nd = d + step;
    if (!(nd > d) || ++n > (1 << 20)) return -1;
    d = nd;
  }
  return n;
}

int frontier_queries_begin(const char* who, const uqs_params* p, int n_flights, int n_frames, int n_queries,
                           const uqs_query* queries, ProbeSet* Q, unsigned long long** dom) {
  const int s_max = frontier_samples(p->res_m);
  if (s_max < 0 || (long long)n_queries * 3 * s_max >= INT_MAX) {
    set_error("%s: %d queries of %d samples per ray exceed the supported probe count", who, n_queries, s_max);
    return UQS_ERR_BAD_ARG;
  }
  cudaStream_t st = g_ctx.stream();
  int rc;
  if ((rc = g_ctx.w->counters.ensure(64 * sizeof(unsigned long long)))) return rc;
  *dom = (unsigned long long*)g_ctx.w->counters.p + 48;
  int* first_bad = (int*)((unsigned long long*)g_ctx.w->counters.p + 49);
  // the queries are checked before anything is written
  int h_bad = INT_MAX;
  cudaError_t e = cudaMemcpyAsync(first_bad, &h_bad, sizeof(int), cudaMemcpyHostToDevice, st);
  if (e == cudaSuccess) {
    k_query_check<<<blocks_for(n_queries, 256), 256, 0, st>>>(n_queries, queries, n_flights, n_frames, first_bad);
    e = cudaGetLastError();
  }
  if (e == cudaSuccess) e = cudaMemcpyAsync(&h_bad, first_bad, sizeof(int), cudaMemcpyDeviceToHost, st);
  if (e == cudaSuccess) e = cudaStreamSynchronize(st);
  if (e != cudaSuccess) return cuda_fail(e, "k_query_check");
  g_ctx.launches += 1;
  if (h_bad != INT_MAX) {
    uqs_query q;
    e = cudaMemcpy(&q, queries + h_bad, sizeof(q), cudaMemcpyDeviceToHost);
    if (e != cudaSuccess) return cuda_fail(e, "query D2H");
    set_error("query %d: flight %d outside [0, %d) or frame %d outside [0, %d)", h_bad, q.flight, n_flights, q.frame, n_frames);
    return UQS_ERR_BAD_ARG;
  }
  Q->n_queries = n_queries;
  Q->s_max = s_max;
  Q->queries = queries;
  const size_t slots = Q->slots();
  if ((rc = g_ctx.w->probe_slots.ensure(slots * 8 + 16))) return rc;
  int* cells = (int*)g_ctx.w->probe_slots.p;
  Q->cells = cells;
  Q->values = (uint32_t*)(cells + slots);
  if ((e = zero_async(*dom, sizeof(unsigned long long), st)) != cudaSuccess) return cuda_fail(e, "memset");
  return UQS_OK;
}

int frontier_probes_recentered(const DevParams& dp, const ProbeSet& Q, const uqs_query* queries, const int* order,
                               const PlanEvent* events, const int* ev_start, const int2* s_min, int gw,
                               unsigned long long* dom) {
  const ProbeOrigins O = { events, ev_start, s_min, order, gw };
  k_frontier_probes<true><<<blocks_for((long long)Q.n_queries * 3, 128), 128, 0, g_ctx.stream()>>>(
      dp, Q.n_queries, Q.s_max, queries, Q.cells, dom, O);
  const cudaError_t e = cudaGetLastError();
  if (e != cudaSuccess) return cuda_fail(e, "k_frontier_probes");
  g_ctx.launches += 1;
  return UQS_OK;
}

int frontier_queries_by_segment(int n_queries, const uqs_query* queries, const PlanEvent* events, const int* ev_start,
                                int n_segments, uqs_query* local, int* order, std::vector<int>* seg_start) {
  cudaStream_t st = g_ctx.stream();
  Work& w = *g_ctx.w;
  const int n = n_queries;
  int end_bit = 1;
  while (end_bit < 64 && ((unsigned long long)n_segments >> end_bit) != 0) end_bit++;
  size_t tmp_bytes = 0;
  unsigned long long *k_in = nullptr, *k_out = nullptr;
  int *i_in = nullptr, *i_out = nullptr;
  cudaError_t e = cub::DeviceRadixSort::SortPairs(nullptr, tmp_bytes, k_in, k_out, i_in, i_out, n, 0, end_bit, st);
  if (e != cudaSuccess) return cuda_fail(e, "segment sort sizing");
  int rc;
  if ((rc = w.probe_keys.ensure((size_t)n * 24)) || (rc = w.probe_tmp.ensure(tmp_bytes)) ||
      (rc = w.probe_start.ensure(((size_t)n_segments + 1) * sizeof(int))))
    return rc;
  k_in = (unsigned long long*)w.probe_keys.p;
  k_out = k_in + n;
  i_in = (int*)(k_out + n);
  i_out = i_in + n;
  int* d_start = (int*)w.probe_start.p;
  k_segment_keys<<<blocks_for(n, 256), 256, 0, st>>>(n, queries, events, ev_start, k_in, i_in);
  e = cudaGetLastError();
  if (e == cudaSuccess) e = cub::DeviceRadixSort::SortPairs(w.probe_tmp.p, tmp_bytes, k_in, k_out, i_in, i_out, n, 0, end_bit, st);
  if (e == cudaSuccess) {
    k_segment_gather<<<blocks_for(n, 256), 256, 0, st>>>(n, k_out, i_out, queries, events, ev_start, n_segments, local, order,
                                                         d_start);
    e = cudaGetLastError();
  }
  seg_start->resize((size_t)n_segments + 1);
  if (e == cudaSuccess)
    e = cudaMemcpyAsync(seg_start->data(), d_start, seg_start->size() * sizeof(int), cudaMemcpyDeviceToHost, st);
  if (e == cudaSuccess) e = cudaStreamSynchronize(st);
  if (e != cudaSuccess) return cuda_fail(e, "frontier queries by segment");
  g_ctx.launches += 3;
  return UQS_OK;
}

int frontier_queries_end(const ProbeSet& Q, const int* order, int32_t* scores, unsigned long long* dom, uqs_stats* stats,
                         uint64_t frames) {
  cudaStream_t st = g_ctx.stream();
  cudaError_t e = cudaSuccess;
  if (Q.s_max > 0)
    k_frontier_reduce<<<blocks_for(Q.n_queries, 128), 128, 0, st>>>(Q.n_queries, Q.s_max, Q.cells, Q.values, order, scores);
  else e = zero_async(scores, (size_t)Q.n_queries * sizeof(int32_t), st);
  if (e == cudaSuccess) e = cudaGetLastError();
  if (e != cudaSuccess) return cuda_fail(e, "k_frontier_reduce");
  g_ctx.launches += 1;
  if (!stats) return UQS_OK;
  int rc;
  if ((rc = fetch_stats(stats, frames))) return rc;
  unsigned long long hdom = 0;
  e = cudaMemcpyAsync(&hdom, dom, sizeof(hdom), cudaMemcpyDeviceToHost, st);
  if (e == cudaSuccess) e = cudaStreamSynchronize(st);
  if (e != cudaSuccess) return cuda_fail(e, "frontier domain D2H");
  if (hdom) { set_error("%llu frontier rays outside the restated sincosf domain", hdom); return UQS_ERR_DOMAIN; }
  return UQS_OK;
}

}  // namespace uqs

using namespace uqs;

extern "C" {

int uqs_replay_frontier_dev(const uqs_params* p, int n_flights, int n_frames, const float* x, const float* y, const float* yaw,
                            const float* ranges, int8_t* grids, int accumulate, int n_queries, const uqs_query* queries,
                            int32_t* scores, uqs_stats* stats) {
  int rc = check_ready();
  if (rc) return rc;
  DevParams dp;
  if ((rc = make_dev_params(p, &dp))) return rc;
  if (n_flights <= 0 || n_frames <= 0 || !x || !y || !yaw || !ranges || !grids || n_queries < 0 ||
      (n_queries > 0 && (!queries || !scores))) {
    set_error("uqs_replay_frontier_dev: NULL pointer or bad size");
    return UQS_ERR_BAD_ARG;
  }
  if (n_queries == 0) {
    if ((rc = replay_device(dp, n_flights, n_frames, x, y, yaw, ranges, nullptr, grids, accumulate, 0, p->H, true))) return rc;
    return fetch_stats(stats, (uint64_t)n_flights * n_frames);
  }
  ProbeSet Q;
  unsigned long long* dom = nullptr;
  if ((rc = frontier_queries_begin("uqs_replay_frontier_dev", p, n_flights, n_frames, n_queries, queries, &Q, &dom))) return rc;
  if (Q.s_max > 0) {
    k_frontier_probes<false><<<blocks_for((long long)n_queries * 3, 128), 128, 0, g_ctx.stream()>>>(dp, n_queries, Q.s_max, queries,
                                                                                                   Q.cells, dom,
                                                                                                   ProbeOrigins{});
    const cudaError_t e = cudaGetLastError();
    if (e != cudaSuccess) return cuda_fail(e, "k_frontier_probes");
    g_ctx.launches += 2;
  }
  // (a step longer than 2.5 m samples nothing: every score is 0 and the replay is the plain one)
  if ((rc = replay_device(dp, n_flights, n_frames, x, y, yaw, ranges, nullptr, grids, accumulate, 0, p->H, true,
                          Q.s_max > 0 ? &Q : nullptr)))
    return rc;
  return frontier_queries_end(Q, nullptr, scores, dom, stats, (uint64_t)n_flights * n_frames);
}

int uqs_replay_frontier(const uqs_params* p, int n_flights, int n_frames, const float* x, const float* y, const float* yaw,
                        const float* ranges, int8_t* grids_out, int n_queries, const uqs_query* queries, int32_t* scores_out,
                        uqs_stats* stats) {
  int rc = check_ready();
  if (rc) return rc;
  if (!p || n_flights <= 0 || n_frames <= 0 || !x || !y || !yaw || !ranges || n_queries < 0 ||
      (n_queries > 0 && (!queries || !scores_out))) {
    set_error("uqs_replay_frontier: NULL pointer or bad size");
    return UQS_ERR_BAD_ARG;
  }
  cudaStream_t st = g_ctx.stream();
  const size_t n = (size_t)n_flights * n_frames, cells = (size_t)n_flights * p->W * p->H;
  auto up = [&](DevBuf& b, const void* src, size_t bytes) -> int {
    const int r = b.ensure(bytes);
    if (r) return r;
    const cudaError_t e = cudaMemcpyAsync(b.p, src, bytes, cudaMemcpyHostToDevice, st);
    return e == cudaSuccess ? UQS_OK : cuda_fail(e, "H2D");
  };
  if ((rc = up(g_ctx.in_x, x, n * 4)) || (rc = up(g_ctx.in_y, y, n * 4)) || (rc = up(g_ctx.in_yaw, yaw, n * 4)) ||
      (rc = up(g_ctx.in_ranges, ranges, n * 128)) || (rc = g_ctx.out_grids.ensure(cells)) ||
      (n_queries && ((rc = up(g_ctx.in_kind, queries, (size_t)n_queries * sizeof(uqs_query))) ||
                     (rc = g_ctx.in_t.ensure((size_t)n_queries * 4)))))
    return rc;
  uqs_stats local;
  if ((rc = uqs_replay_frontier_dev(p, n_flights, n_frames, (float*)g_ctx.in_x.p, (float*)g_ctx.in_y.p, (float*)g_ctx.in_yaw.p,
                                    (float*)g_ctx.in_ranges.p, (int8_t*)g_ctx.out_grids.p, 0, n_queries,
                                    n_queries ? (const uqs_query*)g_ctx.in_kind.p : nullptr,
                                    n_queries ? (int32_t*)g_ctx.in_t.p : nullptr, stats ? stats : &local)))
    return rc;
  cudaError_t e = cudaSuccess;
  if (grids_out) e = cudaMemcpyAsync(grids_out, g_ctx.out_grids.p, cells, cudaMemcpyDeviceToHost, st);
  if (e == cudaSuccess && n_queries) e = cudaMemcpyAsync(scores_out, g_ctx.in_t.p, (size_t)n_queries * 4, cudaMemcpyDeviceToHost, st);
  if (e == cudaSuccess) e = cudaStreamSynchronize(st);
  if (e != cudaSuccess) return cuda_fail(e, "uqs_replay_frontier D2H");
  return UQS_OK;
}

}  // extern "C"
