// uqs_kernels.cu -- the CUDA kernels of the mapping path (sm_100a).
//
//   k_pose_increments / k_pose_chain / k_pose_scan   P0  (builder-defined, DESIGN.md)
//   k_ray_setup        map_update_from_beams() up to the two world_to_grid() calls
//                      (uav_local_nav.c:280-303, :243-244): one thread per beam, one
//                      warp per frame, one 1024-thread CTA per group of 32 frames
//   k_replay_tiles     raycast_update()'s cell loop (uav_local_nav.c:246-277) for whole
//                      logs: persistent warps, each OWNING a sub-tile of one grid in
//                      shared memory and applying, in reference order, exactly the
//                      cell updates that fall inside it
//
// Exactness (SURVEY.md 0.4): the reference clamps after every single update, so
// updates to one cell do not commute.  k_replay_tiles never reorders them: a cell
// has exactly one owner warp, that warp walks frames in log order and beams in
// (d,c) order, and the cells of one ray are distinct, so the 32 lanes of the warp
// can apply one ray's cells at once with plain byte read-modify-writes -- no
// atomics, no races, bit-identical to the sequential loop.
#include <algorithm>
#include <cstdio>

#include "uqs_kernels.cuh"

namespace uqs {

// ===========================================================================
// P0: dead reckoning
// ===========================================================================

// increment of sample i (i >= 1); sample 0 has increment 0.  All binary32, RN, no contraction.
__global__ void k_pose_increments(long long total, int n_samples, const uint32_t* __restrict__ t_ms,
                                  const float* __restrict__ rate_x, const float* __restrict__ rate_y,
                                  const float* __restrict__ h_m, const float* __restrict__ yaw_deg,
                                  const uint8_t* __restrict__ q, float deg2rad,
                                  float* __restrict__ inc_n, float* __restrict__ inc_e,
                                  unsigned long long* __restrict__ /*unused*/) {
  const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= total) return;
  const int s = (int)(i % n_samples);
  float dn = 0.0f, de = 0.0f;
  if (s > 0) {
    const float rx = rate_x[i], ry = rate_y[i], h = h_m[i], yw = yaw_deg[i];
    if (q[i] >= 50 && !isnan(rx) && !isnan(ry) && !isnan(h) && !isnan(yw)) {
      const float dt = __fmul_rn((float)(t_ms[i] - t_ms[i - 1]), 0.001f);
      const float vbx = __fmul_rn(rx, h);
      const float vby = __fmul_rn(ry, h);
      const float a = __fmul_rn(yw, deg2rad);
      float sn, cs;
      sincosf_glibc(a, sn, cs);                                  // every float: Inf yaw gives NaN poses, like libm
      const float vn = __fsub_rn(__fmul_rn(vbx, cs), __fmul_rn(vby, sn));
      const float ve = __fadd_rn(__fmul_rn(vbx, sn), __fmul_rn(vby, cs));
      dn = __fmul_rn(vn, dt);
      de = __fmul_rn(ve, dt);
    }
  }
  inc_n[i] = dn;
  inc_e[i] = de;
}

// One warp per flight replays the summation in sample order.  The order is fixed by the spec (and by bit-exactness:
// binary32 addition is not associative), so the sum itself is a serial chain of dependent FADDs -- 4 cycles each --
// and everything else is arranged so that the chain never waits: the 32 lanes stage 256 increments at a time in
// shared memory (coalesced loads, issued one chunk ahead so that their latency hides behind the chain of the
// previous chunk), lane 0 runs the chain over them with vector loads and writes the running sums back in place, and
// all lanes store the 256 poses coalesced.  x and y are two independent chains interleaved in the same lane.
// One long log (config 2: 360 000 samples, a single warp on the whole chip): 4.6 ms with the former shuffle
// broadcast (one global-load latency per 32 samples on the critical path) -> measured value in profiles/.
constexpr int kChainChunk = 256;              // samples per staged chunk (8 per lane)
constexpr int kChainWarps = 4;                // warps (= flights) per block

__global__ void __launch_bounds__(kChainWarps * 32)
k_pose_chain(int n_flights, int n_samples, const float* __restrict__ inc_n,
             const float* __restrict__ inc_e, float* __restrict__ xo,
             float* __restrict__ yo) {
  __shared__ __align__(16) float s_n[kChainWarps][kChainChunk], s_e[kChainWarps][kChainChunk];
  const int wib = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int flight = blockIdx.x * kChainWarps + wib;
  if (flight >= n_flights) return;
  const size_t base = (size_t)flight * n_samples;
  float* sn = s_n[wib];
  float* se = s_e[wib];
  constexpr int PER = kChainChunk / 32;
  float rn[PER], re[PER];
  auto fetch = [&](int s0) {
#pragma unroll
    for (int u = 0; u < PER; u++) {
      const int s = s0 + u * 32 + lane;
      rn[u] = (s < n_samples) ? __ldg(&inc_n[base + s]) : 0.0f;
      re[u] = (s < n_samples) ? __ldg(&inc_e[base + s]) : 0.0f;
    }
  };
  fetch(0);
  float px = 0.0f, py = 0.0f;
  for (int s0 = 0; s0 < n_samples; s0 += kChainChunk) {
#pragma unroll
    for (int u = 0; u < PER; u++) { sn[u * 32 + lane] = rn[u]; se[u * 32 + lane] = re[u]; }
    if (s0 + kChainChunk < n_samples) fetch(s0 + kChainChunk);     // in flight while lane 0 works through this chunk
    __syncwarp();
    if (lane == 0) {
      // the whole chunk is walked (padding past the end of the log holds zeros: harmless adds); the shared-memory loads
      // run two groups of four ahead of the adds so that their latency (~29 cycles) never sits on the chain
      const float4* vn = reinterpret_cast<const float4*>(sn);
      const float4* ve = reinterpret_cast<const float4*>(se);
      float4 a0 = vn[0], b0 = ve[0], a1 = vn[1], b1 = ve[1];
#pragma unroll 4
      for (int g = 0; g < kChainChunk / 4; g++) {
        const int gn = min(g + 2, kChainChunk / 4 - 1);
        const float4 a2 = vn[gn], b2 = ve[gn];
        float4 a = a0, b = b0;
        a.x = px = __fadd_rn(px, a.x); b.x = py = __fadd_rn(py, b.x);
        a.y = px = __fadd_rn(px, a.y); b.y = py = __fadd_rn(py, b.y);
        a.z = px = __fadd_rn(px, a.z); b.z = py = __fadd_rn(py, b.z);
        a.w = px = __fadd_rn(px, a.w); b.w = py = __fadd_rn(py, b.w);
        reinterpret_cast<float4*>(sn)[g] = a;
        reinterpret_cast<float4*>(se)[g] = b;
        a0 = a1; b0 = b1; a1 = a2; b1 = b2;
      }
    }
    __syncwarp();
#pragma unroll
    for (int u = 0; u < PER; u++) {
      const int s = s0 + u * 32 + lane;
      if (s < n_samples) { xo[base + s] = sn[u * 32 + lane]; yo[base + s] = se[u * 32 + lane]; }
    }
    __syncwarp();                                                  // the chunk is rewritten next turn
  }
}

// Throughput variant: single-pass chained scan with decoupled look-back, binary64
// accumulation, one partition of kScanTile samples per CTA.  state[] per partition:
// flag (0 none, 1 aggregate, 2 inclusive prefix) + two doubles, published with
// __threadfence().  Partitions are claimed through an atomic ticket so that a
// partition's predecessors are always already running.
constexpr int kScanThreads = 256;
constexpr int kScanItems = 8;
constexpr int kScanTile = kScanThreads * kScanItems;

struct ScanState { double agg_n, agg_e, inc_n, inc_e; int flag; int pad; };

__global__ void __launch_bounds__(kScanThreads)
k_pose_scan(int n_flights, int n_samples, int parts_per_flight, const float* __restrict__ inc_n,
            const float* __restrict__ inc_e, float* __restrict__ xo, float* __restrict__ yo,
            volatile ScanState* state, unsigned int* ticket) {
  __shared__ unsigned int s_part;
  __shared__ double s_wn[kScanThreads / 32], s_we[kScanThreads / 32];
  __shared__ double s_prefix_n, s_prefix_e;
  if (threadIdx.x == 0) s_part = atomicAdd(ticket, 1u);
  __syncthreads();
  const unsigned int part = s_part;
  if (part >= (unsigned)(n_flights * parts_per_flight)) return;
  const int flight = part / parts_per_flight, pf = part % parts_per_flight;
  const size_t base = (size_t)flight * n_samples;
  const int s_begin = pf * kScanTile + threadIdx.x * kScanItems;

  double vn[kScanItems], ve[kScanItems];
  double tn = 0.0, te = 0.0;
#pragma unroll
  for (int k = 0; k < kScanItems; k++) {
    const int s = s_begin + k;
    const double a = (s < n_samples) ? (double)inc_n[base + s] : 0.0;
    const double b = (s < n_samples) ? (double)inc_e[base + s] : 0.0;
    tn += a; te += b;
    vn[k] = tn; ve[k] = te;
  }
  // warp inclusive scan of thread totals
  const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5;
  double wn = tn, we = te;
#pragma unroll
  for (int o = 1; o < 32; o <<= 1) {
    const double un = __shfl_up_sync(0xffffffffu, wn, o), ue = __shfl_up_sync(0xffffffffu, we, o);
    if (lane >= o) { wn += un; we += ue; }
  }
  if (lane == 31) { s_wn[wid] = wn; s_we[wid] = we; }
  __syncthreads();
  double off_n = 0.0, off_e = 0.0;
  for (int w = 0; w < wid; w++) { off_n += s_wn[w]; off_e += s_we[w]; }
  const double excl_n = off_n + wn - tn, excl_e = off_e + we - te;   // exclusive thread prefix in tile

  if (threadIdx.x == kScanThreads - 1) {
    const double agg_n = off_n + wn, agg_e = off_e + we;
    double pre_n = 0.0, pre_e = 0.0;
    if (pf == 0) {
      state[part].inc_n = agg_n; state[part].inc_e = agg_e;
      __threadfence();
      state[part].flag = 2;
    } else {
      state[part].agg_n = agg_n; state[part].agg_e = agg_e;
      __threadfence();
      state[part].flag = 1;
      // look back over predecessors of the same flight
      int p = (int)part - 1;
      for (;;) {
        int f;
        while ((f = state[p].flag) == 0) { }
        __threadfence();
        if (f == 2) { pre_n += state[p].inc_n; pre_e += state[p].inc_e; break; }
        pre_n += state[p].agg_n; pre_e += state[p].agg_e;
        p--;
      }
      state[part].inc_n = pre_n + agg_n; state[part].inc_e = pre_e + agg_e;
      __threadfence();
      state[part].flag = 2;
    }
    s_prefix_n = pre_n; s_prefix_e = pre_e;
  }
  __syncthreads();
  const double bn = s_prefix_n + excl_n, be = s_prefix_e + excl_e;
#pragma unroll
  for (int k = 0; k < kScanItems; k++) {
    const int s = s_begin + k;
    if (s < n_samples) {
      xo[base + s] = (float)(bn + vn[k]);
      yo[base + s] = (float)(be + ve[k]);
    }
  }
}

int pose_scan_tile() { return kScanTile; }
int pose_scan_threads() { return kScanThreads; }
size_t pose_scan_state_bytes() { return sizeof(ScanState); }

// ===========================================================================
// ray set-up
// ===========================================================================
//
// TMA (bulk async copy) + mbarrier: the 4 KB of range readings of a block's 32 frames are one contiguous
// span of the log; one thread starts the copy into shared memory, every warp picks its 128 bytes up there.
__device__ __forceinline__ void mbar_init(uint32_t bar, uint32_t count) {
  asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(bar), "r"(count) : "memory");
  asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
}
__device__ __forceinline__ void bulk_load_g2s(uint32_t dst, const void* src, uint32_t bytes, uint32_t bar) {
  asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(bar), "r"(bytes) : "memory");
  asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(dst), "l"(src),
               "r"(bytes), "r"(bar)
               : "memory");
}
__device__ __forceinline__ void mbar_wait(uint32_t bar, uint32_t parity) {
  asm volatile(
      "{\n"
      ".reg .pred p;\n"
      "UQS_WAIT:\n"
      "mbarrier.try_wait.parity.shared::cta.b64 p, [%0], %1;\n"
      "@!p bra UQS_WAIT;\n"
      "}\n" ::"r"(bar),
      "r"(parity)
      : "memory");
}

// grid = (groups_per_flight, n_flights); block = 1024 = 32 frames x 32 beams.
// kind == nullptr: every entry is a frame (pose + 32 ranges).
// kind[i] == 1   : entry i is one raw ray raycast_update(x0,y0,x1,y1,hit) stored as
//                  x=x0, y=y0, yaw=x1, ranges[0]=y1, ranges[1]=hit (drop-in symbol only).
__global__ void __launch_bounds__(1024, 2)
k_ray_setup(const __grid_constant__ DevParams p, int n_frames, const float* __restrict__ x,
            const float* __restrict__ y, const float* __restrict__ yaw_deg,
            const float* __restrict__ ranges, const uint8_t* __restrict__ kind, int want_k0,
            const uint32_t* __restrict__ inv_table, uint4* __restrict__ frames, uint2* __restrict__ groups, uint2* __restrict__ rays,
            unsigned long long* __restrict__ stats /* [4]: U, accepted, skipped, domain */) {
  __shared__ __align__(128) float s_rng[32 * 32];
  __shared__ __align__(8) unsigned long long s_bar;
  __shared__ int s_box[4][32];
  __shared__ unsigned s_cnt[2][32];
  __shared__ int s_org[32][2];
  const int lane = threadIdx.x & 31, w = threadIdx.x >> 5;
  const int flight = blockIdx.y, g = blockIdx.x, groups_per_flight = gridDim.x;
  const int f = g * 32 + w;
  const size_t fbase = (size_t)flight * n_frames;
  const int nfr = min(32, n_frames - g * 32);                     // frames of this block

  // stage the block's range readings: one bulk copy (needs 16-byte alignment; plain loads otherwise).
  // The log holds them as float metres (128 B per frame) or as u16 millimetres (64 B per frame).
  const bool u16 = p.ranges_u16 != 0;
  const unsigned rbytes = u16 ? 64u : 128u;
  const unsigned char* ranges_b = reinterpret_cast<const unsigned char*>(ranges);
  const unsigned char* blk_ranges = ranges_b + (fbase + (size_t)g * 32) * rbytes;
  const bool staged = (reinterpret_cast<size_t>(ranges) & 15) == 0;
  const uint32_t bar_sa = (uint32_t)__cvta_generic_to_shared(&s_bar);
  if (staged) {
    if (threadIdx.x == 0) {
      mbar_init(bar_sa, 1);
      bulk_load_g2s((uint32_t)__cvta_generic_to_shared(s_rng), blk_ranges, (uint32_t)nfr * rbytes, bar_sa);
    }
    __syncthreads();                                               // the barrier object is visible to every waiter
  }

  int xmin = 0x7fff, xmax = 0, ymin = 0x7fff, ymax = 0;
  unsigned cells = 0;
  int accepted = 0, skipped = 0, domain = 0;

  // the start cell is per frame, not per beam: the last warp computes it for the block's 32 frames
  // (lane = frame) while the others are busy with their end points
  if (w == 31) {
    int ox = -1, oy = -1;
    const int fo = g * 32 + lane;
    if (fo < n_frames && !world_to_grid(p, x[fbase + fo], y[fbase + fo], ox, oy)) ox = oy = -1;
    s_org[lane][0] = ox;
    s_org[lane][1] = oy;
  }

  // end point of the beam (everything that does not need the start cell) before the block barrier
  const bool live = f < n_frames;
  const size_t fi = fbase + (live ? f : 0);
  float ex = 0.f, ey = 0.f;
  bool hit = false, raw = false;
  int st = 0;
  if (live) {
    const float px = x[fi], py = y[fi], third = yaw_deg[fi];
    raw = kind != nullptr && kind[fi] == 1;
    if (staged) mbar_wait(bar_sa, 0);
    const unsigned char* rb = staged ? reinterpret_cast<const unsigned char*>(s_rng) + (size_t)w * rbytes : ranges_b + fi * rbytes;
    const float* rr = reinterpret_cast<const float*>(rb);
    if (!raw) {
      const float dist = u16 ? range_from_mm(reinterpret_cast<const uint16_t*>(rb)[lane]) : rr[lane];
      st = beam_endpoint(p, px, py, third, dist, lane, ex, ey, hit);
    } else {
      st = (lane == 0) ? 1 : 0;
      ex = third;
      ey = rr[0];
      hit = rr[1] != 0.0f;
    }
  }
  __syncthreads();

  if (live) {
    const int gx0 = s_org[w][0], gy0 = s_org[w][1];
    const bool have_o = gx0 >= 0;
    uint32_t w0 = 0, w1 = 0;
    if (st < 0) {
      domain = 1;
    } else if (st > 0 && have_o) {
      int gx1, gy1;
      if (world_to_grid(p, ex, ey, gx1, gy1)) {
        const int dx = gx1 - gx0, dy = gy1 - gy0;
        const int m = max(abs(dx), abs(dy));
        if (m > kMaxRayCells) {
          domain = 1;
        } else {
          w0 = ((uint32_t)dx & 0xfffu) | (((uint32_t)dy & 0xfffu) << 12) | (hit ? kRayHit : 0u) |
               kRayValid;
          w1 = __ldg(&inv_table[m]);                           // ceil(2^31 / m), 0 for m == 0
          xmin = min(gx0, gx1); xmax = max(gx0, gx1);
          ymin = min(gy0, gy1); ymax = max(gy0, gy1);
          cells = (unsigned)m + 1u;
          accepted = 1;
        }
      }
    }
    if (!accepted && !domain && !(raw && lane != 0)) skipped = 1;
    rays[fi * 32 + lane] = make_uint2(w0, w1);

    // K0: two accepted beams of this frame can share a cell only at steps k < K0 (DESIGN.md,
    // "same-k lemma" and ring coordinate).  sigma = position of the beam's direction on the
    // unit max-norm ring, in [0,8); cells of step k sit within 1/2 of k*sigma on the ring of
    // radius k, so beams i,j are apart for every k > 1/|sigma_i - sigma_j|.  Conservative
    // float arithmetic (K0 may only be too large) -- it gates a fast path, never a result.
    int k0 = 0;
    bool frame_sorted = false;
    if (want_k0) {                       // only the grid-resident engine reads K0 and the order flag
      const int dx = sext12(w0), dy = sext12(w0 >> 12);
      const int adx = abs(dx), ady = abs(dy);
      const bool xmaj = adx >= ady;
      const int m = accepted ? (xmaj ? adx : ady) : -1;
      const int n = xmaj ? ady : adx;
      const bool xpos = dx >= 0, ypos = dy >= 0;
      float ra, rb;
      if (xmaj) { ra = xpos ? (ypos ? 0.f : 8.f) : 4.f; rb = (xpos == ypos) ? 1.f : -1.f; }
      else      { ra = ypos ? 2.f : 6.f;                rb = (xpos == ypos) ? -1.f : 1.f; }
      float sigma = (m > 0) ? ra + rb * __fdividef((float)n, (float)m) : 0.f;   // feeds the conservative K0 only
      if (sigma >= 8.f) sigma -= 8.f;
      const int mmax = __reduce_max_sync(0xffffffffu, m);
      const unsigned any = __ballot_sync(0xffffffffu, m >= 0);
      const unsigned dir = __ballot_sync(0xffffffffu, m >= 1);     // beams that have a direction
      // Fast path: beams are issued in angular order, so their ring coordinates are normally sorted and the
      // closest pair is a pair of neighbours.  Dropping the per-pair length cap only enlarges the bound.
      const unsigned above = dir & ~(0xffffffffu >> (31 - lane));
      const int nxt = above ? (__ffs(above) - 1) : (__ffs(dir) - 1);
      const float sn = __shfl_sync(0xffffffffu, sigma, nxt & 31);
      const bool has_dir = m >= 1;
      float gap = sn - sigma;                                           // to the next beam, cyclically (K0 only)
      // exact order test: sigma = A + s*n/m as integers (A in {0,2,4,6,8}); sigma_i <= sigma_next  <=>
      // (A' - A)*m*m' + s'*n'*m - s*n*m' >= 0.  8 is the same direction as 0.
      int A = (int)ra, sgn_n = (rb > 0.f) ? n : -n;
      if (A == 8 && n == 0) A = 0;
      const int pk = (A << 24) | ((sgn_n & 0xfff) << 12) | (max(m, 0) & 0xfff);     // m <= 1024 < 4096
      const int pn = __shfl_sync(0xffffffffu, pk, nxt & 31);
      const int A2 = pn >> 24, n2s = (pn << 8) >> 20, m2 = pn & 0xfff;
      const int order = (A2 - A) * m * m2 + n2s * m - sgn_n * m2;
      const bool wraps = has_dir && order < 0;
      // the float gap only feeds the (conservative) K0: make it agree with the exact order first
      if (order == 0) gap = 0.f;                     // parallel beams: shared up to the shorter one's end
      else if (order < 0) gap += 8.f;                // the one passage through 8 -> 0
      gap = fmaxf(gap, 0.f);
      // circularly sorted <=> the cyclic sequence passes 8 -> 0 at most once
      const bool sorted = __popc(__ballot_sync(0xffffffffu, wraps)) <= 1;
      frame_sorted = sorted;
      if (__popc(any) >= 2) {
        if (sorted || __popc(dir) < 2) {
          int kk = 1;                                                   // the start cell is shared by all beams
          // no shared cell once k*gap > 1: steps 0..floor(1/gap) may collide (the float slack only enlarges it)
          if (has_dir && __popc(dir) >= 2) kk = (gap > 1e-4f) ? (int)(1.0f / (gap - 2e-5f)) + 1 : 0x7fffffff;
          k0 = min(__reduce_max_sync(0xffffffffu, kk), mmax + 1);
        } else {
          // beams out of angular order (very short rays quantise coarsely): exact all-pairs bound
#pragma unroll 4
          for (int j = 1; j <= 16; j++) {
            const int pl = (lane + j) & 31;
            const float sp = __shfl_sync(0xffffffffu, sigma, pl);
            const int mp = __shfl_sync(0xffffffffu, m, pl);
            float dlt = fabsf(sigma - sp);
            dlt = fminf(dlt, 8.f - dlt);
            int kk = (dlt > 1e-4f) ? (int)(1.0f / (dlt - 2e-5f)) + 1 : 0x7fffffff;
            if (m < 1 || mp < 1) kk = 1;
            kk = min(kk, min(m, mp) + 1);          // a beam has no step beyond its own length
            if (m >= 0 && mp >= 0) k0 = max(k0, kk);
          }
          k0 = __reduce_max_sync(0xffffffffu, k0);
        }
      }
      // want_k0 - 1: measurement bias (uqs_set_k0_bias), added after the cap at mmax + 1 so that it cannot overflow the
      // 0x7fffffff of parallel beams, and capped the same way (a larger K0 is always safe: more collision-checked steps)
      const int bias = want_k0 - 1;
      k0 = min(k0, mmax + 1 - bias) + bias;
    }

    xmin = __reduce_min_sync(0xffffffffu, xmin);
    xmax = __reduce_max_sync(0xffffffffu, xmax);
    ymin = __reduce_min_sync(0xffffffffu, ymin);
    ymax = __reduce_max_sync(0xffffffffu, ymax);
    if (lane == 0)
      frames[fi] = make_uint4(have_o ? ((uint32_t)gx0 | ((uint32_t)k0 << 16)) : 0u,
                              have_o ? ((uint32_t)gy0 | kFrameHasOrigin | (frame_sorted ? kFrameSorted : 0u)) : 0u,
                              (uint32_t)xmin | ((uint32_t)xmax << 16),
                              (uint32_t)ymin | ((uint32_t)ymax << 16));
  }
  // per-warp counters (two packed words), then one block-level reduce by warp 0
  const unsigned as = __reduce_add_sync(0xffffffffu, (unsigned)accepted | ((unsigned)skipped << 16));
  const unsigned cd = __reduce_add_sync(0xffffffffu, cells | ((unsigned)domain << 21));       // cells <= 32*1025 per warp
  if (lane == 0) {
    s_box[0][w] = xmin; s_box[1][w] = xmax; s_box[2][w] = ymin; s_box[3][w] = ymax;
    s_cnt[0][w] = as; s_cnt[1][w] = cd;
  }
  __syncthreads();
  if (w == 0) {
    const int bx0 = __reduce_min_sync(0xffffffffu, s_box[0][lane]);
    const int bx1 = __reduce_max_sync(0xffffffffu, s_box[1][lane]);
    const int by0 = __reduce_min_sync(0xffffffffu, s_box[2][lane]);
    const int by1 = __reduce_max_sync(0xffffffffu, s_box[3][lane]);
    const unsigned bas = __reduce_add_sync(0xffffffffu, s_cnt[0][lane]);                        // <= 1024 per field
    const unsigned long long bcd = s_cnt[1][lane];
    const unsigned bc = __reduce_add_sync(0xffffffffu, (unsigned)(bcd & 0x1fffffu));            // <= 1024*1025 < 2^21
    const unsigned bd = __reduce_add_sync(0xffffffffu, (unsigned)(bcd >> 21));
    if (lane == 0)
      groups[(size_t)flight * groups_per_flight + g] =
          make_uint2((uint32_t)bx0 | ((uint32_t)bx1 << 16), (uint32_t)by0 | ((uint32_t)by1 << 16));
    if (lane < 4) {
      const unsigned long long t = lane == 0 ? bc : (lane == 1 ? (bas & 0xffffu) : (lane == 2 ? (bas >> 16) : bd));
      if (t) atomicAdd(&stats[lane], t);
    }
  }
}

// Parity hook: end cell of every beam from the records (cells [-1,-1] when skipped).
__global__ void k_records_to_cells(long long n_frames, const uint4* __restrict__ frames,
                                   const uint2* __restrict__ rays, int32_t* __restrict__ cells,
                                   int32_t* __restrict__ origin) {
  const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n_frames * 32) return;
  const long long f = i >> 5;
  const uint4 fr = frames[f];
  const uint2 r = rays[i];
  int cx = -1, cy = -1;
  if (r.x & kRayValid) {
    cx = (int)(fr.x & 0xffffu) + sext12(r.x);
    cy = (int)(fr.y & 0xffffu) + sext12(r.x >> 12);
  }
  cells[2 * i] = cx;
  cells[2 * i + 1] = cy;
  if ((i & 31) == 0) {
    origin[2 * f] = (fr.y & kFrameHasOrigin) ? (int)(fr.x & 0xffffu) : -1;
    origin[2 * f + 1] = (fr.y & kFrameHasOrigin) ? (int)(fr.y & 0xffffu) : -1;
  }
}

__global__ void k_sincosf(size_t n, const float* __restrict__ a, float* __restrict__ s,
                          float* __restrict__ c) {
  const size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  float sn, cs;
  sincosf_glibc(a[i], sn, cs);
  s[i] = sn;
  c[i] = cs;
}

// world_to_grid() for the drop-in symbol: one thread, result in mapped host memory.
__global__ void k_world_to_grid_one(DevParams p, float wx, float wy, int* out /* [3] */) {
  int gx, gy;
  const bool ok = world_to_grid(p, wx, wy, gx, gy);
  out[0] = ok ? 1 : 0;
  out[1] = gx;
  out[2] = gy;
}

// ===========================================================================
// replay: persistent warps owning shared-memory sub-tiles
// ===========================================================================

__device__ __forceinline__ bool box_overlaps(uint32_t xlohi, uint32_t ylohi, int X0, int X1, int Y0,
                                             int Y1) {
  const int bx0 = (int)(xlohi & 0xffffu), bx1 = (int)(xlohi >> 16);
  const int by0 = (int)(ylohi & 0xffffu), by1 = (int)(ylohi >> 16);
  return bx0 < X1 && bx1 >= X0 && by0 < Y1 && by1 >= Y0;
}

// -DUQS_DEBUG_BOUNDS (make debug -> libuqs_mapping_dbg.so): every shared-memory access of the replay kernels is
// checked against the region it is meant for -- a flight's resident box, a warp's collision table, the decode ring,
// a warp's sub-tile, its candidate queue -- and traps with a message otherwise.  compute-sanitizer is closed on the
// pool this was developed on; a stray write into a neighbouring region need not show in the grids, so byte parity
// alone would not catch it.  tests/test_gpu_debug_bounds.py runs the stress and ragged cases under this build.
struct SmemRegion { uint32_t lo, hi; };
#ifdef UQS_DEBUG_BOUNDS
__device__ __noinline__ void uqs_bounds_fail(uint32_t a, uint32_t n, uint32_t lo, uint32_t hi, int line) {
  printf("UQS_DEBUG_BOUNDS: shared access [%u, %u) outside region [%u, %u) at uqs_kernels.cu:%d (block %d thread %d)\n", a, a + n,
         lo, hi, line, (int)blockIdx.x, (int)threadIdx.x);
  __trap();
}
#define UQS_CHECK(a, n, R) do { const uint32_t a_ = (a); if (a_ < (R).lo || a_ + (n) > (R).hi) uqs_bounds_fail(a_, (n), (R).lo, (R).hi, __LINE__); } while (0)
#else
#define UQS_CHECK(a, n, R) ((void)0)
#endif

// shared-memory byte access through 32-bit shared addresses (no generic->shared conversion per use)
__device__ __forceinline__ int lds_s8(uint32_t a) {
  int v;
  asm volatile("ld.shared.s8 %0, [%1];" : "=r"(v) : "r"(a) : "memory");
  return v;
}
__device__ __forceinline__ void sts_u8(uint32_t a, int v) {
  asm volatile("st.shared.u8 [%0], %1;" ::"r"(a), "r"(v) : "memory");
}
__device__ __forceinline__ uint32_t lds_u32(uint32_t a) {
  uint32_t v;
  asm volatile("ld.shared.u32 %0, [%1];" : "=r"(v) : "r"(a) : "memory");
  return v;
}
__device__ __forceinline__ void sts_u32(uint32_t a, uint32_t v) {
  asm volatile("st.shared.u32 [%0], %1;" ::"r"(a), "r"(v) : "memory");
}
__device__ __forceinline__ uint4 lds_v4(uint32_t a) {
  uint4 v;
  asm volatile("ld.shared.v4.u32 {%0,%1,%2,%3}, [%4];" : "=r"(v.x), "=r"(v.y), "=r"(v.z), "=r"(v.w) : "r"(a) : "memory");
  return v;
}
__device__ __forceinline__ void sts_v4(uint32_t a, uint32_t x, uint32_t y, uint32_t z, uint32_t w) {
  asm volatile("st.shared.v4.u32 [%0], {%1,%2,%3,%4};" ::"r"(a), "r"(x), "r"(y), "r"(z), "r"(w) : "memory");
}
// pin a kernel parameter in a register (otherwise it is re-read from the constant bank in inner loops)
__device__ __forceinline__ int in_reg(int v) {
  asm volatile("" : "+r"(v));
  return v;
}


struct TileConsts { int pitch, lo_free, lo_occ, lo_min, lo_max, end_nohit; };
struct TileRegions { SmemRegion tile, queue; };      // debug bounds of the current job (unused in release builds)

// floor(num / den) for 0 <= num < 2^22, 1 <= den <= 1024: one reciprocal multiply and a +-1 fix-up
// (num is exact in binary32; the product is within 1 of the quotient).
__device__ __forceinline__ int div_small(int num, int den) {
  int q = (int)((float)num * __frcp_rn((float)den));
  const int r = num - q * den;
  q += (r >= den) ? 1 : 0;
  q -= (r < 0) ? 1 : 0;
  return q;
}

// Candidate queue of a warp (shared memory, 64 entries, circular): rays whose bounding box meets the warp's
// sub-tile, in (frame, beam) order.  Exact clipping costs ~100 instructions whether one beam of a frame meets the
// sub-tile or all 32 do -- and on fine grids a sub-tile sees one to three beams of a frame -- so candidates of many
// frames are collected first and clipped 32 at a time.
constexpr int kQueueEntries = 64;
constexpr int kQueueBytes = kQueueEntries * 12;          // w0 (dx,dy,flags), w1 (reciprocal), origin cell: three words each
static_assert(kQueueBytes == kReplayQueueBytes, "the host sizes the queues");

// Apply, in queue (= frame, beam) order, the part of `count` <= 32 queued rays that lies inside the warp's
// sub-tile [X0,X1) x [Y0,Y1).
//   1. lane i clips entry i EXACTLY: cell k of a ray is (major0 + k*s, minor0 + s'*q(k)) with
//      q(k) = floor((k*n + m/2)/m) non-decreasing, so "inside the tile" is one interval
//      [ka, kb] of k: the major axis gives it directly, the minor axis by inverting q:
//        q(k) >= a  <=>  k >= ceil((a*m - m/2)/n),   q(k) <= b  <=>  k <= floor(((b+1)*m - m/2 - 1)/n)
//      and packs what the cell loop needs into five words;
//   2. the warp walks the surviving rays in order, lanes along the ray: the cells of one ray
//      are distinct, so plain byte read-modify-writes are race-free and in reference order.
//
// MAP = false: the tile holds int8 log-odds values (the log, or its first time slice, from a known start).
// MAP = true : the tile holds, per cell, the clamp-add MAP of a later time slice -- the function
//   x -> value after the slice's updates when the cell starts at x -- as 32 bits
//   [ a:16 | f(lo_max):8 | f(lo_min):8 ],  f(x) = min(max(x + a, f(lo_min)), f(lo_max)).
//   The two end values are ordinary saturating trajectories; a (plain sum of the deltas, saturated far
//   outside +-(lo_max-lo_min)) only matters while f(lo_min) < f(lo_max), and then it never saturated
//   (DESIGN.md section 3, "time slices").  k_compose_slices applies the maps in slice order.
template <bool MAP>
__device__ __forceinline__ void apply_queued(const TileConsts& A, const TileRegions& DR, uint32_t tile, int lane, uint32_t queue, int head,
                                             int count, int X0, int X1, int Y0, int Y1) {
  (void)DR;
  uint32_t p1, p2, p3, p4, inv_l;      // n2 | m<<16 ; cK | cQ<<16 ; ka | kb<<11 | hit<<22 ; origin address ; reciprocal
  bool live;
  {
    const uint32_t at = queue + 4u * (uint32_t)((head + lane) & (kQueueEntries - 1));
    UQS_CHECK(at, 4u, DR.queue); UQS_CHECK(at + 8u * kQueueEntries, 4u, DR.queue);
    const uint32_t w0 = lds_u32(at), org = lds_u32(at + 8u * kQueueEntries);
    inv_l = lds_u32(at + 4u * kQueueEntries);
    const int gx0 = (int)(org & 0xffffu), gy0 = (int)(org >> 16);
    const int dx = sext12(w0), dy = sext12(w0 >> 12);
    const int adx = abs(dx), ady = abs(dy);
    const bool xmaj = adx >= ady;
    const int m = xmaj ? adx : ady, n = xmaj ? ady : adx, h = m >> 1;
    const bool majpos = (xmaj ? dx : dy) >= 0, minpos = (xmaj ? dy : dx) >= 0;
    const int c0 = xmaj ? gx0 : gy0, c1 = xmaj ? gy0 : gx0;
    const int A0 = xmaj ? X0 : Y0, A1 = xmaj ? X1 : Y1;
    const int B0 = xmaj ? Y0 : X0, B1 = xmaj ? Y1 : X1;
    int ka = max(majpos ? (A0 - c0) : (c0 - (A1 - 1)), 0);
    int kb = min(majpos ? (A1 - 1 - c0) : (c0 - A0), m);
    const int qlo = minpos ? (B0 - c1) : (c1 - (B1 - 1));
    const int qhi = minpos ? (B1 - 1 - c1) : (c1 - B0);
    live = lane < count && qhi >= 0 && qlo <= n;
    if (qlo > 0 && qlo <= n) {                                   // n >= 1 here
      const int num = qlo * m - h;                               // > 0 because qlo*m >= m > h
      ka = max(ka, div_small(num + n - 1, n));
    }
    if (qhi >= 0 && qhi < n) kb = min(kb, div_small((qhi + 1) * m - h - 1, n));
    live = live && ka <= kb;
    const int pitch = A.pitch;
    const int cK = majpos ? (xmaj ? 1 : pitch) : (xmaj ? -1 : -pitch);
    const int cQ = minpos ? (xmaj ? pitch : 1) : (xmaj ? -pitch : -1);
    p1 = (uint32_t)(2 * n) | ((uint32_t)m << 16);
    p2 = ((uint32_t)cK & 0xffffu) | ((uint32_t)cQ << 16);
    p3 = (uint32_t)ka | ((uint32_t)kb << 11) | ((w0 & kRayHit) ? (1u << 22) : 0u);
    p4 = tile + ((uint32_t)((gy0 - Y0) * pitch + (gx0 - X0)) << (MAP ? 2 : 0));
  }
  unsigned active = __ballot_sync(0xffffffffu, live);
  while (active) {
    const int b = __ffs(active) - 1;
    active &= active - 1;
    const uint32_t inv = __shfl_sync(0xffffffffu, inv_l, b);
    const uint32_t q1 = __shfl_sync(0xffffffffu, p1, b);
    const uint32_t q2 = __shfl_sync(0xffffffffu, p2, b);
    const uint32_t q3 = __shfl_sync(0xffffffffu, p3, b);
    const uint32_t base = __shfl_sync(0xffffffffu, p4, b);
    const int n2 = (int)(q1 & 0xffffu), m = (int)(q1 >> 16), h2 = m & ~1;
    const int cK = (int)(short)(q2 & 0xffffu), cQ = (int)q2 >> 16;
    const int k1 = (int)((q3 >> 11) & 0x7ffu);
    const int end_delta = (q3 & (1u << 22)) ? A.lo_occ : A.end_nohit;
    for (int k = (int)(q3 & 0x7ffu) + lane; k <= k1; k += 32) {
      const int q = minor_steps(k, n2, h2, inv);
      const int delta = (k == m) ? end_delta : -A.lo_free;
      if (!MAP) {
        const uint32_t cell = base + (uint32_t)(k * cK + q * cQ);
        UQS_CHECK(cell, 1u, DR.tile);
        const int v = lds_s8(cell) + delta;
        sts_u8(cell, min(max(v, A.lo_min), A.lo_max));
      } else {
        const uint32_t cell = base + ((uint32_t)(k * cK + q * cQ) << 2);
        UQS_CHECK(cell, 4u, DR.tile);
        const uint32_t w = lds_u32(cell);
        int flo = (int)(int8_t)(w & 0xffu), fhi = (int)(int8_t)((w >> 8) & 0xffu), a = (int)w >> 16;
        flo = min(max(flo + delta, A.lo_min), A.lo_max);
        fhi = min(max(fhi + delta, A.lo_min), A.lo_max);
        a = min(max(a + delta, -30000), 30000);
        sts_u32(cell, ((uint32_t)flo & 0xffu) | (((uint32_t)fhi & 0xffu) << 8) | ((uint32_t)a << 16));
      }
    }
    __syncwarp();
  }
}

extern __shared__ __align__(16) unsigned char uqs_smem[];

// PROBE: also serves the job's frontier probes (bucket (flight, slice, sub-tile), frame order).  A probe of frame p is
// read when every ray of frames <= p that reaches the sub-tile has been applied: before the rays of the first hit frame
// g > p are queued (after a flush of the queue, which may still hold rays of frames < g), or when the job ends.
template <bool PROBE>
__global__ void __launch_bounds__(kReplayThreads)
k_replay_tiles(ReplayArgs A, ProbeArgs Q) {
  const int lane = threadIdx.x & 31;
  const int wic = threadIdx.x >> 5;
  int8_t* tile = reinterpret_cast<int8_t*>(uqs_smem) + (size_t)wic * A.tile_bytes;
  const uint32_t tile_s = (uint32_t)__cvta_generic_to_shared(tile);
  // the warp's candidate queue sits behind the CTA's tiles
  const uint32_t queue_s = (uint32_t)__cvta_generic_to_shared(uqs_smem) + (uint32_t)(kReplayWarps * A.tile_bytes + wic * kQueueBytes);
  const int lo_free = in_reg(A.lo_free), lo_occ = in_reg(A.lo_occ), lo_min = in_reg(A.lo_min), lo_max = in_reg(A.lo_max);
  const TileConsts CV = { in_reg(A.pitch), lo_free, lo_occ, lo_min, lo_max, in_reg(A.end_nohit) };     // value tiles
  const TileConsts CM = { in_reg(A.pitch_cells), lo_free, lo_occ, lo_min, lo_max, CV.end_nohit };       // map tiles
  const int subs_per_grid = A.nsx * A.nsy;
  const int S = A.slices;

  for (;;) {
    unsigned long long job = 0;
    if (lane == 0) job = atomicAdd(A.job_counter, 1ull);
    job = __shfl_sync(0xffffffffu, job, 0);
    if (job >= A.total_jobs) break;
    // job order: groups of kJobGroup flights; inside a group every flight's heaviest (most central)
    // tile first -- the launch then ends on light tiles, and a group's records stay L2-resident;
    // the S time slices of a (flight, tile) are separate jobs
    const unsigned long long per_group = (unsigned long long)kJobGroup * subs_per_grid * S;
    const int grp = (int)(job / per_group);
    const int in_grp = (int)(job - (unsigned long long)grp * per_group);
    const int gsize = min(kJobGroup, A.n_flights - grp * kJobGroup);
    const int flight = grp * kJobGroup + in_grp % gsize;
    const int rank = in_grp / gsize;
    const int slice = rank % S;
    const int sub = A.tile_order ? (int)A.tile_order[rank / S] : rank / S;
    const int X0 = (sub % A.nsx) * A.sw, Y0 = A.row0 + (sub / A.nsx) * A.sh;
    const int X1 = min(X0 + A.sw, A.W), Y1 = min(Y0 + A.sh, A.row0 + A.rows);
    const int tw = X1 - X0, th = Y1 - Y0;
    int8_t* grid = A.grids + (size_t)flight * A.W * A.H;
    const bool vec = ((A.W | X0 | tw) & 3) == 0 && ((reinterpret_cast<size_t>(grid) & 3) == 0);
    const bool map = slice > 0;
    TileRegions DR;
    DR.tile.lo = tile_s;
    DR.tile.hi = tile_s + (uint32_t)(map ? A.pitch_cells * th * 4 : A.pitch * th);
    DR.queue.lo = queue_s;
    DR.queue.hi = queue_s + (uint32_t)kQueueBytes;
    (void)DR;

    // ---- start state: the grid (accumulate), zeros, or the identity map -----------------
    if (map) {
      const uint32_t ident = ((uint32_t)lo_min & 0xffu) | (((uint32_t)lo_max & 0xffu) << 8);
      for (int i = lane; i < A.pitch_cells * th; i += 32) reinterpret_cast<uint32_t*>(tile)[i] = ident;
    } else if (A.accumulate) {
      if (vec) {
        const int wpr = tw >> 2;
        for (int i = lane; i < wpr * th; i += 32) {
          const int r = i / wpr, c = i - r * wpr;
          *reinterpret_cast<uint32_t*>(tile + r * A.pitch + 4 * c) =
              *reinterpret_cast<const uint32_t*>(grid + (size_t)(Y0 + r) * A.W + X0 + 4 * c);
        }
      } else {
        for (int i = lane; i < tw * th; i += 32) {
          const int r = i / tw, c = i - r * tw;
          tile[r * A.pitch + c] = grid[(size_t)(Y0 + r) * A.W + X0 + c];
        }
      }
    } else {
      for (int i = lane; i < (A.pitch >> 2) * th; i += 32) reinterpret_cast<uint32_t*>(tile)[i] = 0u;
    }
    __syncwarp();

    // ---- walk the slice's frames in order, culling by group and frame bounding boxes; rays whose own
    // bounding box meets the sub-tile are queued and applied 32 at a time (apply_queued) ------------------
    const uint2* groups = A.groups + (size_t)flight * A.groups_per_flight;
    const uint4* frames = A.frames + (size_t)flight * A.n_frames;
    const uint2* rays = A.rays + (size_t)flight * A.n_frames * 32;
    const int g_begin = slice * A.groups_per_slice;
    const int g_end = min(g_begin + A.groups_per_slice, A.groups_per_flight);
    int qhead = 0, qn = 0;
    auto flush = [&]() {
      const int count = min(qn, 32);
      __syncwarp();
      if (map) apply_queued<true>(CM, DR, tile_s, lane, queue_s, qhead, count, X0, X1, Y0, Y1);
      else     apply_queued<false>(CV, DR, tile_s, lane, queue_s, qhead, count, X0, X1, Y0, Y1);
      qhead = (qhead + count) & (kQueueEntries - 1);
      qn -= count;
    };
    int pb = 0, pe = 0, next_pf = 0x7fffffff;          // this job's probes [pb, pe), frame of the next one
    if (PROBE) {
      const int b = (flight * S + slice) * subs_per_grid + sub;
      pb = Q.start[b];
      pe = Q.start[b + 1];
      if (pb < pe) next_pf = Q.probes[pb].x;
    }
    // read every probe of a frame < fmax (lanes take consecutive probes; the ones taken are a prefix: frame order)
    auto serve = [&](int fmax) {
      if (next_pf >= fmax) return;
      while (qn > 0) flush();
      __syncwarp();
      while (next_pf < fmax) {
        const int i = pb + lane;
        const int4 pr = i < pe ? Q.probes[i] : make_int4(0x7fffffff, 0, 0, 0);
        const bool take = pr.x < fmax;
        if (take) {
          const int gy = pr.y / A.W, gx = pr.y - gy * A.W;
          uint32_t v;
          if (map) {
            const uint32_t cell = tile_s + ((uint32_t)((gy - Y0) * A.pitch_cells + (gx - X0)) << 2);
            UQS_CHECK(cell, 4u, DR.tile);
            v = lds_u32(cell);
          } else {
            const uint32_t cell = tile_s + (uint32_t)((gy - Y0) * A.pitch + (gx - X0));
            UQS_CHECK(cell, 1u, DR.tile);
            v = (uint32_t)lds_s8(cell);
          }
          Q.values[pr.z] = v;
        }
        pb += __popc(__ballot_sync(0xffffffffu, take));
        next_pf = pb < pe ? Q.probes[pb].x : 0x7fffffff;
      }
    };
    for (int g0 = g_begin; g0 < g_end; g0 += 32) {
      bool ghit = false;
      if (g0 + lane < g_end) {
        const uint2 gb = __ldg(&groups[g0 + lane]);
        ghit = box_overlaps(gb.x, gb.y, X0, X1, Y0, Y1);
      }
      unsigned gmask = __ballot_sync(0xffffffffu, ghit);
      while (gmask) {
        const int gi = __ffs(gmask) - 1;
        gmask &= gmask - 1;
        const int f0 = (g0 + gi) * 32;
        uint4 fr = make_uint4(0, 0, kEmptyBoxLoHi, kEmptyBoxLoHi);
        if (f0 + lane < A.n_frames) fr = __ldg(&frames[f0 + lane]);
        unsigned fmask = __ballot_sync(0xffffffffu, box_overlaps(fr.z, fr.w, X0, X1, Y0, Y1));
        // software pipeline: the next hit frame's ray records are in flight while this one is tested
        uint2 rec_next = make_uint2(0, 0);
        if (fmask) rec_next = __ldg(&rays[(size_t)(f0 + __ffs(fmask) - 1) * 32 + lane]);
        while (fmask) {
          const int fi = __ffs(fmask) - 1;
          fmask &= fmask - 1;
          const uint2 rec = rec_next;
          if (fmask) rec_next = __ldg(&rays[(size_t)(f0 + __ffs(fmask) - 1) * 32 + lane]);
          if (PROBE) serve(f0 + fi);
          const int gx0 = (int)(__shfl_sync(0xffffffffu, fr.x, fi) & 0xffffu);
          const int gy0 = (int)(__shfl_sync(0xffffffffu, fr.y, fi) & 0xffffu);
          const int ex = gx0 + sext12(rec.x), ey = gy0 + sext12(rec.x >> 12);
          const bool near = (rec.x & kRayValid) != 0u && min(gx0, ex) < X1 && max(gx0, ex) >= X0 && min(gy0, ey) < Y1 &&
                            max(gy0, ey) >= Y0;
          const unsigned nm = __ballot_sync(0xffffffffu, near);
          if (nm == 0u) continue;
          if (near) {
            const uint32_t at = queue_s + 4u * (uint32_t)((qhead + qn + __popc(nm & ((1u << lane) - 1u))) & (kQueueEntries - 1));
            UQS_CHECK(at, 4u, DR.queue); UQS_CHECK(at + 8u * kQueueEntries, 4u, DR.queue);
            sts_u32(at, rec.x);
            sts_u32(at + 4u * kQueueEntries, rec.y);
            sts_u32(at + 8u * kQueueEntries, (uint32_t)gx0 | ((uint32_t)gy0 << 16));
          }
          qn += __popc(nm);
          if (qn >= 32) flush();                               // at most 63 queued before, at most 31 after
        }
      }
    }
    while (qn > 0) flush();
    __syncwarp();
    if (PROBE) serve(0x7fffffff);                       // frames no ray of which reached the sub-tile

    // ---- write the sub-tile back: values into the grid, maps into the slice scratch ---------
    if (map) {
      uint32_t* out = A.maps + ((size_t)flight * (S - 1) + (slice - 1)) * A.W * A.H;
      for (int i = lane; i < tw * th; i += 32) {
        const int r = i / tw, c = i - r * tw;
        out[(size_t)(Y0 + r) * A.W + X0 + c] = reinterpret_cast<const uint32_t*>(tile)[r * A.pitch_cells + c];
      }
    } else if (vec) {
      const int wpr = tw >> 2;
      for (int i = lane; i < wpr * th; i += 32) {
        const int r = i / wpr, c = i - r * wpr;
        *reinterpret_cast<uint32_t*>(grid + (size_t)(Y0 + r) * A.W + X0 + 4 * c) =
            *reinterpret_cast<const uint32_t*>(tile + r * A.pitch + 4 * c);
      }
    } else {
      for (int i = lane; i < tw * th; i += 32) {
        const int r = i / tw, c = i - r * tw;
        grid[(size_t)(Y0 + r) * A.W + X0 + c] = tile[r * A.pitch + c];
      }
    }
    __syncwarp();
  }
}

// Apply the slice maps 1..S-1, in order, to the value grid left by slice 0 (rows [row0, row0+rows)).
__global__ void k_compose_slices(int8_t* __restrict__ grids, const uint32_t* __restrict__ maps, int n_flights,
                                 int W, int H, int S, int row0, int rows) {
  const size_t per = (size_t)W * rows;
  const size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= per * n_flights) return;
  const int flight = (int)(i / per);
  const size_t cell = (size_t)row0 * W + (i - (size_t)flight * per);
  int8_t* g = grids + (size_t)flight * W * H + cell;
  int v = (int)*g;
  const uint32_t* m = maps + (size_t)flight * (S - 1) * W * H + cell;
  for (int s = 1; s < S; s++, m += (size_t)W * H) {
    const uint32_t w = __ldg(m);
    const int flo = (int)(int8_t)(w & 0xffu), fhi = (int)(int8_t)((w >> 8) & 0xffu), a = (int)w >> 16;
    v = min(max(v + a, flo), fhi);
  }
  *g = (int8_t)v;
}

// ===========================================================================
// replay, whole grid resident: one CTA per flight, frame-synchronous
// ===========================================================================
//
// For grids that fit one CTA's shared memory (<= 227 KB: every 400x400 ensemble member,
// config 5 up to 476x476).  Exactness argument (DESIGN.md "same-k lemma"): all beams of a
// frame start in the same cell, and cell k of a beam is
//     ( x0 + sgn(dx)*rnd(k*|dx|/m),  y0 + sgn(dy)*rnd(k*|dy|/m) ),   rnd(u) = floor(u + 1/2),
// so two beams of one frame can only meet in a cell at the SAME step index k.  The 32 lanes
// of a warp are the 32 beams, and a warp instruction applies step k of all of them at once:
// every intra-frame collision is then inside one instruction; it is detected through a
// per-warp table indexed by ring position (match.any serialises over distinct values and is
// ~10x too slow here) and serialised in lane (= beam = reference) order.  Warps take interleaved k; steps with
// different k never touch the same cell, so warps need no ordering inside a frame, and one
// barrier per frame keeps frames in log order.
// per-lane (= per-beam) state of one frame in the resident engine
struct Beam {
  int m;            // steps 0..m (-1: beam skipped)
  int n2;           // 2 * minor extent
  uint32_t inv;     // ceil(2^31 / m)
  int sM, sN;       // byte stride of a major / minor step in the resident grid
  int ra, rb;       // ring position of step k: ra*k + rb*q
  int end_delta;    // +occ on a hit, -(free/2) otherwise
  int base;         // byte offset of the frame's origin cell
  int k0;           // shared-step bound of the frame
};

__device__ __forceinline__ Beam decode_beam(uint2 rec, uint2 org, int P, int bx0, int by0, int lo_occ, int end_nohit) {
  Beam b;
  const int dx = sext12(rec.x), dy = sext12(rec.x >> 12);
  const int adx = abs(dx), ady = abs(dy);
  const bool xmaj = adx >= ady;
  b.m = (rec.x & kRayValid) ? (xmaj ? adx : ady) : -1;
  b.n2 = 2 * (xmaj ? ady : adx);
  b.inv = rec.y;
  const bool xpos = dx >= 0, ypos = dy >= 0;
  const int sx = xpos ? 1 : -1, sy = ypos ? P : -P;
  b.sM = xmaj ? sx : sy;
  b.sN = xmaj ? sy : sx;
  if (xmaj) { b.ra = xpos ? (ypos ? 0 : 8) : 4; b.rb = (xpos == ypos) ? 1 : -1; }
  else      { b.ra = ypos ? 2 : 6;              b.rb = (xpos == ypos) ? -1 : 1; }
  b.end_delta = (rec.x & kRayHit) ? lo_occ : end_nohit;
  b.base = ((int)(org.y & 0xffffu) - by0) * P + ((int)(org.x & 0xffffu) - bx0);
  b.k0 = (int)(org.x >> 16);
  return b;
}

#ifndef UQS_UN
#define UQS_UN 3      // steps in flight per warp in the free-space loop (measured: 3 and 6 within 1 % of each other, 2/4/5 1-5 % behind)
#endif
#ifndef UQS_MINB
#define UQS_MINB 8
#endif
// FAN = 1: the free-space steps are laid out as 8 beams of ONE sensor x 4 consecutive steps per warp instruction
// (warp w serves sensor w & 3; the NW/4 warps of a sensor interleave blocks of 4 steps) instead of 32 beams x 1 step.
// The eight beams of a 63-degree fan sit in eight different rows (or columns) and the four steps of a beam in one or
// two neighbouring words, so an access costs ~1.9 shared-memory wavefronts instead of ~2.4 (simulated on the
// ensemble's geometry, tools/banksim.py; the four fans of a frame land in unrelated banks, which is what makes the
// 32-beam layout conflict), and the lanes are fuller (25 of 32 instead of 22.7: a short fan no longer idles its lanes
// through the long fans' steps).  Same cells, same order constraints: every (beam, step >= K0) cell of a frame is
// touched by exactly one lane, whichever layout enumerates them.
// PROD = 1: warp specialisation -- an extra (NW+1)-th warp does nothing but decode frames into the ring, two frames
// ahead of the NW consumer warps, and joins the per-frame barrier; the consumers never decode or load raw records.
// PROBE: also serves the flight's frontier probes (bucket = flight, frame order).  The barrier that ends frame f orders
// it before frame f + 1, so the probes of frame f are read right after it, followed by one more barrier (only when f
// has probes: the condition is the same in every thread).  Cells outside the resident box are read from the grid in
// HBM, which the kernel only writes at the end: they still hold their start value.
template <int NW, int FAN, int PROD, bool PROBE = false>
__global__ void __launch_bounds__((NW + PROD) * 32, (NW <= 4) ? (PROD ? 6 : UQS_MINB) : ((NW <= 8) ? 4 : ((NW <= 16) ? 2 : 1)))
k_replay_flights(FlightArgs A, ProbeArgs Q) {
  constexpr int NT = (NW + PROD) * 32;          // threads per CTA
  const bool producer = PROD && (threadIdx.x >> 5) == NW;
  int8_t* grid_s = reinterpret_cast<int8_t*>(uqs_smem);
  __shared__ int s_flight;
  const int lane = threadIdx.x & 31, w = threadIdx.x >> 5;
  const int P = A.pitch;
  // per-warp collision table, indexed by the position of a cell on the max-norm ring of
  // radius k (all step-k cells of a frame lie on that ring; the map cell -> position is injective)
  uint8_t* ring = reinterpret_cast<uint8_t*>(uqs_smem) + (size_t)P * A.max_rows + (size_t)w * A.ring_size;
  const int ring_mask = A.ring_size - 1;
  const uint32_t grid_sa = (uint32_t)__cvta_generic_to_shared(grid_s);
  // The constants of the step loop come back from shared memory through an opaque load: straight from the
  // parameter bank, ptxas rematerialises them as predicated LDCs inside the unrolled loop (two per step).
  __shared__ int s_const[2];
  if (threadIdx.x == 0) { s_const[0] = A.lo_free; s_const[1] = A.lo_min; }
  __syncthreads();
  const uint32_t const_sa = (uint32_t)__cvta_generic_to_shared(s_const);
  const int lo_free = (int)lds_u32(const_sa), lo_min = (int)lds_u32(const_sa + 4u), lo_max = in_reg(A.lo_max);
  const uint32_t ring_sa = (uint32_t)__cvta_generic_to_shared(ring);
  // ring of decoded frames (16-byte aligned, after the collision tables and one spare word per warp)
  const uint32_t dec_sa = (grid_sa + (uint32_t)(P * A.max_rows + NW * A.ring_size + 4 * NW) + 15u) & ~15u;

  for (;;) {
    if (threadIdx.x == 0) s_flight = (int)atomicAdd(A.job_counter, 1ull);
    __syncthreads();
    const int flight = s_flight;
    if (flight >= A.n_flights) break;
    // only the bounding box of the cells this flight can touch is kept resident (k_flight_boxes);
    // everything outside keeps its value in HBM (zero unless accumulating)
    const int4 box = A.boxes[flight];
    const int bx0 = box.x, by0 = box.y, bw = box.z - box.x, bh = box.w - box.y;
    const int8_t* grid_hbm = A.grids + (size_t)flight * A.W * A.H;
    int pb = 0, pe = 0, next_pf = 0x7fffffff;          // this flight's probes [pb, pe), frame of the next one
    if (PROBE) {
      pb = Q.start[flight];
      pe = Q.start[flight + 1];
      if (pb < pe) next_pf = Q.probes[pb].x;
    }
    if (bw <= 0 || bh <= 0) {                           // no accepted ray: every probe reads the start grid
      if (PROBE)
        for (int i = pb + threadIdx.x; i < pe; i += NT) { const int4 pr = Q.probes[i]; Q.values[pr.z] = (uint32_t)(int)grid_hbm[pr.y]; }
      __syncthreads();
      continue;
    }
    int8_t* grid_g = A.grids + (size_t)flight * A.W * A.H + (size_t)by0 * A.W + bx0;
    const bool vec = (((A.W | bx0 | bw) & 3) == 0) && ((reinterpret_cast<size_t>(grid_g) & 3) == 0);

    if (A.accumulate) {
      if (vec) {
        const int wpr = bw >> 2;
        for (int i = threadIdx.x; i < wpr * bh; i += NT) {
          const int r = i / wpr, c = i - r * wpr;
          reinterpret_cast<uint32_t*>(grid_s + r * P)[c] = reinterpret_cast<const uint32_t*>(grid_g + (size_t)r * A.W)[c];
        }
      } else {
        for (int i = threadIdx.x; i < bw * bh; i += NT) {
          const int r = i / bw, c = i - r * bw;
          grid_s[r * P + c] = grid_g[(size_t)r * A.W + c];
        }
      }
    } else {
      for (int i = threadIdx.x; i < ((P * bh) >> 2); i += NT) reinterpret_cast<uint32_t*>(grid_s)[i] = 0u;
    }
    __syncthreads();

    const uint4* frames = A.frames + (size_t)flight * A.n_frames;
    const uint2* rays = A.rays + (size_t)flight * A.n_frames * 32;
    // debug bounds: this flight's resident box, this warp's collision table, the decode ring
    const SmemRegion RG = { grid_sa, grid_sa + (uint32_t)(P * bh) };
    const SmemRegion RR = { ring_sa, ring_sa + (uint32_t)A.ring_size };
    const SmemRegion RD = { dec_sa, dec_sa + (uint32_t)((NW < kDecSlotsMax ? NW : kDecSlotsMax) * kDecSlotBytes) };
    (void)RG; (void)RR; (void)RD;
    // Beam decode is shared: warp (f mod NW) decodes frame f + L into a ring of R = min(NW, 4) slots in shared memory
    // (32 lanes x 2 x 16 B + one frame record per slot); every warp then reads its lane's 32 B per frame.  A warp
    // therefore decodes -- and loads raw records for -- only every NW-th frame, one turn ahead.
    constexpr int R = NW < kDecSlotsMax ? NW : kDecSlotsMax;      // slots of the ring (frame g lives in slot g mod R)
    constexpr int L = R / 2;                                       // frames of decode lead
    auto decode_store = [&](uint2 rec, uint2 org, int slot) {
      const Beam b = decode_beam(rec, org, P, bx0, by0, A.lo_occ, A.end_nohit);
      const int mx = __reduce_max_sync(0xffffffffu, b.m);
      const uint32_t at = dec_sa + (uint32_t)slot * kDecSlotBytes;
      // 16 bytes per beam stored as the registers the free-space loop uses (no unpacking by the NW readers)
      UQS_CHECK(at + 16u * (uint32_t)lane, 16u, RD); UQS_CHECK(at + 512u + 4u * (uint32_t)lane, 4u, RD); UQS_CHECK(at + 1024u, 16u, RD);
      sts_v4(at + 16u * (uint32_t)lane, b.inv, (uint32_t)b.n2, (uint32_t)b.m, (uint32_t)b.sM);
      // (the minor stride and what only the collision and end steps need share one word: sN | rb<0 | ra | end_delta)
      sts_u32(at + 512u + 4u * (uint32_t)lane, ((uint32_t)b.sN << 16) | (b.rb < 0 ? 0x1000u : 0u) | ((uint32_t)b.ra << 8) |
                                                   ((uint32_t)b.end_delta & 0xffu));
      if (lane == 0) sts_v4(at + 1024u, (uint32_t)b.base, (uint32_t)b.k0, (uint32_t)mx, (org.y & kFrameSorted) ? 1u : 0u);
    };
    uint2 raw_rec, raw_org;
    if (PROD) {
      if (producer) {                              // the first L frames, then the records of frame L
        for (int g = 0; g < L && g < A.n_frames; g++)
          decode_store(__ldg(&rays[(size_t)g * 32 + lane]), __ldg(reinterpret_cast<const uint2*>(&frames[g])), g);
        const int g = min(L, A.n_frames - 1);
        raw_rec = __ldg(&rays[(size_t)g * 32 + lane]);
        raw_org = __ldg(reinterpret_cast<const uint2*>(&frames[g]));
      }
    } else {
      if (w < L && w < A.n_frames)
        decode_store(__ldg(&rays[(size_t)w * 32 + lane]), __ldg(reinterpret_cast<const uint2*>(&frames[w])), w);
      // raw records of this warp's next turn (frame w + L), loaded one turn (NW frames) ahead
      const int g = min(w + L, A.n_frames - 1);
      raw_rec = __ldg(&rays[(size_t)g * 32 + lane]);
      raw_org = __ldg(reinterpret_cast<const uint2*>(&frames[g]));
    }
    __syncthreads();
    for (int f = 0; f < A.n_frames; f++) {
      if (producer) {                              // decode frame f + L while the consumers work on frame f
        const int g = f + L;
        if (g < A.n_frames) decode_store(raw_rec, raw_org, g & (R - 1));
        const int gn = min(g + 1, A.n_frames - 1);
        raw_rec = __ldg(&rays[(size_t)gn * 32 + lane]);
        raw_org = __ldg(reinterpret_cast<const uint2*>(&frames[gn]));
        __syncthreads();
        continue;
      }
      const uint32_t at = dec_sa + (uint32_t)(f & (R - 1)) * kDecSlotBytes;
      UQS_CHECK(at + 16u * (uint32_t)lane, 16u, RD); UQS_CHECK(at + 1024u, 16u, RD);
      const uint4 fv = lds_v4(at + 1024u);
      // lane = beam parameters: everything without FAN; with FAN only the warps that have a collision step this frame
      uint4 dv = make_uint4(0u, 0u, 0u, 0u);
      uint32_t dw = 0u;
      if (!FAN || ((w - f - 1) & (NW - 1)) < (int)fv.y) {
        dv = lds_v4(at + 16u * (uint32_t)lane);
        dw = lds_u32(at + 512u + 4u * (uint32_t)lane);
      }
      const uint32_t inv = dv.x;
      const int n2 = (int)dv.y, m = (int)dv.z, h2 = m & ~1;
      const int sM = (int)dv.w, sN = (int)dw >> 16;
      Beam B;
      B.end_delta = (int)(signed char)(dw & 0xffu);
      B.ra = (int)((dw >> 8) & 0xfu);
      B.rb = (dw & 0x1000u) ? -1 : 1;
      B.k0 = (int)fv.y;
      const int base = (int)fv.x, mmax = (int)fv.z;
      const bool sorted = fv.w != 0u;
      const int kshared = B.k0;                      // k_ray_setup caps K0 at mmax + 1

      // ---- steps k < K0: beams may meet in a cell; detect and keep beam order --------------------
      // the warp whose turn it is to decode a frame (w == f mod NW) gets the last of the collision steps, the others
      // the first ones: with K0 ~ 7 and four warps that is 1 step for the decoder and 2 for everyone else
      for (int k = (w - f - 1) & (NW - 1); k < kshared; k += NW) {
        const bool act = k <= m;
        const int q = minor_steps(k, n2, h2, inv);
        const int addr = base + k * sM + q * sN;
        const int delta = (k == m) ? B.end_delta : -lo_free;
        const unsigned actm0 = __ballot_sync(0xffffffffu, act);
        if (sorted && !__any_sync(0xffffffffu, act && k == m)) {
          // Beams in angular order and only free-space steps here: the beams on one cell are a run of
          // consecutive ACTIVE lanes (possibly wrapping from the last to the first), and the -free
          // steps commute, so the head of each run applies the run length at once.
          if (actm0 == 0u) continue;
          if (actm0 == 0xffffffffu) {
            // every beam is running (the usual frame): the previous beam is the previous lane, a run ends where
            // the next head is, and the only run that can wrap is lane 31's into lane 0's
            const int paddr = __shfl_up_sync(0xffffffffu, addr, 1);
            const bool head = lane == 0 || paddr != addr;
            const unsigned heads = __ballot_sync(0xffffffffu, head);
            const unsigned above_h = (heads >> 1) >> lane;                            // heads above this lane, shifted down
            int len = above_h ? __ffs(above_h) : 32 - lane;                           // lanes of my run
            bool apply = head;
            const int a_last = __shfl_sync(0xffffffffu, addr, 31);
            if (heads != 1u && __shfl_sync(0xffffffffu, addr, 0) == a_last) {         // lane 0's run continues lane 31's
              const int len0 = __shfl_sync(0xffffffffu, len, 0);
              if (lane == 31 - __clz(heads)) len += len0;
              if (lane == 0) apply = false;
            }
            if (apply) {
              const uint32_t cell = grid_sa + (uint32_t)addr;
              UQS_CHECK(cell, 1u, RG);
              sts_u8(cell, max(lds_s8(cell) - len * lo_free, lo_min));
            }
            __syncwarp();
            continue;
          }
          const unsigned lower = actm0 & ((1u << lane) - 1u);
          const int prev = lower ? (31 - __clz(lower)) : lane;
          const int paddr = __shfl_sync(0xffffffffu, addr, prev);
          const bool headr = act && (lower == 0u || paddr != addr);
          const unsigned heads = __ballot_sync(0xffffffffu, headr);
          const int first = __ffs(actm0) - 1, last = 31 - __clz(actm0);
          const int a_first = __shfl_sync(0xffffffffu, addr, first), a_last = __shfl_sync(0xffffffffu, addr, last);
          const unsigned above_h = heads & ~(0xffffffffu >> (31 - lane));           // heads above this lane
          const unsigned span = above_h ? ((1u << (__ffs(above_h) - 1)) - 1u) : 0xffffffffu;
          int len = __popc(actm0 & span & ~((1u << lane) - 1u));                     // active lanes of my run
          bool apply = headr;
          if ((heads & (heads - 1u)) != 0u && a_first == a_last) {                   // first run continues the last
            const int len_first = __shfl_sync(0xffffffffu, len, first);
            if (lane == 31 - __clz(heads)) len += len_first;
            if (lane == first) apply = false;
          }
          if (apply) {
            const uint32_t cell = grid_sa + (uint32_t)addr;
            UQS_CHECK(cell, 1u, RG);
            sts_u8(cell, max(lds_s8(cell) - len * lo_free, lo_min));
          }
          __syncwarp();
          continue;
        }
        // runs of consecutive lanes on one cell (beams are ordered by angle, so nearly all
        // collisions are between neighbours); only the head of a run enters the ring table
        const unsigned key = act ? (unsigned)addr : (0x80000000u | (unsigned)lane);
        const unsigned prevkey = __shfl_up_sync(0xffffffffu, key, 1);
        const bool bound = lane == 0 || prevkey != key;
        const bool head = act && bound;
        int pos = B.ra * k + B.rb * q;
        if (pos == 8 * k) pos = 0;
        const int slot = pos & ring_mask;
        if (head) { UQS_CHECK(ring_sa + (uint32_t)slot, 1u, RR); sts_u8(ring_sa + (uint32_t)slot, lane); }
        __syncwarp();
        const bool lost = head && lds_s8(ring_sa + (uint32_t)slot) != lane;
        const unsigned boundm = __ballot_sync(0xffffffffu, bound);
        const unsigned actm = __ballot_sync(0xffffffffu, act);
        unsigned pend = __ballot_sync(0xffffffffu, lost);
        const uint32_t cell = grid_sa + (uint32_t)addr;
        if (act) UQS_CHECK(cell, 1u, RG);
        if ((boundm & actm) == actm && pend == 0u) {
          if (act) sts_u8(cell, min(max(lds_s8(cell) + delta, lo_min), lo_max));
        } else {
          const unsigned upto = 0xffffffffu >> (31 - lane);               // lanes 0..lane
          const int start = 31 - __clz(boundm & upto);
          const unsigned above = boundm & ~upto;
          const int end = above ? (__ffs(above) - 2) : 31;
          unsigned peers = (0xffffffffu >> (31 - end)) & (0xffffffffu << start);
          while (pend) {          // runs that are not neighbours but hit the same cell (rare)
            const int a = __shfl_sync(0xffffffffu, addr, __ffs(pend) - 1);
            const bool same = act && addr == a;
            const unsigned members = __ballot_sync(0xffffffffu, same);
            pend &= ~members;
            if (same) peers = members;
          }
          const unsigned endm = __ballot_sync(0xffffffffu, act && k == m);
          const bool uniform = (peers & endm) == 0u;          // only free-space steps in this cell
          if (act && uniform && lane == __ffs(peers) - 1) {
            // repeated clamp(v - free) == max(v - cnt*free, lo_min)
            sts_u8(cell, max(lds_s8(cell) - __popc(peers) * lo_free, lo_min));
          }
          const bool mixed = act && !uniform;
          const int rank = __popc(peers & ((1u << lane) - 1u));
          const int rounds = __reduce_max_sync(0xffffffffu, mixed ? rank : -1);
          for (int r = 0; r <= rounds; r++) {
            if (mixed && rank == r) sts_u8(cell, min(max(lds_s8(cell) + delta, lo_min), lo_max));
            __syncwarp();
          }
        }
        __syncwarp();      // ring[] is rewritten by the next step
      }

      const uint32_t gbase = grid_sa + (uint32_t)base;
      const int free_delta = -lo_free;
      constexpr int UN = UQS_UN;                    // steps in flight per warp
      if (FAN) {
        // ---- steps k >= K0, fan layout: lane = (beam of this warp's sensor, one of 4 consecutive steps) -----------
        constexpr int NS = NW / 4;                  // warps per sensor
        const uint32_t bq = (uint32_t)((w & 3) * 8 + (lane >> 2));
        const int j = lane & 3;
        UQS_CHECK(at + 16u * bq, 16u, RD); UQS_CHECK(at + 512u + 4u * bq, 4u, RD);
        const uint4 ev = lds_v4(at + 16u * bq);
        const uint32_t ew = lds_u32(at + 512u + 4u * bq);
        const uint32_t inv_f = ev.x;
        const int n2_f = (int)ev.y, m_f = (int)ev.z, h2_f = m_f & ~1, sM_f = (int)ev.w, sN_f = (int)ew >> 16;
        const int fmax = __reduce_max_sync(0xffffffffu, m_f);          // longest beam of the fan
        int kb = kshared + 4 * (w >> 2);                                // first block of 4 steps of this warp
        int mu[UN];                                                     // kb + j + u*4*NS < m_f  <=>  kb < mu[u]
#pragma unroll
        for (int u = 0; u < UN; u++) mu[u] = in_reg(m_f - j - u * 4 * NS);
        for (; kb < fmax; kb += UN * 4 * NS) {
          uint32_t addr[UN];
          int val[UN];
          bool on[UN];
#pragma unroll
          for (int u = 0; u < UN; u++) {
            const int ku = kb + j + u * 4 * NS;
            addr[u] = gbase + (uint32_t)(ku * sM_f + minor_steps(ku, n2_f, h2_f, inv_f) * sN_f);
            on[u] = kb < mu[u];
          }
#pragma unroll
          for (int u = 0; u < UN; u++) if (on[u]) { UQS_CHECK(addr[u], 1u, RG); val[u] = lds_s8(addr[u]); }
#pragma unroll
          for (int u = 0; u < UN; u++) if (on[u]) sts_u8(addr[u], __viaddmax_s32(val[u], free_delta, lo_min));
        }
        // end cells of the fan's beams that end at a step >= K0: one lane per beam, one warp per sensor
        if ((w >> 2) == ((f + 1) & (NS - 1)) && j == 0 && m_f >= kshared) {
          const uint32_t cell = gbase + (uint32_t)(m_f * sM_f + (n2_f >> 1) * sN_f);
          UQS_CHECK(cell, 1u, RG);
          sts_u8(cell, min(max(lds_s8(cell) + (int)(signed char)(ew & 0xffu), lo_min), lo_max));
        }
      } else {
      // ---- steps k >= K0: every cell is touched by one beam only; UN steps in flight, no branches
      // (lanes past their beam's end are predicated off)
      int k = B.k0 + ((w - B.k0) & (NW - 1));          // first step >= K0 of this warp's residue class
      // free-space steps K0 <= k < m only: clamp(v - free) = max(v - free, lo_min) because lo_free >= 0 (one
      // VIADDMNMX); the end cells of these beams are one extra step of one warp below
      int mu[UN];                                   // k + u*NW < m  <=>  k < mu[u]
#pragma unroll
      for (int u = 0; u < UN; u++) mu[u] = in_reg(m - u * NW);
      for (; k < mmax; k += UN * NW) {
        uint32_t addr[UN];
        int val[UN];
        bool on[UN];
#pragma unroll
        for (int u = 0; u < UN; u++) {
          const int ku = k + u * NW;
          addr[u] = gbase + (uint32_t)(ku * sM + minor_steps(ku, n2, h2, inv) * sN);
          on[u] = k < mu[u];
        }
#pragma unroll
        for (int u = 0; u < UN; u++) if (on[u]) { UQS_CHECK(addr[u], 1u, RG); val[u] = lds_s8(addr[u]); }
#pragma unroll
        for (int u = 0; u < UN; u++) if (on[u]) sts_u8(addr[u], __viaddmax_s32(val[u], free_delta, lo_min));
        // (skipping the store for cells already at lo_min was measured 8 % slower: two more ISETPs per step)
      }
      // end cells of the beams that end at a step >= K0 (q(m) = n): distinct cells, touched by nothing else
      // in this frame, so any warp may apply them at any time before the frame's barrier
      if (w == ((f + 1) & (NW - 1)) && mmax >= kshared) {
        if (m >= kshared) {
          const uint32_t cell = gbase + (uint32_t)(m * sM + (n2 >> 1) * sN);
          UQS_CHECK(cell, 1u, RG);
          sts_u8(cell, min(max(lds_s8(cell) + B.end_delta, lo_min), lo_max));
        }
      }
      }   // !FAN
      if (!PROD && (f & (NW - 1)) == w) {           // this warp's turn: decode frame f + L, prefetch its next turn
        const int g = f + L;
        if (g < A.n_frames) decode_store(raw_rec, raw_org, g & (R - 1));
        const int gn = min(g + NW, A.n_frames - 1);
        raw_rec = __ldg(&rays[(size_t)gn * 32 + lane]);
        raw_org = __ldg(reinterpret_cast<const uint2*>(&frames[gn]));
      }
      __syncthreads();
      if (PROBE) {
        while (next_pf == f) {                      // the taken probes are a prefix of [pb, pe) (frame order)
          const int i = pb + (int)threadIdx.x;
          const int4 pr = i < pe ? Q.probes[i] : make_int4(-1, 0, 0, 0);
          const bool take = pr.x == f;
          if (take) {
            const int gy = pr.y / A.W, gx = pr.y - gy * A.W;
            int v;
            if (gx >= bx0 && gx < bx0 + bw && gy >= by0 && gy < by0 + bh) {
              const uint32_t cell = grid_sa + (uint32_t)((gy - by0) * P + (gx - bx0));
              UQS_CHECK(cell, 1u, RG);
              v = lds_s8(cell);
            } else {
              v = (int)grid_hbm[pr.y];
            }
            Q.values[pr.z] = (uint32_t)v;
          }
          pb += __syncthreads_count(take);           // also keeps frame f + 1 from writing before every read is done
          next_pf = pb < pe ? Q.probes[pb].x : 0x7fffffff;
        }
      }
    }

    if (vec) {
      const int wpr = bw >> 2;
      for (int i = threadIdx.x; i < wpr * bh; i += NT) {
        const int r = i / wpr, c = i - r * wpr;
        reinterpret_cast<uint32_t*>(grid_g + (size_t)r * A.W)[c] = reinterpret_cast<const uint32_t*>(grid_s + r * P)[c];
      }
    } else {
      for (int i = threadIdx.x; i < bw * bh; i += NT) {
        const int r = i / bw, c = i - r * bw;
        grid_g[(size_t)r * A.W + c] = grid_s[r * P + c];
      }
    }
    __syncthreads();
  }
}

// Bounding box of every cell a flight can touch = union of its 32-frame group boxes; x is widened to
// multiples of 4 (when W allows) so that rows move as 32-bit words.  dims[0..1] = max width / height.
__global__ void k_flight_boxes(int n_flights, int groups_per_flight, const uint2* __restrict__ groups, int W, int H,
                               int4* __restrict__ boxes, int* __restrict__ dims) {
  const int flight = (int)((blockIdx.x * (long long)blockDim.x + threadIdx.x) >> 5);
  const int lane = threadIdx.x & 31;
  if (flight >= n_flights) return;
  int x0 = 0x7fff, x1 = -1, y0 = 0x7fff, y1 = -1;
  for (int g = lane; g < groups_per_flight; g += 32) {
    const uint2 b = __ldg(&groups[(size_t)flight * groups_per_flight + g]);
    const int bx0 = (int)(b.x & 0xffffu), bx1 = (int)(b.x >> 16), by0 = (int)(b.y & 0xffffu), by1 = (int)(b.y >> 16);
    if (bx0 <= bx1 && by0 <= by1) { x0 = min(x0, bx0); x1 = max(x1, bx1); y0 = min(y0, by0); y1 = max(y1, by1); }
  }
  x0 = __reduce_min_sync(0xffffffffu, x0); x1 = __reduce_max_sync(0xffffffffu, x1);
  y0 = __reduce_min_sync(0xffffffffu, y0); y1 = __reduce_max_sync(0xffffffffu, y1);
  if (lane == 0) {
    int4 box = make_int4(0, 0, 0, 0);
    if (x0 <= x1 && y0 <= y1) {
      x1 += 1; y1 += 1;                                  // exclusive
      if ((W & 3) == 0) { x0 &= ~3; x1 = min((x1 + 3) & ~3, W); }
      box = make_int4(x0, y0, x1, y1);
      atomicMax(&dims[0], x1 - x0);
      atomicMax(&dims[1], y1 - y0);
    }
    boxes[flight] = box;
  }
}

static void (*flight_kernel(int nw, int fan, int prod))(FlightArgs, ProbeArgs) {
  if (prod) return nw == 4 ? k_replay_flights<4, 0, 1> : (nw == 8 ? k_replay_flights<8, 0, 1> : (nw == 32 ? k_replay_flights<16, 0, 1> : k_replay_flights<16, 0, 1>));
  if (fan) return nw == 4 ? k_replay_flights<4, 1, 0> : (nw == 8 ? k_replay_flights<8, 1, 0> : (nw == 32 ? k_replay_flights<32, 1, 0> : k_replay_flights<16, 1, 0>));
  return nw == 4 ? k_replay_flights<4, 0, 0> : (nw == 8 ? k_replay_flights<8, 0, 0> : (nw == 32 ? k_replay_flights<32, 0, 0> : k_replay_flights<16, 0, 0>));
}

// dims -> mapped host memory: a device-to-host memcpy of these two words would queue on the D2H copy engine
// behind the grids of the previous chunk (measured: 1.8 ms per chunk of the host-buffer pipeline)
__global__ void k_publish_dims(const int* __restrict__ dims, volatile int* host_dims) {
  host_dims[0] = dims[0];
  host_dims[1] = dims[1];
  __threadfence_system();
}

cudaError_t flight_boxes_launch(int n_flights, int groups_per_flight, const uint2* groups, int W, int H, int4* boxes,
                                int* dims, int* host_dims_dev, cudaStream_t st) {
  k_flight_boxes<<<(unsigned)((n_flights + 3) / 4), 128, 0, st>>>(n_flights, groups_per_flight, groups, W, H, boxes, dims);
  k_publish_dims<<<1, 1, 0, st>>>(dims, host_dims_dev);
  return cudaGetLastError();
}

// (the producer variant exists for 4, 8 and 16 consumer warps; 32 + 1 warps would exceed a CTA)
static int flight_threads(int nw, int prod) { return (std::min(nw, prod ? 16 : 32) + (prod ? 1 : 0)) * 32; }

cudaError_t flights_prepare(int nw, int fan, int prod, size_t smem, int* ctas_per_sm) {
  cudaError_t e = cudaFuncSetAttribute(flight_kernel(nw, fan, prod), cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
  if (e != cudaSuccess) return e;
  return cudaOccupancyMaxActiveBlocksPerMultiprocessor(ctas_per_sm, flight_kernel(nw, fan, prod), flight_threads(nw, prod), smem);
}

cudaError_t flights_launch(int nw, int fan, int prod, unsigned grid, size_t smem, cudaStream_t st, const FlightArgs& A) {
  flight_kernel(nw, fan, prod)<<<grid, flight_threads(nw, prod), smem, st>>>(A, ProbeArgs{});
  return cudaGetLastError();
}

// the probe variant exists for the default layout only (the fan layout and the decode warp were measured and rejected)
static void (*flight_probe_kernel(int nw))(FlightArgs, ProbeArgs) {
  return nw == 4 ? k_replay_flights<4, 0, 0, true> : (nw == 8 ? k_replay_flights<8, 0, 0, true> : (nw == 32 ? k_replay_flights<32, 0, 0, true> : k_replay_flights<16, 0, 0, true>));
}

cudaError_t flights_probe_prepare(int nw, size_t smem, int* ctas_per_sm) {
  cudaError_t e = cudaFuncSetAttribute(flight_probe_kernel(nw), cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
  if (e != cudaSuccess) return e;
  return cudaOccupancyMaxActiveBlocksPerMultiprocessor(ctas_per_sm, flight_probe_kernel(nw), flight_threads(nw, 0), smem);
}

cudaError_t flights_probe_launch(int nw, unsigned grid, size_t smem, cudaStream_t st, const FlightArgs& A, const ProbeArgs& Q) {
  flight_probe_kernel(nw)<<<grid, flight_threads(nw, 0), smem, st>>>(A, Q);
  return cudaGetLastError();
}

cudaError_t tiles_prepare(bool probe, size_t smem, int* ctas_per_sm) {
  void (*k)(ReplayArgs, ProbeArgs) = probe ? k_replay_tiles<true> : k_replay_tiles<false>;
  cudaError_t e = cudaFuncSetAttribute(k, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
  if (e != cudaSuccess) return e;
  return cudaOccupancyMaxActiveBlocksPerMultiprocessor(ctas_per_sm, k, kReplayThreads, smem);
}

cudaError_t tiles_launch(bool probe, unsigned grid, size_t smem, cudaStream_t st, const ReplayArgs& A, const ProbeArgs& Q) {
  if (probe) k_replay_tiles<true><<<grid, kReplayThreads, smem, st>>>(A, Q);
  else       k_replay_tiles<false><<<grid, kReplayThreads, smem, st>>>(A, Q);
  return cudaGetLastError();
}

// Zero fill as a kernel.  cudaMemsetAsync of a large range can be carried out by a copy engine, where it
// queues behind the D2H of the previous chunk of the host-buffer pipeline (measured: every replay waited
// ~1.8 ms for the neighbouring stream's copy); a kernel only depends on its own stream.
__global__ void k_zero(unsigned char* __restrict__ p, size_t bytes) {
  const size_t head = min(bytes, (size_t)((16 - (reinterpret_cast<size_t>(p) & 15)) & 15));
  const size_t n16 = (bytes - head) >> 4;
  const size_t tid = (size_t)blockIdx.x * blockDim.x + threadIdx.x, nth = (size_t)gridDim.x * blockDim.x;
  uint4* q = reinterpret_cast<uint4*>(p + head);
  for (size_t i = tid; i < n16; i += nth) q[i] = make_uint4(0u, 0u, 0u, 0u);
  const size_t tail0 = head + (n16 << 4);
  if (tid < head) p[tid] = 0;
  if (tid < bytes - tail0) p[tail0 + tid] = 0;
}

cudaError_t zero_async(void* p, size_t bytes, cudaStream_t st) {
  if (bytes == 0) return cudaSuccess;
  const size_t want = (bytes / 16 + 255) / 256;
  const unsigned blocks = (unsigned)std::min<size_t>(std::max<size_t>(want, 1), 148 * 16);
  k_zero<<<blocks, 256, 0, st>>>(reinterpret_cast<unsigned char*>(p), bytes);
  return cudaGetLastError();
}

// ===========================================================================
// on-chip RMW ceiling: the same byte read-modify-write as apply_frame(), with
// conflict-free addresses and no ray arithmetic.
// ===========================================================================
__global__ void __launch_bounds__(kReplayThreads)
k_rmw_peak(int tile_bytes, int iters, int lo_min, int* sink) {
  // Ceiling of the update itself: every warp read-modify-writes bytes of its own shared-memory tile, 32 consecutive
  // bytes per warp instruction (8 banks, one wavefront, no conflict), eight independent updates in flight, and
  // nothing else -- no ray arithmetic, no clipping, no collisions.  tile_bytes must be a power of two >= 2048.
  const int lane = threadIdx.x & 31, wic = threadIdx.x >> 5;
  int8_t* tile = reinterpret_cast<int8_t*>(uqs_smem) + (size_t)wic * tile_bytes;
  for (int i = lane; i < tile_bytes; i += 32) tile[i] = 0;
  __syncwarp();
  const uint32_t base = (uint32_t)__cvta_generic_to_shared(tile) + (uint32_t)lane;
  const uint32_t mask = (uint32_t)tile_bytes - 1u;
  uint32_t off = 0;
  for (int it = 0; it < iters; it++) {
    int v[8];
#pragma unroll
    for (int u = 0; u < 8; u++) v[u] = lds_s8(base + ((off + 32u * u) & mask));
#pragma unroll
    for (int u = 0; u < 8; u++) sts_u8(base + ((off + 32u * u) & mask), max(v[u] - 1, lo_min));
    off += 256u + 32u;
  }
  __syncwarp();
  if (tile[lane] == 77) *sink = 1;
}

// The north star's sketch ("shared-memory grid tiles with integer log-odds atomics") measured: the same conflict-free
// access pattern as k_rmw_peak, but each update is one shared-memory atomic (ATOMS.ADD on a 32-bit word -- the
// hardware has no byte-wide shared atomic, so an int8 grid would need 4x the shared memory or a CAS loop on top of
// this).  bench.py reports the rate next to the plain load/clamp/store rate; it cannot express the per-update clamp
// anyway (uav_local_nav.c:259-260), this only prices the instruction.
__global__ void __launch_bounds__(kReplayThreads)
k_atoms_peak(int tile_bytes, int iters, int* sink) {
  const int lane = threadIdx.x & 31, wic = threadIdx.x >> 5;
  int* tile = reinterpret_cast<int*>(uqs_smem + (size_t)wic * tile_bytes);
  for (int i = lane; i < tile_bytes / 4; i += 32) tile[i] = 0;
  __syncwarp();
  const uint32_t mask = (uint32_t)(tile_bytes / 4) - 1u;
  uint32_t off = (uint32_t)lane;
  for (int it = 0; it < iters; it++) {
#pragma unroll
    for (int u = 0; u < 8; u++) atomicAdd(&tile[(off + 32u * u) & mask], -1);
    off += 256u + 32u;
  }
  __syncwarp();
  if (tile[lane] == 77) *sink = 1;
}

}  // namespace uqs
