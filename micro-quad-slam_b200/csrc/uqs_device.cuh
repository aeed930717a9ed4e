// uqs_device.cuh -- exact device arithmetic of the mapping path (sm_100a).
//
// Every float operation below is an explicit round-to-nearest intrinsic
// (__fadd_rn/__fmul_rn/__fdiv_rn never contract into FMA), mirroring one C
// operator of the reference each, in source order (SURVEY.md Appendix A).  The
// translation unit is additionally compiled with -fmad=false.
#pragma once
#include <cstdint>
#include <cuda_runtime.h>

namespace uqs {

// Device copy of uqs_params plus the constants the reference folds at compile time.
struct DevParams {
  int   W, H, halfW, halfH;
  float res, ox, oy;
  float max_range, min_range, hit_below;  // hit_below = max_range - hit_margin (uav_local_nav.c:292)
  float half_fov;                         // fov * 0.5f                          (:284)
  float col_off[8];                       // ((float)c - 3.5f) / 3.5f * half_fov (:295-296), folded on the host in binary32
  float deg2rad;                          // (float)M_PI / 180.0f                (:299)
  int   lo_free, lo_occ, lo_min, lo_max;
  int   end_nohit;                        // -(lo_free / 2), integer division   (:266)
  int   ranges_u16;                       // the call's range array is u16 millimetres (0xFFFF = no return) instead
                                          // of float metres; converted as uav_local_nav.c:1328 does, (float)mm * 0.001f
};

// range reading b of a frame from either input form
__device__ __forceinline__ float range_from_mm(unsigned mm) {
  return mm == 0xFFFFu ? __int_as_float(0x7fc00000) : __fmul_rn((float)mm, 0.001f);
}

// Ray record, 8 bytes:  w0 = dx[12 signed] | dy[12 signed]<<12 | hit<<24 | valid<<25
//                       w1 = ceil(2^31 / m), m = max(|dx|,|dy|)  (0 when m == 0)
// Frame record, 16 bytes: x = origin cell gx | K0<<16, y = gy | kFrameHasOrigin
//                         (K0: beams of the frame can share a cell only at steps k < K0),
//                         z = xmin | xmax<<16, w = ymin | ymax<<16  (bbox of all cells the
//                         frame's accepted rays touch; empty bbox = min 0x7fff, max 0)
constexpr int      kMaxRayCells   = 1024;       // magic-division exactness bound (see DESIGN.md)
constexpr uint32_t kRayHit        = 1u << 24;
constexpr uint32_t kRayValid      = 1u << 25;
constexpr uint32_t kFrameHasOrigin = 1u << 16;
constexpr uint32_t kFrameSorted    = 1u << 17;   // the frame's beams are in circular angular order (exact test)
constexpr uint32_t kEmptyBoxLoHi  = 0x00007fffu;  // min = 0x7fff, max = 0  -> never overlaps

// ---------------------------------------------------------------------------
// glibc 2.39 sincosf, FMA build, restated (SURVEY.md Appendix B): all three branches, so every
// float input gives libm's bits.  |y| < 120 is the straight-line path below; |y| >= 120 is glibc's
// reduce_large (24-bit mantissa x 96 bits of 2/pi in integer arithmetic) -- the CPU restatement of the same
// code equals libm on every float (tests/test_arith_kats.py); Inf/NaN give y - y
// with x86's NaN bits (they only matter to the parity hook: lrintf of any NaN is the same cell).
// Always returns true (kept for callers that still test it).
// ---------------------------------------------------------------------------
static __constant__ uint32_t kInvPio4[24] = {
  0xa2, 0xa2f9, 0xa2f983, 0xa2f9836e, 0xf9836e4e, 0x836e4e44, 0x6e4e4415, 0x4e441529, 0x441529fc, 0x1529fc27,
  0x29fc2757, 0xfc2757d1, 0x2757d1f5, 0x57d1f534, 0xd1f534dd, 0xf534ddc0, 0x34ddc0db, 0xddc0db62, 0xc0db6295,
  0xdb629599, 0x6295993c, 0x95993c43, 0x993c4390, 0x3c439041 };

// the polynomial tail shared by both reductions: x reduced, xs = x with the quadrant's sign, swap = n & 1,
// neg_cos = the second coefficient table (cosine coefficients negated)
__device__ __forceinline__ void sincosf_poly(double x, double xs, bool swap, bool neg_cos, float& sn, float& cs) {
  const double x2 = __dmul_rn(x, x);
  const double x3 = __dmul_rn(x2, xs);
  const double x4 = __dmul_rn(x2, x2);
  const double s1 = __fma_rn(x2, -0x1.994eb3774cf24p-13, 0x1.1107605230bc4p-7);
  const double c2 = __fma_rn(x2, 0x1.99343027bf8c3p-16, -0x1.6c087e89a359dp-10);
  const double c1 = __fma_rn(x2, -0x1.ffffffd0c621cp-2, 1.0);
  const double x5 = __dmul_rn(x2, x3);
  const double x6 = __dmul_rn(x2, x4);
  double S = __fma_rn(x3, -0x1.555545995a603p-3, xs);
  double C = __fma_rn(x4, 0x1.55553e1068f19p-5, c1);
  S = __fma_rn(x5, s1, S);
  C = __fma_rn(x6, c2, C);
  if (neg_cos) C = -C;
  const float fs = __double2float_rn(S), fc = __double2float_rn(C);
  if (swap) { cs = fs; sn = fc; } else { sn = fs; cs = fc; }
}

static __device__ __noinline__ void sincosf_large(float y, float& sn, float& cs) {
  uint32_t xi = __float_as_uint(y);
  if (((xi >> 20) & 0x7ffu) >= 0x7f8u) {       // Inf, NaN: y - y as x86 computes it
    const uint32_t nan = ((xi & 0x7fffffffu) == 0x7f800000u) ? 0xffc00000u : (xi | 0x00400000u);
    sn = cs = __uint_as_float(nan);
    return;
  }
  const int sign = (int)(xi >> 31);
  const uint32_t* arr = &kInvPio4[(xi >> 26) & 15u];
  const int shift = (int)((xi >> 23) & 7u);
  xi = ((xi & 0xffffffu) | 0x800000u) << shift;
  unsigned long long res0 = (unsigned long long)(uint32_t)(xi * arr[0]);
  const unsigned long long res1 = (unsigned long long)xi * arr[4];
  const unsigned long long res2 = (unsigned long long)xi * arr[8];
  res0 = (res2 >> 32) | (res0 << 32);
  res0 += res1;
  const unsigned long long nn = (res0 + (1ull << 61)) >> 62;
  res0 -= nn << 62;
  const double x = __dmul_rn(__ll2double_rn((long long)res0), 0x1.921FB54442D18p-62);
  const int n = (int)nn;
  const double xs = (((n + sign) + 1) & 2) ? -x : x;          // sign table {+,-,-,+}[(n + sign) & 3]
  sincosf_poly(x, xs, (n & 1) != 0, ((n + sign) & 2) != 0, sn, cs);
}

__device__ __forceinline__ bool sincosf_glibc(float y, float& sn, float& cs) {
  const uint32_t top12 = (__float_as_uint(y) >> 20) & 0x7ffu;
  if (top12 >= 0x42fu) {                      // |y| >= 120, Inf, NaN: the rare branch, out of line
    sincosf_large(y, sn, cs);
    return true;
  }
  // glibc skips the reduction when |y| < 0.75 (top12 < 0x3f4); running it there gives n = 0 and leaves x
  // unchanged bit for bit (|y * 2/pi| < 0.48 rounds to 0, fma(-0.0, pi/2, x) == x), so one straight-line
  // path serves both cases and a warp never executes the polynomial twice.
  double x = (double)y;
  const double r = __dmul_rn(x, 0x1.45f306dc9c883p+23);
  const int n = (__double2int_rz(r) + 0x800000) >> 24;
  x = __fma_rn(-(double)n, 0x1.921fb54442d18p+0, x);
  const double xs = ((n + 1) & 2) ? -x : x;   // sign table {+,-,-,+}[n & 3]
  const double x2 = __dmul_rn(x, x);
  const double x3 = __dmul_rn(x2, xs);
  const double x4 = __dmul_rn(x2, x2);
  const double s1 = __fma_rn(x2, -0x1.994eb3774cf24p-13, 0x1.1107605230bc4p-7);
  const double c2 = __fma_rn(x2, 0x1.99343027bf8c3p-16, -0x1.6c087e89a359dp-10);
  const double c1 = __fma_rn(x2, -0x1.ffffffd0c621cp-2, 1.0);
  const double x5 = __dmul_rn(x2, x3);
  const double x6 = __dmul_rn(x2, x4);
  double S = __fma_rn(x3, -0x1.555545995a603p-3, xs);
  double C = __fma_rn(x4, 0x1.55553e1068f19p-5, c1);
  S = __fma_rn(x5, s1, S);
  C = __fma_rn(x6, c2, C);
  if (n & 2) C = -C;                          // second table = cosine coefficients negated
  const float fs = __double2float_rn(S), fc = __double2float_rn(C);
  const bool tiny = top12 < 0x398u;           // |y| < 2^-12: glibc returns (y, 1.0f) before any arithmetic
  if (n & 1) { cs = fs; sn = fc; } else { sn = fs; cs = fc; }
  if (tiny) { sn = y; cs = 1.0f; }
  return true;
}

// (int)lrintf(q): x86-64 cvtss2si yields 0x8000000000000000 for NaN and |q| >= 2^63,
// whose low 32 bits are 0; in range the cast keeps the low 32 bits.
__device__ __forceinline__ int lrintf_as_int(float q) {
  if (fabsf(q) < 2147483520.0f) return __float2int_rn(q);          // fits int32: same value, 32-bit convert
  const long long r = (fabsf(q) < 9223372036854775808.0f) ? __float2ll_rn(q)
                                                          : (long long)0x8000000000000000ull;
  return (int)r;
}

// world_to_grid(), uav_local_nav.c:205-214, with the map origin (ox, oy) (map_origin_x/y, which recentering moves)
__device__ __forceinline__ bool world_to_grid_at(const DevParams& p, float ox, float oy, float wx, float wy, int& gx,
                                                 int& gy) {
  const float ddx = __fsub_rn(wx, ox);
  const float ddy = __fsub_rn(wy, oy);
  const int ix = (int)((unsigned)lrintf_as_int(__fdiv_rn(ddx, p.res)) + (unsigned)p.halfW);
  const int iy = (int)((unsigned)lrintf_as_int(__fdiv_rn(ddy, p.res)) + (unsigned)p.halfH);
  gx = ix;
  gy = iy;
  return !(ix < 0 || ix >= p.W || iy < 0 || iy >= p.H);
}

// world_to_grid(), uav_local_nav.c:205-214, with the origin of p
__device__ __forceinline__ bool world_to_grid(const DevParams& p, float wx, float wy, int& gx,
                                              int& gy) {
  const float ddx = __fsub_rn(wx, p.ox);
  const float ddy = __fsub_rn(wy, p.oy);
  const int ix = (int)((unsigned)lrintf_as_int(__fdiv_rn(ddx, p.res)) + (unsigned)p.halfW);
  const int iy = (int)((unsigned)lrintf_as_int(__fdiv_rn(ddy, p.res)) + (unsigned)p.halfH);
  gx = ix;
  gy = iy;
  return !(ix < 0 || ix >= p.W || iy < 0 || iy >= p.H);
}

// Beam b of map_update_from_beams(), uav_local_nav.c:286-303, up to the end point.
//   returns 0: skipped (:289-290), 1: end point computed, -1: angle outside the restated domain
__device__ __forceinline__ int beam_endpoint(const DevParams& p, float px, float py, float yaw_deg,
                                             float dist, int b, float& ex, float& ey, bool& hit) {
  if (isnan(dist)) return 0;
  if (dist <= p.min_range) return 0;
  hit = dist < p.hit_below;
  if (dist > p.max_range) dist = p.max_range;
  const int d = b >> 3, c = b & 7;
  // {0, 90, 180, -90}[d] without a branch (uav_local_nav.c:283)
  const float centre = (d & 1) ? ((d & 2) ? -90.0f : 90.0f) : ((d & 2) ? 180.0f : 0.0f);
  const float off = p.col_off[c];
  const float ang_deg = __fadd_rn(__fadd_rn(yaw_deg, centre), off);
  const float ang = __fmul_rn(ang_deg, p.deg2rad);
  float sn, cs;
  if (!sincosf_glibc(ang, sn, cs)) return -1;
  ex = __fadd_rn(px, __fmul_rn(dist, cs));
  ey = __fadd_rn(py, __fmul_rn(dist, sn));
  return 1;
}

__device__ __forceinline__ int sext12(uint32_t v) { return ((int)(v << 20)) >> 20; }

// frontier_score_dir(), uav_local_nav.c:356-385, piece by piece (k_frontier_scores and the probe set-up of
// uqs_frontier.cu share them).  Ray r (0, +15, -15 degrees, :360) of a query: its angle (:367) ...
__device__ __forceinline__ float frontier_ray_angle(const DevParams& p, float yaw_deg, float offset_deg, int r) {
  const float ro = (r == 0) ? 0.0f : (r == 1) ? 15.0f : -15.0f;
  return __fmul_rn(__fadd_rn(__fadd_rn(yaw_deg, offset_deg), ro), p.deg2rad);
}
// ... its first sample distance and step (:361-362: d = step, step + step, ... <= 2.5f) ...
__device__ __forceinline__ float frontier_step(const DevParams& p) { return __fmul_rn(p.res, 2.0f); }
constexpr float kFrontierRange = 2.5f;
// ... the cell of the sample at distance d in the window of map origin (ox, oy) (:373-375; false = off the window, which
// ends the ray) ...
__device__ __forceinline__ bool frontier_point(const DevParams& p, float ox, float oy, float x, float y, float d, float ca,
                                               float sa, int& gx, int& gy) {
  const float px = __fadd_rn(x, __fmul_rn(d, ca));
  const float py = __fadd_rn(y, __fmul_rn(d, sa));
  return world_to_grid_at(p, ox, oy, px, py, gx, gy);
}
// ... and the score's weight of the cell's value (:378-383): unknown +3, free +1, occupied -4
__device__ __forceinline__ int frontier_weight(int v) {
  return (v >= -1 && v <= 1) ? 3 : (v > 10) ? -4 : (v < -10) ? 1 : 0;
}

// q(k) = floor((k*n + m/2) / m) without a divide: n2 = 2n, h2 = 2*(m>>1), inv = ceil(2^31/m).
// Exact for m <= 1289 (t*m < 2^31 with t <= m*m + m/2); m is capped at kMaxRayCells.
__device__ __forceinline__ int minor_steps(int k, int n2, int h2, uint32_t inv) {
  return (int)__umulhi((uint32_t)(k * n2 + h2), inv);
}

}  // namespace uqs
