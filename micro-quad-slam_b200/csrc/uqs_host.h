// uqs_host.h -- state shared by the host-side translation units of libuqs_mapping.so.
#pragma once
#include <cstddef>
#include <cstdint>
#include <cuda_runtime.h>
#include <vector>

#include "../../include/uqs_mapping.h"
#include "uqs_kernels.cuh"

namespace uqs {

constexpr int kDefaultDecodeWarp = 0;           // resident engine: 1 = an extra warp per CTA that only decodes (measured choice)
constexpr int kDefaultFanLayout = 0;            // resident engine: 0 = 32 beams x 1 step, 1 = 8 beams x 4 steps (measured choice)

// grow-only device buffer
struct DevBuf {
  void* p = nullptr;
  size_t cap = 0;
  int ensure(size_t bytes);
  void release();
};

// scratch of one in-flight replay: ray/frame records, counters, P0 increments (+ an optional
// stream override, used by the host-buffer pipeline to keep two chunks' kernels in flight)
struct Work {
  DevBuf rays, frames, groups, counters, inc, scan, order, maps, boxes;
  DevBuf probe_slots, probe_keys, probe_sorted, probe_start, probe_tmp;   // frontier probes and buckets (uqs_frontier.cu)
  int order_nsx = 0, order_nsy = 0;             // geometry the cached tile order was built for
  cudaStream_t stream = nullptr;
  int* h_dims = nullptr;                        // mapped host words the box kernel publishes its maxima to
  bool boxes_valid = false;                     // `boxes` holds the touched boxes of the last replay_device call's
  int boxes_n = 0, box_w = 0, box_h = 0;        //   boxes_n flights (one internal chunk), maxima box_w x box_h
  void release() {
    if (h_dims) cudaFreeHost(h_dims);
    h_dims = nullptr;
    DevBuf* all[] = { &rays, &frames, &groups, &counters, &inc, &scan, &order, &maps, &boxes, &probe_slots, &probe_keys, &probe_sorted,
                      &probe_start, &probe_tmp };
    order_nsx = order_nsy = 0;
    for (DevBuf* b : all) b->release();
  }
};

struct Context {
  bool ready = false;
  int device = -1;
  int sm_count = 0;
  cudaStream_t own_stream = nullptr;
  cudaStream_t ext_stream = nullptr;
  bool use_ext = false;
  int tune_sw = 0, tune_sh = 0, tune_slices = 0;
  int engine = 0;                               // 0 auto, 1 warp-owned sub-tiles, 2 grid resident per CTA
  int flight_warps = 0;                         // warps per CTA of the resident engine (0 = 16)
  int k0_bias = 0;                              // measurement: extra collision-checked steps per frame (uqs_set_k0_bias)
  int pitch_mod = -1;                           // experiment: resident row pitch in words mod 32 (uqs_set_resident_pitch_mod)
  int flight_prod = kDefaultDecodeWarp;         // dedicated decode warp (uqs_set_decode_warp)
  int flight_fan = kDefaultFanLayout;           // lane layout of its free-space steps (uqs_set_fan_layout)
  int host_chunk = 0;                           // flights per chunk of the host-buffer pipeline (0 = auto)
  bool copy_only = false;                       // measurement: host-buffer calls skip their kernels (uqs_set_copy_only)
  bool chip_shared = false;                     // a multi-chunk host-buffer call is in flight: chunks share the chip
  size_t scratch_budget = (size_t)12 << 30;     // ray/frame records held at once
  unsigned long long launches = 0;              // kernels launched by this library
  DevBuf inv_table;                             // ceil(2^31 / m) for m = 0..kMaxRayCells (0 at m = 0)
  // scratch: works[0] serves the device-pointer API and the drop-in, works[1..2] the pipeline
  Work works[3];
  Work* w = &works[0];
  // staging for the host-buffer entry points
  DevBuf in_t, in_rx, in_ry, in_h, in_yaw, in_q, in_x, in_y, in_ranges, in_kind, out_grids;
  void* pipeline = nullptr;                     // streams and staging of the host-buffer pipeline (uqs_pipeline.cu)
  void* comm = nullptr;                         // ncclComm_t of this device (uqs_multi.cu), nullptr = none
  int comm_rank = 0, comm_nranks = 1;
  int band_edges[17] = { 0 };                   // row cuts of the last banded replay (uqs_band_edges)

  // optional per-kernel timing (uqs_set_profiling): event pairs on the launching stream
  bool profiling = false;
  struct Span { cudaEvent_t a, b; int kind; };   // kind 0 pose, 1 ray set-up, 2 replay, 3 H2D, 4 D2H (pipeline copies)
  std::vector<Span> spans;

  cudaStream_t stream() const { return w->stream ? w->stream : (use_ext ? ext_stream : own_stream); }
  cudaStream_t user_stream() const { return use_ext ? ext_stream : own_stream; }
  void release_all() {
    DevBuf* all[] = { &in_t, &in_rx, &in_ry, &in_h, &in_yaw, &in_q, &in_x, &in_y, &in_ranges, &in_kind, &out_grids };
    for (DevBuf* b : all) b->release();
    for (Work& k : works) k.release();
    inv_table.release();
  }
};

constexpr size_t kFlightSmemMax = 227u * 1024u - 64u;   // dynamic + the kernel's few static bytes

// One Context per device.  A process that drives one GPU (the usual case: one process per GPU) only ever has the
// first; uqs_multi_init() creates one per device and uqs_multi_select() switches the current one, so every entry
// point below works unchanged on whichever device is current.
extern Context* g_cur;
#define g_ctx (*::uqs::g_cur)
int context_init(Context& c, int device);     // stream + properties on `device` (leaves it current)
void context_shutdown(Context& c);
void context_select_single();                 // back to the context of uqs_init()

void set_error(const char* fmt, ...);
int cuda_fail(cudaError_t e, const char* what);
int check_ready();
int make_dev_params(const uqs_params* p, DevParams* d);
// Frontier queries answered inside a replay (uqs_frontier.cu).  Query q owns the probe slots (q*3 + r)*s_max + k: ray
// r's k-th sample, cells[slot] = its cell or -1 (past the grid's edge).  values[slot] receives the cell's value at the
// query's frame.
struct ProbeSet {
  int n_queries = 0, s_max = 0;
  const uqs_query* queries = nullptr;
  const int* cells = nullptr;
  uint32_t* values = nullptr;
  size_t slots() const { return (size_t)n_queries * 3 * s_max; }
};
// Sort the probes of flights [f0, f0 + nf) into buckets (launch-local flight ids): per flight when slices == 0,
// per (flight, time slice, sub-tile) otherwise.  Asynchronous on the current stream.
int probe_buckets(const ProbeSet& Q, int f0, int nf, int n_frames, int W, int slices, int groups_per_slice, int sw,
                  int sh, int nsx, int nsy, ProbeArgs* out);
// value = map word of slice s >= 1 applied after slice 0's value and the maps of slices 1..s-1 (before k_compose_slices)
int probe_resolve_slices(const ProbeArgs& A, int n_probes_max, const int8_t* grids, const uint32_t* maps, int W, int H,
                         int slices, int groups_per_slice);

// probes == nullptr: the plain replay.  With probes the engine and geometry are chosen exactly as without them.
int replay_device(const DevParams& dp, int n_flights, int n_frames, const float* x, const float* y,
                  const float* yaw, const float* ranges, const uint8_t* kind, int8_t* grids,
                  int accumulate, int row0, int rows, bool reset_stats, const ProbeSet* probes = nullptr);
int fetch_stats(uqs_stats* stats, uint64_t frames);
int ensure_inv_table();
// uqs_generic.cu: the unrestricted replay and the start-grid range check
cudaError_t generic_launch(const DevParams& dp, int n_flights, int n_frames, const float* x, const float* y, const float* yaw,
                           const float* ranges, const uint8_t* kind, int8_t* grids, int accumulate, int row0, int rows,
                           unsigned long long* stats, cudaStream_t st, const ProbeArgs* Q = nullptr);
cudaError_t range_check_launch(const int8_t* grids, int n_flights, int W, int H, int row0, int rows, int lo_min, int lo_max,
                               unsigned long long* bad, cudaStream_t st);
int fetch_stats_mask(uqs_stats* stats, uint64_t frames, unsigned mask);
void dropin_release();
void pipeline_release();
void comm_release();                          // uqs_multi.cu: destroys the current context's communicator
int pose_device(int n_flights, int n_samples, const uint32_t* t_ms, const float* rx, const float* ry,
                const float* h, const float* yaw, const uint8_t* q, float* xo, float* yo, int mode);

// RAII-free helper: records an event pair around a kernel launch when profiling is on
struct KernelTimer {
  int kind;
  cudaStream_t st;
  cudaEvent_t a = nullptr, b = nullptr;
  explicit KernelTimer(int k, cudaStream_t on = nullptr) : kind(k), st(on ? on : g_ctx.stream()) {
    if (g_ctx.profiling && cudaEventCreate(&a) == cudaSuccess && cudaEventCreate(&b) == cudaSuccess)
      cudaEventRecord(a, st);
  }
  void stop() {
    if (a && b) {
      cudaEventRecord(b, st);
      g_ctx.spans.push_back({a, b, kind});
    }
  }
};

}  // namespace uqs
