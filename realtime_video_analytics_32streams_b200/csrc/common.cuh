// Internal helpers shared by the libb200va translation units.
#pragma once

#include <cuda_runtime.h>
#include <stdint.h>

#include <atomic>
#include <cstdarg>
#include <cstdio>
#include <cstring>
#include <map>
#include <mutex>
#include <string>
#include <tuple>
#include <utility>
#include <vector>

#include "b200va.h"

#define B200VA_MAX_BATCH 128
// Frames per kernel launch: per-frame descriptors travel as kernel parameters (<= 4 KB).
#define B200VA_LAUNCH_FRAMES 64

struct TrackerState;  // tracker.cu
struct TapCache;      // preprocess.cu

// status_flags[] slots written by kernels (device int32), mirrored on demand by b200va_check.
enum {
  FLAG_CAND_OVERFLOW = 0,   // a frame produced more candidates than max_candidates
  FLAG_DET_OVERFLOW = 1,    // a frame kept more detections than max_dets
  FLAG_TRACK_OVERFLOW = 2,  // a stream needed more than max_tracks live tracks
  FLAG_TRACK_ROWS = 3,      // a stream holds more tracks than the caller's output table has rows (b200va_tracks.rows)
  FLAG_COUNT = 8
};

struct b200va_ctx {
  b200va_config cfg;
  int num_sms = 0;
  std::string last_error;
  std::atomic<int64_t> launches{0};
  std::recursive_mutex mu;  // recursive: b200va_tick holds it while calling the per-step entry points

  // ---- post-process scratch (device), all [max_batch, max_candidates] ----
  unsigned long long* cand_key = nullptr;  // (score bits << 32) | anchor tie rule | slot (cand_key() in postprocess.cu)
  float4* cand_box = nullptr;              // xyxy, frame pixels
  int32_t* cand_cls = nullptr;
  int32_t* cand_count = nullptr;           // [max_batch]
  // b200va_tick schedule 4 (software-pipelined tick) decodes tick k into one candidate set while NMS + tracker of
  // tick k-1 still read the other: every cand_* array holds two sets, `cand_set` is the one the next decode writes
  size_t cand_set_elems = 0;               // elements per set of cand_key / cand_box / cand_cls
  int cand_set_frames = 0;                 // frames per set (entries of cand_count per set)
  int cand_set = 0;
  void* pending_chain = nullptr;           // postprocess.cu: parameters of the NMS + tracker launch still owed
  int32_t* status_flags = nullptr;         // device int32[FLAG_COUNT]
  // ---- preprocess ----
  TapCache* taps = nullptr;
  // ---- roi rasteriser scratch ----
  void* roi_scratch = nullptr;  // device, ROI_SCRATCH_BYTES
  // ---- tracker ----
  TrackerState* tracker = nullptr;
  // ---- device-side gates (gates.cu): skip mask read by the letterbox, decode, NMS and tracker kernels ----
  const uint8_t* skip_dev = nullptr;  // DEVICE uint8 [batch] or NULL (b200va_set_skip_mask)
  void* gates = nullptr;              // gates.cu: per-slot gate state
  void* dense_nms = nullptr;          // postprocess.cu: scratch of the dense-scene NMS (suppressor lists)
  void* egress = nullptr;  // egress.cu: INTER_AREA tables per geometry, device copy of the rectangle list
  // ---- b200va_tick: second stream for the post-process + tracker branch ----
  cudaStream_t side_stream = nullptr;    // non-blocking, highest priority (its 32-CTA kernels slot in first)
  cudaEvent_t ev_fork = nullptr, ev_join = nullptr, ev_decoded = nullptr;
  cudaEvent_t hook_after_decode = nullptr;  // when set, b200va_postprocess records it right after the decode launch
  bool hook_recorded = false;               // ... and reports here that it did
  // b200va_tick schedule 3: the decode kernel runs on the caller's stream, everything after it (NMS, tracker) on
  // `post_tail_stream`, which first waits for the hook event; the letterbox launched next on the caller's stream is
  // a programmatic dependent of the decode kernel (`pdl_preprocess`) and fills the SMs next to it
  cudaStream_t post_tail_stream = nullptr;
  bool pdl_preprocess = false;
  bool pdl_preprocess_wait = false;  // ... and the letterbox waits for its primary's completion before its first load
  // ---- NMS variant selection: host-mapped statistic written by k_sort_nms ----
  int* nms_stats_host = nullptr;
  int* nms_stats_dev = nullptr;
  int nms_dense_ttl = 0;  // launches left on the grid variant after the last dense sighting
  int trk_rows = 512;     // rows of the tracker's shared-memory working table (tracker_pick_smem_tracks)
  int trk_rows_ttl = 0;   // launches left before trk_rows falls back to 512
  // ---- b200va_set_profiling: one timed event pair per phase ----
  bool profiling = false;
  cudaEvent_t prof_ev[B200VA_PHASE_COUNT][2] = {};
  bool prof_rec[B200VA_PHASE_COUNT] = {};
  // ---- developer tuning knobs, read once from B200VA_* environment variables (0 = automatic) ----
  struct Tune {
    int decode_impl = 0, decode_ta = 0, decode_rows = 0, decode_stages = 0, decode_ctas_per_sm = 0;
    int fuse_post_track = 1;  // B200VA_FUSE_POST_TRACK=0: always launch NMS and tracker as two kernels
    int pdl = 1;              // B200VA_PDL=0: no programmatic dependent launches
    int uniform_carveout = 0; // B200VA_UNIFORM_CARVEOUT=1: every tick kernel prefers the all-shared-memory split
    int lb_smem_floor = 33 * 1024;  // B200VA_LB_SMEM_FLOOR=bytes: least dynamic shared memory of a letterbox CTA (caps CTAs per SM, see preprocess.cu)
    int dense_carveout = -1;  // B200VA_DENSE_CARVEOUT=pct: preferred carve-out of the dense-scene NMS kernels (-1: driver default)
    int post_carveout = -1;   // B200VA_POST_CARVEOUT=pct: preferred shared-memory carve-out of k_post_track (0: driver default)
    int dense_impl = 0;       // B200VA_DENSE_IMPL=1: dense scenes stay on the single-kernel NMS (k_sort_nms<true>); 2: every launch is 'dense'
    int dense_ctas_per_sm = 0; // B200VA_DENSE_CTAS=n: CTAs per SM of k_dense_pairs (default 8)
    int trk_max_threads = 0;  // B200VA_TRK_THREADS=n: widest tracker update of a stream (0: the CTA's width)
    int trk_smem_tracks = 0;  // B200VA_TRK_SMEM_TRACKS=n: fix the tracker's shared-memory table at n rows (tests)
  } tune;
  // ---- developer phase timing (only written by builds with -DB200VA_PHASE_TIMING) ----
  long long* dbg = nullptr;  // device int64[DBG_SLOTS]
};

#define DBG_SLOTS 64
#ifdef B200VA_PHASE_TIMING
#define PHASE_STAMP(buf, slot)                                              \
  do {                                                                      \
    if (blockIdx.x == 0 && blockIdx.y == 0 && threadIdx.x == 0) (buf)[slot] = clock64(); \
  } while (0)
#else
#define PHASE_STAMP(buf, slot) \
  do {                         \
  } while (0)
#endif

// Timeline stamps (timing builds only): first CTA start / last CTA end of a kernel in %globaltimer nanoseconds,
// dbg[slot] = min start, dbg[slot + 1] = max end.  Slots: 40 decode, 42 letterbox, 44 NMS / fused NMS + tracker, 46 tracker.
#ifdef B200VA_PHASE_TIMING
#define TIMELINE_BEGIN(buf, slot)                                                                   \
  do {                                                                                              \
    if (threadIdx.x == 0) {                                                                         \
      unsigned long long _t;                                                                        \
      asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(_t));                                        \
      atomicMin((unsigned long long*)&(buf)[slot], _t);                                             \
    }                                                                                               \
  } while (0)
#define TIMELINE_END(buf, slot)                                                                     \
  do {                                                                                              \
    if (threadIdx.x == 0) {                                                                         \
      unsigned long long _t;                                                                        \
      asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(_t));                                        \
      atomicMax((unsigned long long*)&(buf)[(slot) + 1], _t);                                       \
    }                                                                                               \
  } while (0)
#else
#define TIMELINE_BEGIN(buf, slot) do { } while (0)
#define TIMELINE_END(buf, slot) do { } while (0)
#endif

#define ROI_SCRATCH_BYTES (1 << 20)

inline int set_error(b200va_ctx* h, int code, const char* fmt, ...) {
  if (h) {
    char buf[512];
    va_list ap;
    va_start(ap, fmt);
    vsnprintf(buf, sizeof(buf), fmt, ap);
    va_end(ap);
    h->last_error = buf;
  }
  return code;
}

#define CUDA_TRY(h, expr)                                                                            \
  do {                                                                                               \
    cudaError_t _e = (expr);                                                                         \
    if (_e != cudaSuccess)                                                                           \
      return set_error((h), B200VA_ERR_CUDA, "%s failed: %s (%s:%d)", #expr, cudaGetErrorString(_e), \
                       __FILE__, __LINE__);                                                          \
  } while (0)

#define LAUNCH_CHECK(h)                                                                      \
  do {                                                                                       \
    (h)->launches.fetch_add(1, std::memory_order_relaxed);                                   \
    cudaError_t _e = cudaGetLastError();                                                     \
    if (_e != cudaSuccess)                                                                   \
      return set_error((h), B200VA_ERR_CUDA, "kernel launch failed: %s (%s:%d)",             \
                       cudaGetErrorString(_e), __FILE__, __LINE__);                          \
  } while (0)

#define REQUIRE(h, cond, ...)                                             \
  do {                                                                    \
    if (!(cond)) return set_error((h), B200VA_ERR_INVALID, __VA_ARGS__); \
  } while (0)

// NVTX range "b200va:<phase>" around an entry point's launches, plus the phase's event pair when profiling is on.
// Declared after the argument checks, so error returns before it record nothing.
const char* phase_name(int phase);  // api.cu
struct PhaseScope {
  b200va_ctx* h;
  int phase;
  cudaStream_t st;
  bool timed = false;
  PhaseScope(b200va_ctx* h_, int phase_, cudaStream_t st_);
  ~PhaseScope();
  PhaseScope(const PhaseScope&) = delete;
  PhaseScope& operator=(const PhaseScope&) = delete;
};

#ifdef __CUDACC__
// An SM can only change its L1 / shared-memory carve-out while it is empty, so kernels with different preferences
// never share an SM: measured with the timing build's timeline (tools/timeline.py), a letterbox launched as a
// programmatic dependent of the (shared-memory-free) decode kernel does not start until the decode CTAs begin to retire,
// and does start at t = 2 us once every kernel of the tick asks for the same split (B200VA_UNIFORM_CARVEOUT=1).  It is
// NOT the default: k_decode_cm keeps ~114 KB of loads in flight per SM through L1 and slows from 22.7 to 30.3 us with
// the 28 KB L1 that is left, which costs more than the overlap gains (tick 72 us against 64.5 us).
template <typename K>
inline cudaError_t prefer_max_shared(K kernel) {
  return cudaFuncSetAttribute(kernel, cudaFuncAttributePreferredSharedMemoryCarveout, (int)cudaSharedmemCarveoutMaxShared);
}

// The dynamic shared-memory limit is a property of the FUNCTION, shared by every handle of the process: only ever
// raise it (a second handle with smaller capacities must not pull it below what the first one launches with).
template <typename K>
inline cudaError_t raise_dyn_smem(K kernel, size_t bytes) {
  cudaFuncAttributes a;
  cudaError_t e = cudaFuncGetAttributes(&a, kernel);
  if (e != cudaSuccess) return e;
  if ((size_t)a.maxDynamicSharedSizeBytes >= bytes) return cudaSuccess;
  return cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)bytes);
}

// launch on `st` as a programmatic dependent of the kernel before it (its prologue overlaps that kernel's tail)
template <typename... KArgs, typename... Args>
inline cudaError_t launch_pdl(void (*kernel)(KArgs...), dim3 grid, dim3 block, size_t smem, cudaStream_t st, bool pdl, Args&&... args) {
  cudaLaunchConfig_t cfg = {};
  cfg.gridDim = grid;
  cfg.blockDim = block;
  cfg.dynamicSmemBytes = smem;
  cfg.stream = st;
  cudaLaunchAttribute attr[1];
  attr[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
  attr[0].val.programmaticStreamSerializationAllowed = 1;
  cfg.attrs = attr;
  cfg.numAttrs = pdl ? 1 : 0;
  return cudaLaunchKernelEx(&cfg, kernel, std::forward<Args>(args)...);
}

#endif

struct DeviceGuard {
  int prev = -1;
  explicit DeviceGuard(int dev) {
    cudaGetDevice(&prev);
    if (prev != dev) cudaSetDevice(dev);
    else prev = -1;
  }
  ~DeviceGuard() {
    if (prev >= 0) cudaSetDevice(prev);
  }
};

// ---- letterbox tap tables (preprocess.cu builds them; filters.cu's fused pass reads them too) ----
struct __align__(16) TapX {
  int off0, off1;  // byte offsets of the two taps inside a source row; off0 < 0: pad column
  short a0, a1;    // 11-bit coefficients
  int mx0;         // x0 | (x1 << 16): pixel indices for the ROI mask row
};
struct __align__(16) TapY {
  int y0, y1;  // source rows; y0 < 0: pad row
  short b0, b1;
  int pad_;
};

// What the fused motion + letterbox pass needs for one (source size, letterbox geometry): arena offsets (in 16-byte
// entries) of the column / row tap tables, of rowmap[src_h] (destination row whose FIRST source row is r, or -1)
// and of colstart[strips + 1] (first destination column whose first tap lies in 256-pixel strip s).
struct FusePlan {
  int xtab, ytab, rowmap, colstart;
  bool eligible;  // every destination row taps rows (y0, y0 + 1) or y0 alone, y0 strictly increasing; same for columns
};
int letterbox_fuse_plan(b200va_ctx* h, int src_h, int src_w, int new_h, int new_w, int pad_top, int pad_left, int dst_h,
                        int dst_w, FusePlan* out);
const int4* tap_arena(b200va_ctx* h);

// The Ultralytics post-process options (b200va_postprocess_ultralytics, b200va_tick_ultralytics; postprocess.cu).
struct UltraOpts {
  const int* src_h;
  const int* src_w;
  int in_h, in_w, agnostic, max_det;
};

// per-module state owned by the handle
int tap_cache_create(b200va_ctx* h);
void tap_cache_destroy(b200va_ctx* h);
int tracker_state_create(b200va_ctx* h);
void tracker_state_destroy(b200va_ctx* h);

#ifdef __CUDACC__
__device__ __forceinline__ int warp_sum(int v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
  return v;
}

// programmatic dependent launch: a kernel launched with cudaLaunchAttributeProgrammaticStreamSerialization may start
// while its predecessor in the stream is still running; everything before griddep_wait() overlaps the predecessor's
// tail, everything after it sees the predecessor's writes (a no-op for ordinary launches)
__device__ __forceinline__ void griddep_wait() { asm volatile("griddepcontrol.wait;" ::: "memory"); }
__device__ __forceinline__ void griddep_launch_dependents() { asm volatile("griddepcontrol.launch_dependents;" ::: "memory"); }

// ---- mbarrier + 1-D bulk async copy (TMA engine, UBLKCP in SASS) -----------------------
__device__ __forceinline__ uint32_t smem_u32(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }

__device__ __forceinline__ void mbar_init(uint64_t* bar, uint32_t count) {
  asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count) : "memory");
}
__device__ __forceinline__ void mbar_fence_init() {
  asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
}
__device__ __forceinline__ void mbar_expect_tx(uint64_t* bar, uint32_t bytes) {
  asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)), "r"(bytes)
               : "memory");
}
__device__ __forceinline__ void mbar_arrive(uint64_t* bar) {
  asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(smem_u32(bar)) : "memory");
}
__device__ __forceinline__ void mbar_wait(uint64_t* bar, uint32_t parity) {
  asm volatile(
      "{\n"
      ".reg .pred p;\n"
      "WAIT_LOOP:\n"
      "mbarrier.try_wait.parity.shared::cta.b64 p, [%0], %1;\n"
      "@p bra DONE;\n"
      "bra WAIT_LOOP;\n"
      "DONE:\n"
      "}\n" ::"r"(smem_u32(bar)),
      "r"(parity)
      : "memory");
}
// global -> shared bulk copy; dst, src and bytes must be multiples of 16.
__device__ __forceinline__ void bulk_g2s(void* smem_dst, const void* gmem_src, uint32_t bytes, uint64_t* bar) {
  asm volatile(
      "cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(
          smem_u32(smem_dst)),
      "l"(gmem_src), "r"(bytes), "r"(smem_u32(bar))
      : "memory");
}

// 16-byte async global->shared copy (LDGSTS), L2-only caching: streamed frame rows.
__device__ __forceinline__ void cp_async16(void* smem_dst, const void* gmem_src) {
  asm volatile("cp.async.cg.shared.global [%0], [%1], 16;\n" ::"r"(smem_u32(smem_dst)), "l"(gmem_src) : "memory");
}
__device__ __forceinline__ void cp_async_commit() { asm volatile("cp.async.commit_group;\n" ::: "memory"); }
template <int N>
__device__ __forceinline__ void cp_async_wait() {
  asm volatile("cp.async.wait_group %0;\n" ::"n"(N) : "memory");
}

// ---- NV12 -> BGR (preprocess.cu's letterbox taps, egress.cu's INTER_AREA) ---------------------
// cv::cvtColor YUV2BGR_NV12 (modules/imgproc/src/color_yuv.simd.hpp, 8-bit path): ITU-R BT.601 limited range in
// 20-bit fixed point, rounded by the 1 << 19 bias and saturated.  `uv` = Cb | Cr << 8 of the pixel's 2 x 2 block.
// Returns the pixel packed as B | G << 8 | R << 16 (byte 3 is zero).
constexpr int kNv12Y = 1220542, kNv12UB = 2116026, kNv12VG = 852492, kNv12UG = 409993, kNv12VR = 1673527;
__device__ __forceinline__ uint32_t nv12_bgr(int Y, uint32_t uv) {
  const int y = max(Y - 16, 0) * kNv12Y + (1 << 19);
  const int u = (int)(uv & 0xffu) - 128, v = (int)(uv >> 8) - 128;
  const uint32_t b = (uint32_t)min(max((y + kNv12UB * u) >> 20, 0), 255);
  const uint32_t g = (uint32_t)min(max((y - kNv12VG * v - kNv12UG * u) >> 20, 0), 255);
  const uint32_t r = (uint32_t)min(max((y + kNv12VR * v) >> 20, 0), 255);
  return b | (g << 8) | (r << 16);
}

// The same conversion split for pixels that share one chroma pair (a 2 x 2 block starting at an even x and y): the
// three chroma terms once, then per luma value y = nv12_luma(Y) the channels (y + term) >> 20, saturated.  The sums
// are nv12_bgr's (no term overflows int), so each channel is bit for bit the same.  nv12_sat clamps before the shift,
// min(max(y + term, 0), 2^28 - 1) >> 20 == min(max((y + term) >> 20, 0), 255), as one fused add / min / relu
// (VIADDMNMX.RELU, sm_90 and later) and a shift instead of an add, a shift and two min / max.
__device__ __forceinline__ int nv12_luma(int Y) { return max(Y - 16, 0) * kNv12Y + (1 << 19); }
__device__ __forceinline__ int3 nv12_chroma(uint32_t uv) {
  const int u = (int)(uv & 0xffu) - 128, v = (int)(uv >> 8) - 128;
  return make_int3(kNv12UB * u, -kNv12VG * v - kNv12UG * u, kNv12VR * v);
}
__device__ __forceinline__ uint32_t nv12_sat(int y, int term) { return (uint32_t)(__viaddmin_s32_relu(y, term, (1 << 28) - 1) >> 20); }
#endif
