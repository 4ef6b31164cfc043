// a3-a7: YOLO head post-process for a batch of frames.
//
// Replaces _TensorRTBaseDetector._postprocess (detector.py:266-338), _xywh2xyxy (:352-359),
// _scale_boxes (:340-350), _nms (:361-375), _iou (:469-481) and filter_detections (:99-103).
// All float32 arithmetic uses explicit round-to-nearest intrinsics in NumPy's operation order
// (no FMA contraction, true division), so kept indices, scores and boxes are bit-identical.
//
//   k_decode_cm / k_decode_am   one pass over the head tensor (the only HBM-heavy step; k_decode16_* read a float16
//       head in place with the same code):
//       objectness x class score, first-max argmax, confidence / class filter, xywh -> xyxy,
//       un-letterbox, clip; survivors are compacted per frame with warp ballots.
//   k_sort_nms                  one CTA per frame: bitonic sort of (score, anchor) keys in shared
//       memory, then exact greedy NMS in 64-box chunks -- an in-chunk 64x64 IoU bit matrix
//       resolved by one warp, after which the chunk's survivors suppress every later box in
//       parallel -- and ordered emission with the float64 re-threshold folded in.
#include <cuda.h>  // CUtensorMap (types only: the encoder is fetched with cudaGetDriverEntryPoint)
#include <cuda_fp16.h>

#include <algorithm>
#include <cmath>

#include "common.cuh"
#include "tracker_body.cuh"

namespace {

struct PostFrame {
  float left, top, scale, xmax, ymax;
};

constexpr int kClassMaskIds = 2048;  // class ids the whitelist bitmap covers (the host refuses larger ids the head can produce)

struct PostParams {
  PostFrame f[B200VA_LAUNCH_FRAMES];
  uint32_t class_mask[kClassMaskIds / 32];  // whitelist bitmap over class ids (np.isin, detector.py:313-314)
  const void* head;  // float32, or float16 for the k_decode16_* kernels
  unsigned long long* cand_key;
  float4* cand_box;
  int32_t* cand_cls;
  int32_t* cand_count;
  int C, A, max_cand, use_mask;
  int cls0;     // first class channel: 5 (column 4 is objectness) or 4 (scores = pred[:, 4:])
  int use_obj;  // multiply class scores by column 4
  float conf_thr;
  long long* dbg;  // timing builds: timeline stamps
  const uint8_t* skip;  // device-side gates: frames with a non-zero flag are not decoded (indexed by frame0 + frame)
  int ultra;    // Ultralytics semantics: strict `>` threshold, boxes stay in network-input pixels, equal scores keep
                // the lower anchor first (torchvision's stable descending sort)
};
static_assert(sizeof(PostParams) <= 4000, "kernel parameter block too large");

__device__ __forceinline__ uint32_t order_bits(float v) {
  // monotone map float -> uint32 (larger float, larger integer)
  uint32_t b = __float_as_uint(v);
  return b ^ ((b & 0x80000000u) ? 0xffffffffu : 0x80000000u);
}
__device__ __forceinline__ float unorder_bits(uint32_t u) {
  uint32_t b = (u & 0x80000000u) ? (u ^ 0x80000000u) : ~u;
  return __uint_as_float(b);
}

// Candidate key, descending order = NMS order: [63:32] order_bits(score) | [31:14] anchor tie rule | [13] the score is
// -0.0 | [12:0] candidate slot (max_candidates <= 8192).  -0.0 and +0.0 rank equal, as NumPy and torch compare them:
// both take the key of +0.0 and bit 13 keeps the sign for the emitted confidence.  Bit 13 never decides an order
// because the tie field above it is unique within a frame.
constexpr unsigned long long kKeySlotMask = 0x1fffull;
constexpr unsigned long long kKeyNegZero = 1ull << 13;
__device__ __forceinline__ unsigned long long cand_key(float conf, uint32_t tie, int slot) {
  const bool neg_zero = __float_as_uint(conf) == 0x80000000u;
  return ((unsigned long long)order_bits(neg_zero ? 0.f : conf) << 32) | ((unsigned long long)tie << 14) |
         (neg_zero ? kKeyNegZero : 0ull) | (unsigned long long)(uint32_t)slot;
}
__device__ __forceinline__ float key_conf(unsigned long long k) {
  return (k & kKeyNegZero) ? -0.f : unorder_bits((uint32_t)(k >> 32));
}
__device__ __forceinline__ int key_slot(unsigned long long k) { return (int)(k & kKeySlotMask); }

// ultralytics scale_boxes + clip_boxes (utils/ops.py): un-pad, true division by float32(gain), clamp to [0, w] x [0, h]
// (torch CPU semantics; torch CUDA multiplies by the float32 reciprocal instead).
// NaN-propagating maximum / minimum (FMNMX.NAN / FMNMX3.NAN): the result is NaN as soon as one input is -- what
// np.maximum, np.minimum and np.clip do; fmaxf / fminf return the other operand instead
__device__ __forceinline__ float max_nan(float a, float b) {
  float d;
  asm("max.NaN.f32 %0, %1, %2;" : "=f"(d) : "f"(a), "f"(b));
  return d;
}
__device__ __forceinline__ float min_nan(float a, float b) {
  float d;
  asm("min.NaN.f32 %0, %1, %2;" : "=f"(d) : "f"(a), "f"(b));
  return d;
}
__device__ __forceinline__ float max3_nan(float a, float b, float c) {
  float d;
  asm("max.NaN.f32 %0, %1, %2, %3;" : "=f"(d) : "f"(a), "f"(b), "f"(c));
  return d;
}
__device__ __forceinline__ float clip_nan(float x, float lo, float hi) { return min_nan(max_nan(x, lo), hi); }  // np.clip

__device__ __forceinline__ float4 ultra_scale_box(float4 b, const PostFrame& f) {
  b.x = clip_nan(__fdiv_rn(__fsub_rn(b.x, f.left), f.scale), 0.f, f.xmax);  // (clamp_ keeps a NaN)
  b.y = clip_nan(__fdiv_rn(__fsub_rn(b.y, f.top), f.scale), 0.f, f.ymax);
  b.z = clip_nan(__fdiv_rn(__fsub_rn(b.z, f.left), f.scale), 0.f, f.xmax);
  b.w = clip_nan(__fdiv_rn(__fsub_rn(b.w, f.top), f.scale), 0.f, f.ymax);
  return b;
}

// detector.py:352-359 then :340-350, float32, NumPy operation order.  raw = true stops after xywh -> xyxy
// (ultralytics xywh2xyxy does the same two operations; its NMS runs on network-input pixels).
__device__ __forceinline__ float4 decode_box(float cx, float cy, float w, float h, const PostFrame& f, bool raw = false) {
  const float hw = __fmul_rn(w, 0.5f), hh = __fmul_rn(h, 0.5f);  // w / 2.0 is exact either way
  float x1 = __fsub_rn(cx, hw), y1 = __fsub_rn(cy, hh), x2 = __fadd_rn(cx, hw), y2 = __fadd_rn(cy, hh);
  if (raw) return make_float4(x1, y1, x2, y2);
  x1 = __fdiv_rn(__fsub_rn(x1, f.left), f.scale);
  x2 = __fdiv_rn(__fsub_rn(x2, f.left), f.scale);
  y1 = __fdiv_rn(__fsub_rn(y1, f.top), f.scale);
  y2 = __fdiv_rn(__fsub_rn(y2, f.top), f.scale);
  x1 = clip_nan(x1, 0.f, f.xmax);  // np.clip keeps a NaN (fminf / fmaxf would turn it into a frame edge)
  x2 = clip_nan(x2, 0.f, f.xmax);
  y1 = clip_nan(y1, 0.f, f.ymax);
  y2 = clip_nan(y2, 0.f, f.ymax);
  return make_float4(x1, y1, x2, y2);
}

__device__ __forceinline__ bool class_allowed(const PostParams& p, int cls) {
  if (!p.use_mask) return true;
  if (cls >= kClassMaskIds) return false;  // (never whitelisted: the host refuses such an id)
  return (p.class_mask[cls >> 5] >> (cls & 31)) & 1u;
}

__device__ __forceinline__ void emit_candidate(const PostParams& p, int frame, int pos, int anchor, float conf, int cls,
                                               float4 box) {
  if (pos >= p.max_cand) return;  // overflow is flagged by k_sort_nms from the raw count
  const size_t o = (size_t)frame * p.max_cand + pos;
  const uint32_t tie = p.ultra ? (0x3ffffu - (uint32_t)anchor) : (uint32_t)anchor;  // descending sort: which anchor first on equal scores
  p.cand_key[o] = cand_key(conf, tie, pos);
  p.cand_box[o] = box;
  p.cand_cls[o] = cls;
}

// Head elements.  The head is float32, or IEEE binary16 (B200VA_HEAD_F16); the decode bodies below are templates
// over that element type T, wrapped by one __global__ function per type.  HeadVec<T, N> is N consecutive elements
// of one channel row fetched by ONE load and held as loaded -- packed halves for float16, so the rows a thread keeps
// in flight cost N * sizeof(T) bytes of registers each -- and v[k] widens element k to float32 where it is used.
// float16 -> float32 is exact (subnormals included: cvt.f32.f16 does not flush), so everything after the load is
// the float32 code and an fp16 head decodes exactly like its float32 widening.
__device__ __forceinline__ float half_bits_to_float(uint32_t bits) { return __half2float(__ushort_as_half((unsigned short)bits)); }

template <typename T, int N>
struct HeadVec;
template <>
struct HeadVec<float, 1> {
  float q;
  __device__ __forceinline__ void load(const float* s) { q = __ldg(s); }
  __device__ __forceinline__ float operator[](int) const { return q; }
};
template <>
struct HeadVec<float, 4> {  // 16-byte load: 4-anchor aligned row offset, 16-byte aligned base
  float q[4];
  __device__ __forceinline__ void load(const float* s) {
    const float4 v = __ldg(reinterpret_cast<const float4*>(s));
    q[0] = v.x, q[1] = v.y, q[2] = v.z, q[3] = v.w;
  }
  __device__ __forceinline__ float operator[](int k) const { return q[k]; }
};
template <>
struct HeadVec<__half, 1> {
  __half q;
  __device__ __forceinline__ void load(const __half* s) { q = __ldg(s); }
  __device__ __forceinline__ float operator[](int) const { return __half2float(q); }
};
template <>
struct HeadVec<__half, 4> {  // 8-byte load
  uint2 q;
  __device__ __forceinline__ void load(const __half* s) { q = __ldg(reinterpret_cast<const uint2*>(s)); }
  __device__ __forceinline__ float operator[](int k) const {
    const uint32_t w = k < 2 ? q.x : q.y;
    return half_bits_to_float((k & 1) ? w >> 16 : w & 0xffffu);
  }
};
template <>
struct HeadVec<__half, 8> {  // 16-byte load
  uint4 q;
  __device__ __forceinline__ void load(const __half* s) { q = __ldg(reinterpret_cast<const uint4*>(s)); }
  __device__ __forceinline__ float operator[](int k) const {
    const uint32_t w = k < 2 ? q.x : k < 4 ? q.y : k < 6 ? q.z : q.w;
    return half_bits_to_float((k & 1) ? w >> 16 : w & 0xffffu);
  }
};
__device__ __forceinline__ float head_at(const float* s) { return __ldg(s); }
__device__ __forceinline__ float head_at(const __half* s) { return __half2float(__ldg(s)); }

// channel-major head [B, C, A].  A thread owns VEC consecutive anchors (one 16-byte load per channel
// row when VEC * sizeof(T) = 16) and walks the class rows in order; the next eight rows are already in flight
// while the current eight are scored (software double buffering), so ~16 independent 16-byte loads
// per thread keep HBM busy.
template <typename T, int VEC>
__device__ __forceinline__ void decode_cm(const PostParams& p, int frame0) {
  griddep_launch_dependents();  // the NMS kernel may start its prologue now; its griddep_wait() still waits for this grid
  TIMELINE_BEGIN(p.dbg, 40);
  const int frame = blockIdx.y;
  if (p.skip && p.skip[frame0 + frame]) return;
  const int lane = threadIdx.x & 31;
  const int a0 = (blockIdx.x * blockDim.x + threadIdx.x) * VEC;
  const T* __restrict__ hd = static_cast<const T*>(p.head) + (size_t)(frame0 + frame) * p.C * p.A;
  const int A = p.A, C = p.C;
  float best[VEC];
  int cls[VEC];
  unsigned pass = 0;      // bit k: anchor a0 + k is a candidate
  unsigned nan_seen = 0;  // bit k: some score of anchor a0 + k is NaN (np.argmax then lands on a NaN,
                          // whose confidence fails the >= filter: the anchor is never a candidate)
#pragma unroll
  for (int k = 0; k < VEC; ++k) {
    best[k] = 0.f;
    cls[k] = 0;
  }
  auto load = [&](int c, HeadVec<T, VEC>& v) { v.load(hd + (size_t)c * A + a0); };
  if (a0 < A) {
    float obj[VEC];
    if (p.use_obj) {
      HeadVec<T, VEC> o;
      load(4, o);
#pragma unroll
      for (int k = 0; k < VEC; ++k) obj[k] = o[k];
    } else {
#pragma unroll
      for (int k = 0; k < VEC; ++k) obj[k] = 1.0f;  // x * 1.0f is exact: scores = pred[:, 4:]
    }
    const int cls0 = p.cls0;
    {
      // REF_COMPAT: scores = class_probs * objectness for both model types (detector.py:294-305)
      HeadVec<T, VEC> first;
      load(cls0, first);
      HeadVec<T, VEC> cur[8], nxt[8];
      int c = cls0 + 1;
      const bool have0 = c + 8 <= C;
      if (have0) {
#pragma unroll
        for (int u = 0; u < 8; ++u) load(c + u, cur[u]);
      }
#pragma unroll
      for (int k = 0; k < VEC; ++k) {
        best[k] = __fmul_rn(first[k], obj[k]);
        nan_seen |= (unsigned)(best[k] != best[k]) << k;
      }
      while (c + 8 <= C) {
        const bool more = c + 16 <= C;
        if (more) {
#pragma unroll
          for (int u = 0; u < 8; ++u) load(c + 8 + u, nxt[u]);
        }
#pragma unroll
        for (int u = 0; u < 8; ++u)
#pragma unroll
          for (int k = 0; k < VEC; ++k) {
            const float sc = __fmul_rn(cur[u][k], obj[k]);
            nan_seen |= (unsigned)(sc != sc) << k;
            if (sc > best[k]) {  // np.argmax: first maximum wins
              best[k] = sc;
              cls[k] = c + u - cls0;
            }
          }
        c += 8;
        if (more) {
#pragma unroll
          for (int u = 0; u < 8; ++u) cur[u] = nxt[u];
        }
      }
      for (; c < C; ++c) {
        HeadVec<T, VEC> v;
        load(c, v);
#pragma unroll
        for (int k = 0; k < VEC; ++k) {
          const float sc = __fmul_rn(v[k], obj[k]);
          nan_seen |= (unsigned)(sc != sc) << k;
          if (sc > best[k]) {
            best[k] = sc;
            cls[k] = c - cls0;
          }
        }
      }
    }
#pragma unroll
    for (int k = 0; k < VEC; ++k)
      if (!((nan_seen >> k) & 1u) && (p.ultra ? best[k] > p.conf_thr : best[k] >= p.conf_thr) && class_allowed(p, cls[k]))
        pass |= 1u << k;
  }
  // warp-aggregated compaction: one atomic per warp
  const int mine = __popc(pass);
  int incl = mine;
#pragma unroll
  for (int o = 1; o < 32; o <<= 1) {
    const int t = __shfl_up_sync(0xffffffffu, incl, o);
    if (lane >= o) incl += t;
  }
  const int total = __shfl_sync(0xffffffffu, incl, 31);
  if (total == 0) {
    TIMELINE_END(p.dbg, 40);
    return;
  }
  int base = 0;
  if (lane == 31) base = atomicAdd(p.cand_count + frame, total);
  base = __shfl_sync(0xffffffffu, base, 31);
  int pos = base + incl - mine;
  if (pass) {
    HeadVec<T, VEC> cx, cy, w, h;
    load(0, cx);
    load(1, cy);
    load(2, w);
    load(3, h);
#pragma unroll
    for (int k = 0; k < VEC; ++k)
      if (pass & (1u << k)) {
        emit_candidate(p, frame, pos, a0 + k, best[k], cls[k], decode_box(cx[k], cy[k], w[k], h[k], p.f[frame], p.ultra != 0));
        ++pos;
      }
  }
  TIMELINE_END(p.dbg, 40);
}
template <int VEC>
__global__ void __launch_bounds__(64) k_decode_cm(const __grid_constant__ PostParams p, int frame0) {
  decode_cm<float, VEC>(p, frame0);
}
// float16 head: VEC = 8 (16-byte loads; A % 8 == 0, 16-byte aligned base) or 1
template <int VEC>
__global__ void __launch_bounds__(64) k_decode16_cm(const __grid_constant__ PostParams p, int frame0) {
  decode_cm<__half, VEC>(p, frame0);
}

// channel-major head, class rows split over the warps of a CTA -- the SMALL-BATCH variant.  k_decode_cm walks its
// 80-odd rows in ~10 dependent rounds of loads; with a few frames per launch (4 streams per GPU when 32 streams are
// sharded over 8 GPUs) nothing overlaps those round trips and one frame costs 12.7 us.  Here lane l of EVERY warp owns
// the same four anchors; warp j scores rows [cls0 + j*per, cls0 + (j+1)*per) with all of its loads in flight at once
// (a warp still reads 512 contiguous bytes per row), the partial (best, class) pairs meet in shared memory and warp 0
// merges them in class order -- `>` keeps the first maximum, exactly np.argmax -- then compacts and emits as before.
// At 32 frames per launch the kernel is HBM-bound and this variant is slower (22 us against 20 us): the host picks.
// The float16 variant keeps four anchors per lane (8-byte loads: A % 4 == 0, 8-byte aligned base).
template <typename T, int kSplitParts, int kSplitRows>  // kSplitRows: rows one warp holds in flight (<= kSplitParts * kSplitRows class rows)
__device__ __forceinline__ void decode_cm_split(const PostParams& p, int frame0) {
  griddep_launch_dependents();  // the NMS kernel may start its prologue now; its griddep_wait() still waits for this grid
  __shared__ float s_best[kSplitParts - 1][4][32];
  __shared__ int s_cls[kSplitParts - 1][4][32];
  __shared__ unsigned s_nan[kSplitParts - 1][32];
  const int frame = blockIdx.y;
  if (p.skip && p.skip[frame0 + frame]) return;
  TIMELINE_BEGIN(p.dbg, 40);
  const int lane = threadIdx.x & 31, part = threadIdx.x >> 5;
  const int a0 = (blockIdx.x * 32 + lane) * 4;
  const int A = p.A, C = p.C, cls0 = p.cls0;
  const T* __restrict__ hd = static_cast<const T*>(p.head) + (size_t)(frame0 + frame) * C * A;
  const int per = (C - cls0 + kSplitParts - 1) / kSplitParts;
  const int c_lo = cls0 + part * per, c_hi = min(C, c_lo + per);
  const bool in_range = a0 < A;
  float best[4] = {0.f, 0.f, 0.f, 0.f};
  int cls[4] = {0, 0, 0, 0};
  unsigned nan_seen = 0;
  bool any = false;
  // the warp that emits (part 0) fetches the four box rows together with its class rows: one round of loads per launch
  // instead of a second, dependent one for the anchors that pass (a launch of a few frames is latency-bound)
  HeadVec<T, 4> cx{}, cy{}, w{}, hh{};
  if (part == 0 && in_range) {
    cx.load(hd + a0);
    cy.load(hd + (size_t)A + a0);
    w.load(hd + (size_t)2 * A + a0);
    hh.load(hd + (size_t)3 * A + a0);
  }
  if (in_range && c_lo < c_hi) {
    any = true;
    float obj[4] = {1.f, 1.f, 1.f, 1.f};  // x * 1.0f is exact: scores = pred[:, 4:]
    if (p.use_obj) {
      HeadVec<T, 4> o;
      o.load(hd + (size_t)4 * A + a0);
#pragma unroll
      for (int k = 0; k < 4; ++k) obj[k] = o[k];
    }
    HeadVec<T, 4> v[kSplitRows];
#pragma unroll
    for (int u = 0; u < kSplitRows; ++u)
      if (c_lo + u < c_hi) v[u].load(hd + (size_t)(c_lo + u) * A + a0);
#pragma unroll
    for (int u = 0; u < kSplitRows; ++u)
      if (c_lo + u < c_hi) {
        const float sc[4] = {__fmul_rn(v[u][0], obj[0]), __fmul_rn(v[u][1], obj[1]), __fmul_rn(v[u][2], obj[2]),
                             __fmul_rn(v[u][3], obj[3])};
#pragma unroll
        for (int k = 0; k < 4; ++k) {
          nan_seen |= (unsigned)(sc[k] != sc[k]) << k;
          if (u == 0 || sc[k] > best[k]) {  // np.argmax: first maximum wins
            best[k] = sc[k];
            cls[k] = c_lo + u - cls0;
          }
        }
      }
  }
  if (part > 0) {
#pragma unroll
    for (int k = 0; k < 4; ++k) {
      s_best[part - 1][k][lane] = any ? best[k] : __int_as_float(0xff800000);  // -inf never wins a `>`
      s_cls[part - 1][k][lane] = cls[k];
    }
    s_nan[part - 1][lane] = nan_seen;
  }
  __syncthreads();
  if (part > 0) return;
  unsigned pass = 0;
  if (in_range) {
#pragma unroll
    for (int j = 0; j < kSplitParts - 1; ++j) {
      nan_seen |= s_nan[j][lane];
#pragma unroll
      for (int k = 0; k < 4; ++k) {
        const float b = s_best[j][k][lane];
        if (b > best[k]) {
          best[k] = b;
          cls[k] = s_cls[j][k][lane];
        }
      }
    }
#pragma unroll
    for (int k = 0; k < 4; ++k)
      if (!((nan_seen >> k) & 1u) && (p.ultra ? best[k] > p.conf_thr : best[k] >= p.conf_thr) && class_allowed(p, cls[k]))
        pass |= 1u << k;
  }
  // warp-aggregated compaction: one atomic per warp
  const int mine = __popc(pass);
  int incl = mine;
#pragma unroll
  for (int o = 1; o < 32; o <<= 1) {
    const int t = __shfl_up_sync(0xffffffffu, incl, o);
    if (lane >= o) incl += t;
  }
  const int total = __shfl_sync(0xffffffffu, incl, 31);
  TIMELINE_END(p.dbg, 40);  // (warps with survivors run a little longer)
  if (total == 0) return;
  int base = 0;
  if (lane == 31) base = atomicAdd(p.cand_count + frame, total);
  base = __shfl_sync(0xffffffffu, base, 31);
  int pos = base + incl - mine;
  if (pass) {
#pragma unroll
    for (int k = 0; k < 4; ++k)
      if (pass & (1u << k)) {
        emit_candidate(p, frame, pos, a0 + k, best[k], cls[k], decode_box(cx[k], cy[k], w[k], hh[k], p.f[frame], p.ultra != 0));
        ++pos;
      }
  }
}
template <int kSplitParts, int kSplitRows>
__global__ void __launch_bounds__(32 * kSplitParts) k_decode_cm_split(const __grid_constant__ PostParams p, int frame0) {
  decode_cm_split<float, kSplitParts, kSplitRows>(p, frame0);
}
__global__ void __launch_bounds__(256) k_decode16_cm_split(const __grid_constant__ PostParams p, int frame0) {
  decode_cm_split<__half, 8, 12>(p, frame0);
}

// channel-major head, TMA-fed and persistent -- the LARGE-BATCH variant.  k_decode_cm is a one-wave kernel whose CTAs
// walk the class rows in lock step: every thread waits ~10 dependent load round trips, nothing is in flight while the
// last one drains and the epilogue runs, and launch, ramp and tail are paid on a 14 us stream (0.70 of the HBM peak
// at [32, 84, 8400]).  Here a CTA is a producer warp plus consumer warps around a shared-memory ring, like
// k_letterbox / k_motion_tile: one elected lane feeds the bulk-copy engine (cp.async.bulk -> UBLKCP) with row pieces
// of `ta` anchors (1-2 KB each), `rows` channel rows per stage, always `stages` stages ahead and running on into the
// CTA's next tile while the consumers finish the current one; consumer thread g owns anchors 4g..4g+3 of the tile
// and reads its rows from shared memory with conflict-free 16-byte loads.  The grid is sized so that every CTA is
// resident and owns the same number of tiles: all CTAs share the bus equally and finish together.
constexpr int kRingMaxStages = 8;
constexpr int kRingWarps = 4;  // consumer warps -> tiles of up to 512 anchors
struct RingCfg {
  int ta;               // anchors per tile = boxes * bw
  int bw;               // anchors per TMA box (<= 256: the box-dimension limit), multiple of 4
  int boxes;            // boxes per stage (1 or 2)
  int rows;             // channel rows per stage (= box height, >= cls0 + 1)
  int stages;           // ring depth
  int tiles_per_frame;  // ceil(A / ta)
  int n_tiles;          // tiles_per_frame * frames of the launch
  int warps;            // consumer warps that own anchors: ceil(ta / 128)
};

// candidate filter + warp-aggregated compaction + emit for the four anchors a0..a0+3 of one thread; called by all 32
// lanes of a warp (lanes without anchors pass in_range = false)
__device__ __forceinline__ void emit_quad(const PostParams& p, int frame, int lane, int a0, bool in_range, const float (&best)[4],
                                          const int (&cls)[4], unsigned nan_seen, const float4 cx, const float4 cy,
                                          const float4 w, const float4 h) {
  unsigned pass = 0;
  if (in_range) {
#pragma unroll
    for (int k = 0; k < 4; ++k)
      if (!((nan_seen >> k) & 1u) && (p.ultra ? best[k] > p.conf_thr : best[k] >= p.conf_thr) && class_allowed(p, cls[k]))
        pass |= 1u << k;
  }
  const int mine = __popc(pass);
  int incl = mine;
#pragma unroll
  for (int o = 1; o < 32; o <<= 1) {
    const int t = __shfl_up_sync(0xffffffffu, incl, o);
    if (lane >= o) incl += t;
  }
  const int total = __shfl_sync(0xffffffffu, incl, 31);
  if (total == 0) return;
  int base = 0;
  if (lane == 31) base = atomicAdd(p.cand_count + frame, total);
  base = __shfl_sync(0xffffffffu, base, 31);
  int pos = base + incl - mine;
  if (pass) {
    const float cxa[4] = {cx.x, cx.y, cx.z, cx.w}, cya[4] = {cy.x, cy.y, cy.z, cy.w};
    const float wa[4] = {w.x, w.y, w.z, w.w}, ha[4] = {h.x, h.y, h.z, h.w};
#pragma unroll
    for (int k = 0; k < 4; ++k)
      if (pass & (1u << k)) {
        emit_candidate(p, frame, pos, a0 + k, best[k], cls[k], decode_box(cxa[k], cya[k], wa[k], ha[k], p.f[frame], p.ultra != 0));
        ++pos;
      }
  }
}

// One stage = `rows` consecutive channel rows of a tile, fetched by ONE tensor-map copy per 256-anchor box
// (cp.async.bulk.tensor.3d -> UTMALDG): coordinates (anchor, channel, frame) of a [B, C, A] float32 tensor; rows past C
// and anchors past A are out of bounds for the map and arrive as zeros without touching memory.  Row-by-row 1-D bulk
// copies are NOT an option here: one thread sustains only ~4 M cp.async.bulk per second (250 ns each, measured with
// tools/scratch/readbw.cu), so 1-2 KB row pieces cap a CTA at 4-8 GB/s -- 2 KB pieces reached 3.1 TB/s, 1 KB 1.8 TB/s.
__device__ __forceinline__ void tma_load_3d(void* smem_dst, const CUtensorMap* map, int c0, int c1, int c2, uint64_t* bar) {
  asm volatile(
      "cp.async.bulk.tensor.3d.shared::cluster.global.tile.mbarrier::complete_tx::bytes [%0], [%1, {%2, %3, %4}], [%5];" ::"r"(
          smem_u32(smem_dst)),
      "l"(reinterpret_cast<uint64_t>(map)), "r"(c0), "r"(c1), "r"(c2), "r"(smem_u32(bar))
      : "memory");
}

__global__ void __launch_bounds__(32 * (kRingWarps + 1)) k_decode_ring(const __grid_constant__ PostParams p, int frame0,
                                                                        const RingCfg rc,
                                                                        const __grid_constant__ CUtensorMap tmap) {
  extern __shared__ __align__(128) uint8_t s_ring[];
  __shared__ __align__(8) uint64_t full[kRingMaxStages], empty[kRingMaxStages];
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int C = p.C, A = p.A, S = rc.stages, cls0 = p.cls0;
  const uint32_t box_bytes = (uint32_t)rc.rows * (uint32_t)rc.bw * 4u;
  const uint32_t stage_bytes = box_bytes * (uint32_t)rc.boxes;
  griddep_launch_dependents();
  if (threadIdx.x == 0) {
    for (int s = 0; s < S; ++s) {
      mbar_init(&full[s], 1);
      mbar_init(&empty[s], (uint32_t)rc.warps);
    }
    mbar_fence_init();
  }
  __syncthreads();

  if (warp == kRingWarps) {
    // ---- producer: one lane drives the TMA engine, a ring ahead of the consumers ----
    if (lane != 0) return;
    asm volatile("prefetch.tensormap [%0];" ::"l"(reinterpret_cast<uint64_t>(&tmap)) : "memory");
    int st = 0, use = 0;
    for (int tile = blockIdx.x; tile < rc.n_tiles; tile += gridDim.x) {
      const int frame = tile / rc.tiles_per_frame;
      const int a0 = (tile - frame * rc.tiles_per_frame) * rc.ta;
      for (int r0 = 0; r0 < C; r0 += rc.rows) {
        if (use > 0) mbar_wait(&empty[st], (uint32_t)(use - 1) & 1u);
        const int nb = min(rc.boxes, (A - a0 + rc.bw - 1) / rc.bw);  // boxes wholly past the last anchor are not fetched
        mbar_expect_tx(&full[st], (uint32_t)nb * box_bytes);
        uint8_t* dst = s_ring + (size_t)st * stage_bytes;
        for (int b = 0; b < nb; ++b) tma_load_3d(dst + (size_t)b * box_bytes, &tmap, a0 + b * rc.bw, r0, frame, &full[st]);  // the map starts at frame0
        if (++st == S) {
          st = 0;
          ++use;
        }
      }
    }
    return;
  }
  if (warp >= rc.warps) return;

  // ---- consumers: thread g owns anchors 4g .. 4g+3 of the tile ----
  // The class scan is the instruction-heavy part (80 rows x 4 anchors per thread): rows are taken four at a time,
  // the group's maximum (FMNMX3) is compared with the running best, and only the index of the winning GROUP is
  // kept -- 9 instructions per anchor and group instead of ~11 per anchor and ROW.  `>` on the group maxima keeps
  // the first group that reaches the overall maximum and emit resolves the first row inside it (np.argmax: first
  // maximum wins).  The maxima are NaN-propagating: one NaN score turns `best` into NaN for good, which fails the
  // confidence filter exactly like NumPy's argmax landing on the NaN does.
  const int g = warp * 32 + lane;
  const int ta = rc.ta, bw = rc.bw;
  const int gbox = (4 * g) / bw;                                 // which box of a stage holds this thread's anchors
  const uint32_t goff = (uint32_t)gbox * box_bytes + (uint32_t)(4 * g - gbox * bw) * 4u;
  const float ninf = __int_as_float(0xff800000);
  int st = 0;
  uint32_t ph = 0;
  for (int tile = blockIdx.x; tile < rc.n_tiles; tile += gridDim.x) {
    const int frame = tile / rc.tiles_per_frame;
    const int a_tile = (tile - frame * rc.tiles_per_frame) * ta;
    const bool active = 4 * g < min(ta, A - a_tile);
    float4 cx, cy, bwid, bh, obj = make_float4(1.f, 1.f, 1.f, 1.f);  // x * 1.0f is exact: scores = pred[:, 4:]
    float best[4] = {ninf, ninf, ninf, ninf};
    int grp[4] = {0, 0, 0, 0};  // first class of the winning group
    for (int r0 = 0; r0 < C; r0 += rc.rows) {
      const int r1 = min(C, r0 + rc.rows);
      mbar_wait(&full[st], ph);
      const float* rowp = reinterpret_cast<const float*>(s_ring + (size_t)st * stage_bytes + (active ? goff : 0u));
      if (r0 == 0) {
        cx = *reinterpret_cast<const float4*>(rowp);
        cy = *reinterpret_cast<const float4*>(rowp + bw);
        bwid = *reinterpret_cast<const float4*>(rowp + 2 * bw);
        bh = *reinterpret_cast<const float4*>(rowp + 3 * bw);
        if (p.use_obj) obj = *reinterpret_cast<const float4*>(rowp + 4 * bw);  // column 4 as objectness (detector.py:294-305)
        rowp += (size_t)cls0 * bw;
      }
      int c = (r0 == 0 ? cls0 : r0) - cls0;  // class index of the stage's first class row
      const int c_end = r1 - cls0;
      for (; c + 4 <= c_end; c += 4, rowp += 4 * bw) {
        const float4 v0 = *reinterpret_cast<const float4*>(rowp), v1 = *reinterpret_cast<const float4*>(rowp + bw);
        const float4 v2 = *reinterpret_cast<const float4*>(rowp + 2 * bw), v3 = *reinterpret_cast<const float4*>(rowp + 3 * bw);
        const float m[4] = {
            max_nan(max3_nan(__fmul_rn(v0.x, obj.x), __fmul_rn(v1.x, obj.x), __fmul_rn(v2.x, obj.x)), __fmul_rn(v3.x, obj.x)),
            max_nan(max3_nan(__fmul_rn(v0.y, obj.y), __fmul_rn(v1.y, obj.y), __fmul_rn(v2.y, obj.y)), __fmul_rn(v3.y, obj.y)),
            max_nan(max3_nan(__fmul_rn(v0.z, obj.z), __fmul_rn(v1.z, obj.z), __fmul_rn(v2.z, obj.z)), __fmul_rn(v3.z, obj.z)),
            max_nan(max3_nan(__fmul_rn(v0.w, obj.w), __fmul_rn(v1.w, obj.w), __fmul_rn(v2.w, obj.w)), __fmul_rn(v3.w, obj.w))};
#pragma unroll
        for (int k = 0; k < 4; ++k) {
          grp[k] = m[k] > best[k] ? c : grp[k];
          best[k] = max_nan(best[k], m[k]);
        }
      }
      for (; c < c_end; ++c, rowp += bw) {  // fewer than four rows left in the stage: groups of one
        const float4 v = *reinterpret_cast<const float4*>(rowp);
        const float m[4] = {__fmul_rn(v.x, obj.x), __fmul_rn(v.y, obj.y), __fmul_rn(v.z, obj.z), __fmul_rn(v.w, obj.w)};
#pragma unroll
        for (int k = 0; k < 4; ++k) {
          grp[k] = m[k] > best[k] ? c : grp[k];
          best[k] = max_nan(best[k], m[k]);
        }
      }
      __syncwarp();
      if (lane == 0) mbar_arrive(&empty[st]);
      if (++st == S) {
        st = 0;
        ph ^= 1u;
      }
    }
    // resolve the class of the (rare) anchors that pass the confidence filter: first row of the winning group whose
    // score equals the maximum; the rows come back from L2.  That row's score is the confidence: max.NaN.f32 makes
    // +0.0 of a -0.0 / +0.0 pair, np.argmax sees them equal and reports the first
    int cls[4] = {0, 0, 0, 0};
    if (active) {
      const float* hd = static_cast<const float*>(p.head) + (size_t)(frame0 + frame) * C * A + a_tile + 4 * g;
      const float oa[4] = {obj.x, obj.y, obj.z, obj.w};
#pragma unroll
      for (int k = 0; k < 4; ++k) {
        if (!(p.ultra ? best[k] > p.conf_thr : best[k] >= p.conf_thr)) continue;
        cls[k] = grp[k];
        for (int j = 0; j < 4 && grp[k] + j < C - cls0; ++j) {
          const float s = __fmul_rn(__ldg(hd + (size_t)(cls0 + grp[k] + j) * A + k), oa[k]);
          if (s == best[k]) {
            cls[k] = grp[k] + j;
            best[k] = s;
            break;
          }
        }
      }
    }
    emit_quad(p, frame, lane, a_tile + 4 * g, active, best, cls, 0u, cx, cy, bwid, bh);
  }
}

// anchor-major head [B, A, C]: a warp owns one anchor and strides its lanes over the channels
template <typename T>
__device__ __forceinline__ void decode_am(const PostParams& p, int frame0) {
  griddep_launch_dependents();  // the NMS kernel may start its prologue now; its griddep_wait() still waits for this grid
  const int frame = blockIdx.y;
  if (p.skip && p.skip[frame0 + frame]) return;
  const int lane = threadIdx.x & 31;
  const int a = blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
  if (a >= p.A) return;
  const int C = p.C;
  const T* __restrict__ row = static_cast<const T*>(p.head) + ((size_t)(frame0 + frame) * p.A + a) * C;
  const float obj = p.use_obj ? head_at(row + 4) : 1.0f;
  const int cls0 = p.cls0;
  float best = -INFINITY;
  int cls = 0x7fffffff;
  bool have = false, bad = false;
  for (int c = cls0 + lane; c < C; c += 32) {
    const float s = __fmul_rn(head_at(row + c), obj);
    bad |= (s != s);
    if (!have || s > best) {
      best = s;
      cls = c - cls0;
      have = true;
    }
  }
  // a NaN score makes np.argmax land on it and the >= filter drop the anchor
  bad = __any_sync(0xffffffffu, bad);
  if (!(best == best)) best = -INFINITY;
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) {
    const float ob = __shfl_xor_sync(0xffffffffu, best, o);
    const int oc = __shfl_xor_sync(0xffffffffu, cls, o);
    if (oc != 0x7fffffff && (cls == 0x7fffffff || ob > best || (ob == best && oc < cls))) {
      best = ob;
      cls = oc;
    }
  }
  if (bad) return;
  if (lane == 0) {
    if ((p.ultra ? best > p.conf_thr : best >= p.conf_thr) && class_allowed(p, cls)) {
      const int pos = atomicAdd(p.cand_count + frame, 1);
      emit_candidate(p, frame, pos, a, best, cls,
                     decode_box(head_at(row), head_at(row + 1), head_at(row + 2), head_at(row + 3), p.f[frame], p.ultra != 0));
    }
  }
}
__global__ void __launch_bounds__(256) k_decode_am(const __grid_constant__ PostParams p, int frame0) { decode_am<float>(p, frame0); }
__global__ void __launch_bounds__(256) k_decode16_am(const __grid_constant__ PostParams p, int frame0) { decode_am<__half>(p, frame0); }

// ---- sort + NMS + emit ----------------------------------------------------------------------

struct NmsParams {
  const unsigned long long* cand_key;
  const float4* cand_box;
  const int32_t* cand_cls;
  int32_t* cand_count;  // read, then reset to 0 for the next call
  int32_t* flags;
  float* out_box;
  float* out_conf;
  int32_t* out_cls;
  int32_t* out_count;
  int max_cand, max_dets, cap_pow2;
  float iou_thr;
  double filter_thr;
  int use_filter;
  int class_aware;  // 0: the reference's class-agnostic NMS (detector.py:361-375); 1: suppress same class only
  long long* dbg;
  // Ultralytics semantics (ops.non_max_suppression + scale_boxes): NMS on network-input boxes shifted by
  // class * 7680 in float32 (0 when agnostic), torchvision's IoU test, at most max_det_cap boxes kept, then
  // un-letterbox with f[frame]
  int ultra, ultra_agnostic, max_det_cap;
  int grid_off;  // byte offset of the NmsGrid in dynamic shared memory; 0 = no grid (survivors-vs-tail scan instead)
  int* stats;    // host-mapped word: set by frames with more than 256 candidates (the host picks the next variant from it)
  double iou_thr64;
  const uint8_t* skip;  // device-side gates (already offset to this launch's first frame): flagged frames emit nothing
  int dbg_reps;         // timing builds only
  PostFrame f[B200VA_LAUNCH_FRAMES];
};
static_assert(sizeof(NmsParams) <= 4000, "kernel parameter block too large");

// _iou of detector.py:469-481 in float32; returns true when box j must be suppressed by box i.
__device__ __forceinline__ bool suppresses(const float4 a, const float4 b, float thr) {
  // np.maximum / np.minimum / np.clip propagate NaN: a box with a NaN coordinate has IoU NaN with every box, and
  // `iou <= thr` is False for NaN -- it suppresses, and is suppressed by, everything
  const float x1 = max_nan(a.x, b.x), y1 = max_nan(a.y, b.y), x2 = min_nan(a.z, b.z), y2 = min_nan(a.w, b.w);
  const float iw = max_nan(0.f, __fsub_rn(x2, x1)), ih = max_nan(0.f, __fsub_rn(y2, y1));
  const float inter = __fmul_rn(iw, ih);
  const float area_a = __fmul_rn(__fsub_rn(a.z, a.x), __fsub_rn(a.w, a.y));
  const float area_b = __fmul_rn(__fsub_rn(b.z, b.x), __fsub_rn(b.w, b.y));
  const float uni = __fsub_rn(__fadd_rn(area_a, area_b), inter);
  // disjoint boxes (the common case): 0 / max(union, 1e-6) is exactly +-0 for any finite union
  if (inter == 0.f && fabsf(uni) <= 3.0e38f) return !(0.f <= thr);
  const float iou = __fdiv_rn(inter, max_nan(uni, 1e-6f));
  return !(iou <= thr);
}

// A box with a NaN coordinate has IoU NaN with every box whatever its other coordinates say (NaN * 0 is NaN), so the
// "these two are apart on one axis: IoU 0" short-cuts must not see the finite coordinates of such a box: the NMS
// kernels work on this view of it (every coordinate NaN; the predicate is the same) and emit the box as decoded.
__device__ __forceinline__ float4 nan_box_view(float4 b) {
  const bool ok = b.x == b.x && b.y == b.y && b.z == b.z && b.w == b.w;
  const float q = __int_as_float(0x7fffffff);
  return ok ? b : make_float4(q, q, q, q);
}

// torchvision.ops.nms (csrc/ops/cpu/nms_kernel.cpp): inter / (area_i + area_j - inter) > thr, no epsilon.
__device__ __forceinline__ bool suppresses_tv(const float4 a, const float4 b, double thr) {
  const float x1 = fmaxf(a.x, b.x), y1 = fmaxf(a.y, b.y), x2 = fminf(a.z, b.z), y2 = fminf(a.w, b.w);
  const float iw = fmaxf(0.f, __fsub_rn(x2, x1)), ih = fmaxf(0.f, __fsub_rn(y2, y1));
  const float inter = __fmul_rn(iw, ih);
  const float area_a = __fmul_rn(__fsub_rn(a.z, a.x), __fsub_rn(a.w, a.y));
  const float area_b = __fmul_rn(__fsub_rn(b.z, b.x), __fsub_rn(b.w, b.y));
  const float iou = __fdiv_rn(inter, __fsub_rn(__fadd_rn(area_a, area_b), inter));
  return (double)iou > thr;  // NaN (0 / 0) never suppresses
}

// Uniform grid over the frame for the kept boxes (reference mode: boxes are clipped to the frame, so every
// coordinate is finite and inside [0, xmax] x [0, ymax]).  A candidate can only be suppressed by a kept box it
// overlaps, and two overlapping boxes share at least one cell, so a candidate is tested against the kept boxes
// registered in the cells it touches (plus the overflow list: boxes that span too many cells or hit a full cell)
// instead of against every survivor of every earlier chunk: O(candidates x local density) instead of
// O(candidates x kept).
constexpr int kGX = 16, kGY = 12, kCells = kGX * kGY, kCellCap = 32, kMaxCellsPerBox = 24;
struct NmsGrid {
  int cnt[kCells];
  int n_over;
  int pad_[3];
  uint16_t list[kCells][kCellCap];
  // followed by: uint32_t over_mark[cap_pow2 / 32]; uint16_t over[cap_pow2];
};
__device__ __forceinline__ void cell_range(const float4 b, float inv_w, float inv_h, int& cx0, int& cx1, int& cy0, int& cy1) {
  cx0 = min(kGX - 1, max(0, (int)(b.x * inv_w)));
  cx1 = min(kGX - 1, max(0, (int)(b.z * inv_w)));
  cy0 = min(kGY - 1, max(0, (int)(b.y * inv_h)));
  cy1 = min(kGY - 1, max(0, (int)(b.w * inv_h)));
  if (cx1 < cx0) cx1 = cx0;  // inverted boxes (negative width) never overlap anything; keep the range well formed
  if (cy1 < cy0) cy1 = cy0;
}

constexpr int kNmsThreads = 1024;     // k_sort_nms
constexpr int kNmsThreadsSmall = 256;  // k_post_track: sparse scenes, NMS and tracker of a stream in one CTA

// Sort + NMS + emit of one frame by one CTA of NT threads.
// GRID: carries the kept-box grid code.  Two instantiations because the grid path's registers and stack slots slow
// the common small-n launch (which never runs it) from 9.5 to 14 us when it is compiled in; the host picks per launch
// from the candidate counts the previous launch reported (NmsParams::stats).
// Small frames (n <= kSmallN candidates) use their own compact shared-memory layout and a barrier-light schedule:
// ONE round of global loads (count, keys, boxes and classes of the first kSmallN slots are fetched together,
// before the count is known), rank sort, gather from shared memory, the whole symmetric n x n suppression bit matrix
// at once with all threads, then ONE warp resolves the greedy recursion chunk by chunk from the matrix alone (the
// ballot fixed point per 64 boxes, kept rows OR-ed into the suppression bitmap of the later chunks).  Six block
// barriers in total instead of four per 64-box chunk; measured on 72 candidates: 15.4 k -> ~7 k SM cycles.
constexpr int kSmallN = 256;
constexpr int kSmallPairs = 1536;
struct SmallNms {
  unsigned long long keys[kSmallN];
  unsigned long long sorted[kSmallN];
  float4 box[kSmallN];   // sorted order (class-shifted in Ultralytics mode)
  float4 ubox[kSmallN];  // by candidate slot, as decoded
  int ucls[kSmallN];     // by candidate slot
  uint16_t scl[kSmallN]; // sorted order
  uint32_t M[kSmallN][kSmallN / 32];  // M[i] bit j: boxes i and j suppress each other (symmetric predicate)
  uint32_t supp[kSmallN / 32], keep_w[kSmallN / 32];
  int keep_off[kSmallN / 64 + 1];
  int n_pairs;
  uint32_t pairs[kSmallPairs];  // pairs that are not disjoint: lo | hi << 16
};

// What the fused kernel's NMS half leaves in shared memory for its tracker half (k_post_track): the first chunk of
// detections already converted the way the tracker stages them, and the detection count.
struct DetHandover {
  TrkShared* sh;
  double scale;
  int has_scale;
};

// Sort + NMS + emit of one frame by one CTA of NT threads.
// GRID: carries the kept-box grid code.  Two instantiations because the grid path's registers and stack slots slow
// the common small-n launch (which never runs it) from 9.5 to 14 us when it is compiled in; the host picks per launch
// from the candidate counts the previous launch reported (NmsParams::stats).
// Bitonic sort of np2 (a power of two >= 64) 64-bit keys in shared memory, descending, by a CTA of NT threads; ends with
// a block barrier.  Only the warps that own a compare-exchange take part (named barrier 1).  Thread q owns the q-th
// pair of a step; for j <= 32 the 32 pairs of a warp lie inside one aligned block of 64 keys, so consecutive steps
// with j <= 32 depend on nothing another warp writes and a __syncwarp separates them; the block-wide barrier is paid
// only around the steps with j > 32 (20 of the 66 steps at 2048 keys).
template <int NT>
__device__ __forceinline__ void block_bitonic_sort_desc(unsigned long long* keys, const int np2) {
  const int tid = threadIdx.x;
  const int sort_threads = min(NT, max(32, np2 >> 1));
  if (tid < sort_threads) {
    for (int k = 2; k <= np2; k <<= 1) {
      for (int j = k >> 1; j > 0; j >>= 1) {
        for (int q = tid; q < (np2 >> 1); q += sort_threads) {
          // q-th pair of this round: i has bit j clear
          const int i = ((q & ~(j - 1)) << 1) | (q & (j - 1));
          const int ixj = i | j;
          const unsigned long long a = keys[i], b = keys[ixj];
          const bool desc = (i & k) == 0;
          if (desc ? (a < b) : (a > b)) {
            keys[i] = b;
            keys[ixj] = a;
          }
        }
        const int j_next = j > 1 ? (j >> 1) : k;  // first step of the next stage has j = (2k) / 2 = k
        if (sort_threads == 32 || (j <= 32 && j_next <= 32)) __syncwarp();
        else asm volatile("bar.sync 1, %0;" ::"r"(sort_threads) : "memory");
      }
    }
  }
  __syncthreads();
}

// The general path of nms_frame (more than kSmallN candidates): bitonic sort, greedy NMS in 64-box chunks, emit.
// Deliberately NOT inlined: the latency-bound CTAs of a sparse tick stall on instruction fetch more than on anything
// else (ncu: stall_no_inst 29-33 % of all samples in k_post_track), so the code a small frame never runs must not
// sit between the lines it does run.
template <bool GRID, int NT>
__device__ __forceinline__ void nms_general_body(const NmsParams& p, const int frame, uint8_t* const smem_raw, const int n) {
  const int tid = threadIdx.x;
  const size_t cbase = (size_t)frame * p.max_cand;
  int np2 = 64;
  while (np2 < n) np2 <<= 1;
  constexpr bool small = false;
  unsigned long long* keys = reinterpret_cast<unsigned long long*>(smem_raw);              // [cap_pow2]
  float4* box = reinterpret_cast<float4*>(smem_raw + (size_t)p.cap_pow2 * 8);               // [cap_pow2]
  uint32_t* supp = reinterpret_cast<uint32_t*>(smem_raw + (size_t)p.cap_pow2 * 24);         // [cap_pow2/32]
  uint32_t* keep_w = supp + p.cap_pow2 / 32;                                                // [cap_pow2/32]
  int* keep_off = reinterpret_cast<int*>(keep_w + p.cap_pow2 / 32);                         // [cap_pow2/64 + 1]
  uint16_t* scl = reinterpret_cast<uint16_t*>(keep_off + p.cap_pow2 / 64 + 1);              // [cap_pow2] class ids (class-aware mode)
  NmsGrid* const grid = p.grid_off ? reinterpret_cast<NmsGrid*>(smem_raw + p.grid_off) : nullptr;
  uint32_t* const over_mark = grid ? reinterpret_cast<uint32_t*>(grid + 1) : nullptr;       // [cap_pow2/32]
  uint16_t* const over = grid ? reinterpret_cast<uint16_t*>(over_mark + p.cap_pow2 / 32) : nullptr;  // [cap_pow2]
  __shared__ uint32_t rows[64][2];
  __shared__ float4 kbox[64];
  __shared__ int kcl[64];
  SmallNms& sm = *reinterpret_cast<SmallNms*>(smem_raw);  // (never touched here: `small` is false)
  const DetHandover* const hand = nullptr;
  const bool aware = p.class_aware != 0;
  const bool ultra = p.ultra != 0;
  const float thr = p.iou_thr;
  const bool thr_nonneg = ultra ? p.iou_thr64 >= 0.0 : thr >= 0.f;
  const int nchunks = (n + 63) >> 6;

  for (int i = tid; i < np2; i += NT) keys[i] = i < n ? p.cand_key[cbase + i] : 0ull;
  for (int i = tid; i < np2 / 32; i += NT) supp[i] = 0u;
  __syncthreads();

  PHASE_STAMP(p.dbg, 17);
  block_bitonic_sort_desc<NT>(keys, np2);
  PHASE_STAMP(p.dbg, 18);
  // gather boxes and class ids of the sorted candidates into shared memory in one round of global loads
  for (int i = tid; i < n; i += NT) {
    const size_t o = cbase + key_slot(keys[i]);
    float4 b = p.cand_box[o];
    const int cl = p.cand_cls[o];
    if (p.ultra && !p.ultra_agnostic) {  // boxes = x[:, :4] + x[:, 5:6] * max_wh, float32 (the rounding is part of the semantics)
      const float c = __fmul_rn((float)cl, 7680.f);
      b = make_float4(__fadd_rn(b.x, c), __fadd_rn(b.y, c), __fadd_rn(b.z, c), __fadd_rn(b.w, c));
    }
    box[i] = p.ultra ? b : nan_box_view(b);
    scl[i] = (uint16_t)cl;
  }
  __syncthreads();

  PHASE_STAMP(p.dbg, 19);
  // few candidates: the survivors-vs-tail scan is cheaper than keeping the grid
  // (the grid assumes finite coordinates: a NaN box suppresses, and is suppressed by, boxes anywhere in the frame)
  bool finite = true;
  if (GRID && grid != nullptr && !ultra && thr_nonneg && n > 256) {
    int bad = 0;
    for (int i = tid; i < n; i += NT) {
      const float4 b = box[i];
      bad |= !(fabsf(b.x) <= 3.0e38f && fabsf(b.y) <= 3.0e38f && fabsf(b.z) <= 3.0e38f && fabsf(b.w) <= 3.0e38f);
    }
    finite = !__syncthreads_or(bad);
  }
  const bool use_grid = GRID && grid != nullptr && !ultra && thr_nonneg && n > 256 && finite;
  const float inv_cw = (float)kGX / (p.f[frame].xmax + 1.0f), inv_ch = (float)kGY / (p.f[frame].ymax + 1.0f);
  if (GRID && use_grid) {
    for (int c = tid; c < kCells; c += NT) grid->cnt[c] = 0;
    for (int w = tid; w < (n + 31) / 32; w += NT) over_mark[w] = 0u;
    if (tid == 0) grid->n_over = 0;
    __syncthreads();
  }
#ifdef B200VA_PHASE_TIMING
  long long acc_a = 0, acc_b = 0, acc_c = 0, acc_q = 0, t_mark = clock64();
#define NMS_MARK(acc) do { const long long _t = clock64(); acc += _t - t_mark; t_mark = _t; } while (0)
#else
#define NMS_MARK(acc) do { } while (0)
#endif
  for (int ch = 0; ch < nchunks; ++ch) {
    const int c0 = ch << 6;
    const int m = min(64, n - c0);
    if (tid < 128) rows[tid >> 1][tid & 1] = 0u;
    __syncthreads();
    // (q) grid mode: is box i of this chunk suppressed by a box kept in an EARLIER chunk?  Eight threads per box
    // (the first sixteen warps) take the cells it touches.  Pass 1 only collects the kept boxes that overlap box i
    // (four compares each); pass 2 runs the IoU formula on them with the warp converged.  The CTA is issue-bound
    // in this loop (all 32 warps busy on one SM), so what counts is warp-instructions: ~1.3 k per query warp and
    // chunk, against ~4 k per chunk for the survivors-vs-tail scan it replaces in dense scenes.
    // (Writes supp[], which (a) does not read: no barrier before (a).)
    if (GRID && use_grid && ch > 0 && tid < 512) {
      // eight lanes per box: lane = (cell slot 0..3, entry half 0..1); a lane tests at most four entries per cell visit
      const int i = tid >> 3, part = tid & 3, half = (tid >> 2) & 1;
#ifdef B200VA_PHASE_TIMING
      long long q0 = clock64();
#endif
      const bool active = i < m;
      const int self = c0 + (active ? i : 0);
      const float4 bi = box[self];
      const int ci = scl[self];
      int cx0, cx1, cy0, cy1;
      cell_range(bi, inv_cw, inv_ch, cx0, cx1, cy0, cy1);
      const int cw = cx1 - cx0 + 1, ncell = active ? cw * (cy1 - cy0 + 1) : 0;
      const float rcw = 1.0f / (float)cw;
      constexpr int kQ = 4;  // overlapping kept boxes a lane can defer; more are evaluated on the spot
      unsigned long long cand = 0ull;  // up to four 16-bit indices, packed (an indexed array would live in local memory)
      int nc = 0;
      bool hit = false;
      auto consider = [&](int k) {
        const float4 bk = box[k];
        if (bk.z <= bi.x || bi.z <= bk.x || bk.w <= bi.y || bi.w <= bk.y) return;  // disjoint: IoU 0 <= thr
        if (aware && scl[k] != ci) return;
        if (nc < kQ) cand |= (unsigned long long)k << (16 * nc++);
        else if (suppresses(bk, bi, thr)) hit = true;
      };
#ifdef B200VA_PHASE_TIMING
      long long q1 = clock64();
#endif
#pragma unroll 1
      for (int c = part; c < ncell; c += 4) {
        const int row = (int)(((float)c + 0.5f) * rcw);  // c / cw for these small integers
        const int cell = (cy0 + row) * kGX + cx0 + (c - row * cw);
        const int cnt = min(grid->cnt[cell], kCellCap);
#pragma unroll 1  // unrolled, this loop alone was 1700 instructions of mostly predicated-off code
        for (int e = 4 * half; e < cnt; e += 8) {  // one 8-byte load brings four indices
          const uint2 kk = *reinterpret_cast<const uint2*>(&grid->list[cell][e]);
          const int k4[4] = {(int)(kk.x & 0xffffu), (int)(kk.x >> 16), (int)(kk.y & 0xffffu), (int)(kk.y >> 16)};
#pragma unroll
          for (int u = 0; u < 4; ++u)
            if (e + u < cnt) consider(k4[u]);
        }
      }
#ifdef B200VA_PHASE_TIMING
      long long q2 = clock64();
#endif
      if (active) {
        const int nover = grid->n_over;
#pragma unroll 1
        for (int e = (tid & 7); e < nover; e += 8) consider(over[e]);
      }
#ifdef B200VA_PHASE_TIMING
      long long q3 = clock64();
#endif
#pragma unroll
      for (int u = 0; u < kQ; ++u) {
        if (!__any_sync(0xffffffffu, u < nc && !hit)) break;
        if (u < nc && !hit && suppresses(box[(int)((cand >> (16 * u)) & 0xffffull)], bi, thr)) hit = true;
      }
      if (hit) atomicOr(&supp[self >> 5], 1u << (self & 31));
#ifdef B200VA_PHASE_TIMING
      if (blockIdx.x == 0 && tid == 0) {
        const long long q4 = clock64();
        p.dbg[32] += q1 - q0;
        p.dbg[33] += q2 - q1;
        p.dbg[34] += q3 - q2;
        p.dbg[35] += q4 - q3;
      }
#endif
    }
    NMS_MARK(acc_q);
    // (a) in-chunk IoU bits: thread -> row i = tid / 16, columns 4 * (tid % 16) ..; the predicate is
    // symmetric, so only pairs j > i are evaluated and a hit sets both (i, j) and (j, i)
    for (int task = tid; task < 1024; task += NT) {
      const int i = task >> 4, jb = (task & 15) << 2;
      if (i < m && jb + 3 > i) {
        const float4 bi = box[c0 + i];
#pragma unroll
        for (int q = 0; q < 4; ++q) {
          const int j = jb + q;
          if (j <= i || j >= m) continue;
          const float4 bj = box[c0 + j];
          if (thr_nonneg && (bj.z <= bi.x || bi.z <= bj.x || bj.w <= bi.y || bi.w <= bj.y)) continue;  // disjoint: IoU 0
          if ((!aware || scl[c0 + i] == scl[c0 + j]) && (ultra ? suppresses_tv(bi, bj, p.iou_thr64) : suppresses(bi, bj, thr))) {
            atomicOr(&rows[i][j >> 5], 1u << (j & 31));
            atomicOr(&rows[j][i >> 5], 1u << (i & 31));
          }
        }
      }
    }
    __syncthreads();
    NMS_MARK(acc_a);
    // (b) greedy resolution inside the chunk: kept_i = alive_i and no kept j < i suppresses i.  That
    // recursion has a unique solution; iterating it from kept = alive fixes box i after at most i
    // rounds, so one warp (two boxes per lane) repeats it until nothing changes -- a handful of
    // ballots for typical clusters instead of 64 dependent steps.
    if (tid < 32) {
      const unsigned long long lo_mask = (1ull << tid) - 1ull, hi_mask = (1ull << (tid + 32)) - 1ull;
      const unsigned long long e0 = (((unsigned long long)rows[tid][1] << 32) | rows[tid][0]) & lo_mask;
      const unsigned long long e1 = (((unsigned long long)rows[tid + 32][1] << 32) | rows[tid + 32][0]) & hi_mask;
      const unsigned long long valid = m == 64 ? ~0ull : ((1ull << m) - 1ull);
      const unsigned long long alive = ~(((unsigned long long)supp[(c0 >> 5) + 1] << 32) | supp[c0 >> 5]) & valid;
      const bool a0 = (alive >> tid) & 1ull, a1 = (alive >> (tid + 32)) & 1ull;
      bool k0 = a0, k1 = a1;
      unsigned long long kept;
      while (true) {
        kept = ((unsigned long long)__ballot_sync(0xffffffffu, k1) << 32) | __ballot_sync(0xffffffffu, k0);
        const bool n0 = a0 && !(e0 & kept), n1 = a1 && !(e1 & kept);
        const unsigned changed = __ballot_sync(0xffffffffu, n0 != k0 || n1 != k1);
        k0 = n0;
        k1 = n1;
        if (!changed) break;
      }
      if (tid == 0) {
        keep_w[2 * ch] = (uint32_t)kept;
        keep_w[2 * ch + 1] = (uint32_t)(kept >> 32);
      }
    }
    __syncthreads();
    NMS_MARK(acc_b);
    // (c) this chunk's survivors suppress every later box.  The survivors are first packed into a
    // dense list; g threads share one later box (each takes a slice of the list), g shrinking as the
    // tail grows so that all 1024 threads stay busy.
    const unsigned long long kept = ((unsigned long long)keep_w[2 * ch + 1] << 32) | keep_w[2 * ch];
    const int tail = n - (c0 + 64);
    if (GRID && use_grid) {
      // (c') register this chunk's survivors in the cells they touch (16 threads per survivor)
      const int b = tid >> 4, part = tid & 15;
      if (tail > 0 && ((kept >> b) & 1ull)) {
        const int idx = c0 + b;
        int cx0, cx1, cy0, cy1;
        cell_range(box[idx], inv_cw, inv_ch, cx0, cx1, cy0, cy1);
        const int cw = cx1 - cx0 + 1, ncell = cw * (cy1 - cy0 + 1);
        bool spill = ncell > kMaxCellsPerBox && part == 0;
        if (ncell <= kMaxCellsPerBox) {
          const float rcw = 1.0f / (float)cw;
          for (int c = part; c < ncell; c += 16) {
            const int row = (int)(((float)c + 0.5f) * rcw);
            const int cell = (cy0 + row) * kGX + cx0 + (c - row * cw);
            const int pos = atomicAdd(&grid->cnt[cell], 1);
            if (pos < kCellCap) grid->list[cell][pos] = (uint16_t)idx;
            else spill = true;
          }
        }
        // a box that does not fit its cells goes to the overflow list, once
        if (spill && !(atomicOr(&over_mark[idx >> 5], 1u << (idx & 31)) & (1u << (idx & 31))))
          over[atomicAdd(&grid->n_over, 1)] = (uint16_t)idx;
      }
    } else if (kept && tail > 0) {
      const int nk = __popcll(kept);
      if (tid < 64 && ((kept >> tid) & 1ull)) {
        const int q = __popcll(kept & ((1ull << tid) - 1ull));
        kbox[q] = box[c0 + tid];
        kcl[q] = scl[c0 + tid];
      }
      __syncthreads();
      int g = 16;
      while (g > 1 && tail * g > NT) g >>= 1;
      const int part = tid & (g - 1);
      const int per = (nk + g - 1) / g;
      const int qb = part * per, qe = min(nk, qb + per);
      if (qb < qe) {
        for (int j = c0 + 64 + tid / g; j < n; j += NT / g) {
          if ((supp[j >> 5] >> (j & 31)) & 1u) continue;
          const float4 bj = box[j];
          const int cj = scl[j];
          // pass 1 (uniform across the warp): which survivors can touch box j at all.  Disjoint boxes have
          // intersection exactly 0 -> IoU 0 -> kept whenever thr >= 0 (four compares instead of the full formula;
          // NaN coordinates fail every compare and stay candidates).  Pass 2 runs the full formula only on those
          // -- a handful per box -- so a warp no longer drags all 32 lanes through the division each time ONE lane
          // meets its overlapping survivor (dense config: this phase 172 k -> 129 k SM cycles, post-process 183 -> 161 us).
          unsigned long long cand = 0ull;
          for (int q = qb; q < qe; ++q) {
            const float4 bi = kbox[q];
            const bool apart = thr_nonneg && (bj.z <= bi.x || bi.z <= bj.x || bj.w <= bi.y || bi.w <= bj.y);
            const bool same = !aware || kcl[q] == cj;
            cand |= (unsigned long long)(!apart && same) << (q - qb);
          }
          while (cand) {
            const int q = qb + __ffsll((long long)cand) - 1;
            cand &= cand - 1ull;
            if (ultra ? suppresses_tv(kbox[q], bj, p.iou_thr64) : suppresses(kbox[q], bj, thr)) {
              atomicOr(&supp[j >> 5], 1u << (j & 31));
              break;
            }
          }
        }
      }
    }
    __syncthreads();
    NMS_MARK(acc_c);
  }
#ifdef B200VA_PHASE_TIMING
  if (blockIdx.x == 0 && tid == 0) {
    p.dbg[24] = acc_a;
    p.dbg[25] = acc_b;
    p.dbg[26] = acc_c;
    p.dbg[27] = acc_q;
    if (use_grid) {
      int mx = 0, tot = 0;
      for (int c = 0; c < kCells; ++c) {
        mx = max(mx, grid->cnt[c]);
        tot += grid->cnt[c];
      }
      p.dbg[28] = mx;
      p.dbg[29] = grid->n_over;
      p.dbg[30] = tot;
    }
  }
#endif
  PHASE_STAMP(p.dbg, 20);
  // ultralytics: `i = i[:max_det]` on the NMS survivors, before anything else looks at them
  if (ultra) {
    if (tid == 0) {
      int acc = 0;
      for (int ch = 0; ch < nchunks; ++ch) {
        for (int w = 0; w < 2; ++w) {
          uint32_t bits = keep_w[2 * ch + w];
          const int room = p.max_det_cap - acc;
          if (room <= 0) {
            bits = 0u;
          } else if (__popc(bits) > room) {
            uint32_t kept_bits = 0u;
            for (int r = 0; r < room; ++r) {  // keep the `room` lowest set bits
              const uint32_t low = bits & (0u - bits);
              kept_bits |= low;
              bits ^= low;
            }
            bits = kept_bits;
          }
          keep_w[2 * ch + w] = bits;
          acc += __popc(bits);
        }
      }
    }
    __syncthreads();
  }
  // filter_detections (detector.py:99-103): float64 compare on the kept boxes only
  if (p.use_filter) {
    for (int i = tid; i < n; i += NT) {
      if ((keep_w[i >> 5] >> (i & 31)) & 1u) {
        const float conf = key_conf(keys[i]);
        if (!((double)conf >= p.filter_thr)) atomicAnd(&keep_w[i >> 5], ~(1u << (i & 31)));
      }
    }
    __syncthreads();
  }
  PHASE_STAMP(p.dbg, 54);
  if (tid == 0) {
    int acc = 0;
    for (int ch = 0; ch < nchunks; ++ch) {
      keep_off[ch] = acc;
      acc += __popc(keep_w[2 * ch]) + __popc(keep_w[2 * ch + 1]);
    }
    keep_off[nchunks] = acc;
    p.out_count[frame] = min(acc, p.max_dets);
    if (acc > p.max_dets) atomicOr(p.flags + FLAG_DET_OVERFLOW, 1);
  }
  PHASE_STAMP(p.dbg, 55);
  __syncthreads();
  PHASE_STAMP(p.dbg, 56);
  for (int i = tid; i < n; i += NT) {
    const unsigned long long w = ((unsigned long long)keep_w[2 * (i >> 6) + 1] << 32) | keep_w[2 * (i >> 6)];
    if ((w >> (i & 63)) & 1ull) {
      const int pos = keep_off[i >> 6] + __popcll(w & ((1ull << (i & 63)) - 1ull));
      if (pos < p.max_dets) {
        const size_t o = (size_t)frame * p.max_dets + pos;
        float4 b = box[i];
        const int slot = key_slot(keys[i]);
        if (ultra) b = ultra_scale_box(small ? sm.ubox[slot] : p.cand_box[cbase + slot], p.f[frame]);  // the un-shifted box
        else if (b.x != b.x) b = small ? sm.ubox[slot] : p.cand_box[cbase + slot];  // (nan_box_view: emit the box as decoded)
        const float cf = key_conf(keys[i]);
        const int cl = small ? sm.ucls[slot] : p.cand_cls[cbase + slot];  // the full int32 class id (scl[] holds 16 bits)
        reinterpret_cast<float4*>(p.out_box)[o] = b;
        p.out_conf[o] = cf;
        p.out_cls[o] = cl;
        if (hand && small && pos < kDetChunk) stage_detection(hand->sh->sd, pos, b, cf, cl, hand->scale, hand->has_scale != 0);
      }
    }
  }
  PHASE_STAMP(p.dbg, 21);
}

// The part of the small-frame set-up that does not depend on the frame: cleared matrix, bitmap and pair counter.
template <int NT>
__device__ __forceinline__ void nms_small_init(uint8_t* const smem_raw) {
  SmallNms& sm = *reinterpret_cast<SmallNms*>(smem_raw);
  for (int w = threadIdx.x; w < kSmallN * (kSmallN / 32); w += NT) (&sm.M[0][0])[w] = 0u;
  if (threadIdx.x < kSmallN / 32) sm.supp[threadIdx.x] = 0u;
  if (threadIdx.x == 0) sm.n_pairs = 0;
}

template <bool GRID, int NT>
__device__ __noinline__ void nms_general(const NmsParams& p, const int frame, uint8_t* const smem_raw, const int n) {
  nms_general_body<GRID, NT>(p, frame, smem_raw, n);
}

// COLD_GENERAL: the general path sits behind a call (the fused sparse-scene kernel); otherwise it is inlined (the
// kernels the host picks for dense scenes, where that path is the one that runs).
// ULTRA_OK = false: the caller guarantees reference semantics (p.ultra == 0) and the Ultralytics variants of the
// predicate, the class shift and the un-letterbox step are compiled out of the small-frame path.
template <bool GRID, int NT, bool COLD_GENERAL, bool ULTRA_OK>
__device__ __forceinline__ void nms_frame(const NmsParams& p, const int frame, uint8_t* const smem_raw,
                                          const DetHandover* hand = nullptr, const bool pre_init = false) {
  static_assert(!GRID || NT == 1024, "the kept-box grid code assumes 1024 threads");
  static_assert(NT >= kSmallN && NT % 32 == 0, "bad CTA width");
  const int tid = threadIdx.x;
  PHASE_STAMP(p.dbg, 16);
  const size_t cbase = (size_t)frame * p.max_cand;
  // speculative: the first kSmallN candidate slots, fetched in the same round trip as the count (slots past the count
  // hold stale rows of earlier frames; they are masked below)
  unsigned long long k_spec = 0ull;
  float4 b_spec = make_float4(0.f, 0.f, 0.f, 0.f);
  int c_spec = 0;
  if (tid < kSmallN && tid < p.max_cand) {
    k_spec = p.cand_key[cbase + tid];
    b_spec = p.cand_box[cbase + tid];
    c_spec = p.cand_cls[cbase + tid];
  }
  const int n_raw = (p.skip && p.skip[frame]) ? 0 : p.cand_count[frame];  // a gated frame was not decoded either
  const int n = min(n_raw, p.max_cand);
  const bool small = n <= kSmallN;
  SmallNms& sm = *reinterpret_cast<SmallNms*>(smem_raw);


  __syncthreads();
  if (tid == 0) {
    if (p.stats && n > 256) *(volatile int*)p.stats = n;  // posted write, dense frames only (an atomic to host memory cost 25 us)
    p.cand_count[frame] = 0;
    if (n_raw > p.max_cand) atomicOr(p.flags + FLAG_CAND_OVERFLOW, 1);
    if (hand) hand->sh->s_prestaged = n == 0 ? 0 : -1;
  }
  PHASE_STAMP(p.dbg, 50);
  if (n == 0) {
    if (tid == 0) p.out_count[frame] = 0;
    return;
  }
  const bool aware = p.class_aware != 0;
  const bool ultra = ULTRA_OK && p.ultra != 0;
  const float thr = p.iou_thr;
  const bool thr_nonneg = ultra ? p.iou_thr64 >= 0.0 : thr >= 0.f;
  const int nchunks = (n + 63) >> 6;
  if (!small) {
    if (COLD_GENERAL) nms_general<GRID, NT>(p, frame, smem_raw, n);
    else nms_general_body<GRID, NT>(p, frame, smem_raw, n);
    return;
  }
  unsigned long long* const keys = sm.keys;
  float4* const box = sm.box;
  uint32_t* const keep_w = sm.keep_w;
  int* const keep_off = sm.keep_off;
  {
    // ---- small frame: one load round, rank sort, full bit matrix, one-warp resolution ----
    const int words = (n + 31) >> 5;
    if (tid < kSmallN) {
      sm.keys[tid] = tid < n ? k_spec : 0ull;
      sm.ubox[tid] = b_spec;
      sm.ucls[tid] = c_spec;
    }
    if (!pre_init) {  // (the fused kernel did this while it waited for the decode kernel)
      for (int w = tid; w < n * (kSmallN / 32); w += NT) (&sm.M[0][0])[w] = 0u;
      if (tid < kSmallN / 32) sm.supp[tid] = 0u;
      if (tid == 0) sm.n_pairs = 0;
    }
    __syncthreads();
    PHASE_STAMP(p.dbg, 17);
    if (tid < n) {  // rank sort: keys are unique, rank = number of larger keys
      const unsigned long long ki = sm.keys[tid];
      int r0 = 0, r1 = 0, r2 = 0, r3 = 0;
      int j = 0;
      for (; j + 4 <= n; j += 4) {
        r0 += sm.keys[j] > ki;
        r1 += sm.keys[j + 1] > ki;
        r2 += sm.keys[j + 2] > ki;
        r3 += sm.keys[j + 3] > ki;
      }
      for (; j < n; ++j) r0 += sm.keys[j] > ki;
      sm.sorted[r0 + r1 + r2 + r3] = ki;
    }
    __syncthreads();
    PHASE_STAMP(p.dbg, 18);
    if (tid < n) {
      const unsigned long long k = sm.sorted[tid];
      const int slot = key_slot(k);
      float4 b = sm.ubox[slot];
      const int cl = sm.ucls[slot];
      if (ultra && !p.ultra_agnostic) {  // boxes = x[:, :4] + x[:, 5:6] * max_wh, float32 (the rounding is part of the semantics)
        const float c = __fmul_rn((float)cl, 7680.f);
        b = make_float4(__fadd_rn(b.x, c), __fadd_rn(b.y, c), __fadd_rn(b.z, c), __fadd_rn(b.w, c));
      }
      sm.keys[tid] = k;
      sm.box[tid] = ultra ? b : nan_box_view(b);
      sm.scl[tid] = (uint16_t)cl;
    }
    __syncthreads();
    PHASE_STAMP(p.dbg, 19);
    // The CTA is latency-bound: what a phase costs is the instruction count of its longest warp times ~4.5 cycles, and
    // a warp in which ONE lane meets an overlapping pair walks all 32 lanes through the IoU formula.  So: pass 1 only
    // sorts the pairs i < j into "disjoint" (nothing to do: IoU 0 <= thr) and "candidate" (appended to a list), with
    // every pair visited once and the rows spread evenly -- thread (part, i) takes the pairs {i, i + k mod n} for
    // k = 1 + part, 1 + part + parts, .. <= n / 2 -- and pass 2 runs the formula on one listed pair per thread, all
    // lanes converged.  (72 candidates: 7.0 k -> ~1.2 k SM cycles for this phase.)
    {
      const int part = (int)(((float)tid + 0.5f) * (1.0f / (float)n));  // tid / n for these small integers
      const int i = tid - part * n;
      const int parts = NT / n, half = n >> 1;
      const float4 bi = sm.box[i];
      const int ci = sm.scl[i];
      // which of this thread's pairs are candidates: bit `it` of (c_lo, c_hi) <-> k = 1 + part + it * parts
      // (at most 128 iterations: n <= 256, parts >= 1)
      unsigned long long c_lo = 0ull, c_hi = 0ull;
      if (part < parts) {
        const bool even = !(n & 1);
#pragma unroll 1
        for (int hw = 0; hw < 2; ++hw) {
          unsigned long long mm = 0ull;
          const int kb = 1 + part + hw * 64 * parts;
          // branch-free body, unrolled once: two iterations' loads in flight (code size matters more than latency here)
#pragma unroll 2
          for (int b = 0; b < 64; ++b) {
            const int k = kb + b * parts;
            if (k > half) break;
            int j = i + k;
            j -= j >= n ? n : 0;
            const float4 bj = sm.box[j];
            bool c = !(thr_nonneg && (bj.z <= bi.x || bi.z <= bj.x || bj.w <= bi.y || bi.w <= bj.y));  // disjoint: IoU 0
            if (aware) c = c && ci == sm.scl[j];
            c = c && !(even && k == half && i >= half);  // even n: the antipodal pairs come up twice
            mm |= (unsigned long long)c << b;
          }
          if (hw == 0) c_lo = mm;
          else c_hi = mm;
          if (kb + 64 * parts > half) break;
        }
      }
      // one list reservation per warp: exclusive prefix of the lanes' counts, lane 31 draws the block
      const int mine = __popcll(c_lo) + __popcll(c_hi);
      int incl = mine;
#pragma unroll
      for (int o = 1; o < 32; o <<= 1) {
        const int v = __shfl_up_sync(0xffffffffu, incl, o);
        if ((tid & 31) >= o) incl += v;
      }
      int base = 0;
      if ((tid & 31) == 31 && incl > 0) base = atomicAdd(&sm.n_pairs, incl);
      base = __shfl_sync(0xffffffffu, base, 31);
      int slot = base + incl - mine;
#pragma unroll 1
      for (int half_w = 0; half_w < 2; ++half_w) {
        unsigned long long bits = half_w ? c_hi : c_lo;
        while (bits) {
          const int it = __ffsll((long long)bits) - 1 + 64 * half_w;
          bits &= bits - 1ull;
          int j = i + 1 + part + it * parts;
          if (j >= n) j -= n;
          const int lo = min(i, j), hi = max(i, j);
          if (slot < kSmallPairs) sm.pairs[slot] = (uint32_t)lo | ((uint32_t)hi << 16);
          ++slot;
        }
      }
    }
    PHASE_STAMP(p.dbg, 51);
    __syncthreads();
    PHASE_STAMP(p.dbg, 52);
    {
      const int listed = sm.n_pairs;
      if (listed > kSmallPairs) {
        // more overlapping pairs than the list holds (one dense cluster): the chunked general path takes the frame
        // from its candidate arrays, which are untouched
        if (COLD_GENERAL) nms_general<GRID, NT>(p, frame, smem_raw, n);
        else nms_general_body<GRID, NT>(p, frame, smem_raw, n);
        return;
      }
#pragma unroll 1
      for (int q = tid; q < listed; q += NT) {
        const uint32_t pr = sm.pairs[q];
        const int lo = (int)(pr & 0xffffu), hi = (int)(pr >> 16);
        if (ultra ? suppresses_tv(sm.box[lo], sm.box[hi], p.iou_thr64) : suppresses(sm.box[lo], sm.box[hi], thr)) {
          atomicOr(&sm.M[lo][hi >> 5], 1u << (hi & 31));
          atomicOr(&sm.M[hi][lo >> 5], 1u << (lo & 31));
        }
      }
    }
    __syncthreads();
    PHASE_STAMP(p.dbg, 57);
    if (tid < 32) {
      // greedy resolution, chunk by chunk: kept_i = alive_i and no kept j < i of the chunk suppresses i (fixed point
      // of ballots, see the general path); a chunk's kept rows then mark the later chunks' boxes.  The same warp
      // then derives what is EMITTED from what is kept -- Ultralytics' `i[:max_det]`, then filter_detections
      // (detector.py:99-103, float64 compare) -- and the output offsets, so no further block-wide phase is needed.
      int acc_kept = 0, acc_emit = 0;
#pragma unroll 1
      for (int ch = 0; ch < nchunks; ++ch) {
        const int c0 = ch << 6, m = min(64, n - c0);
        const unsigned long long lo_mask = (1ull << tid) - 1ull, hi_mask = (1ull << (tid + 32)) - 1ull;
        const int r0 = min(c0 + tid, kSmallN - 1), r1 = min(c0 + tid + 32, kSmallN - 1);
        const unsigned long long e0 = (((unsigned long long)sm.M[r0][2 * ch + 1] << 32) | sm.M[r0][2 * ch]) & lo_mask;
        const unsigned long long e1 = (((unsigned long long)sm.M[r1][2 * ch + 1] << 32) | sm.M[r1][2 * ch]) & hi_mask;
        const unsigned long long valid = m == 64 ? ~0ull : ((1ull << m) - 1ull);
        const unsigned long long alive = ~(((unsigned long long)sm.supp[2 * ch + 1] << 32) | sm.supp[2 * ch]) & valid;
        const bool a0 = (alive >> tid) & 1ull, a1 = (alive >> (tid + 32)) & 1ull;
        bool k0 = a0, k1 = a1;
        unsigned long long kept;
        while (true) {
          kept = ((unsigned long long)__ballot_sync(0xffffffffu, k1) << 32) | __ballot_sync(0xffffffffu, k0);
          const bool n0 = a0 && !(e0 & kept), n1 = a1 && !(e1 & kept);
          const unsigned changed = __ballot_sync(0xffffffffu, n0 != k0 || n1 != k1);
          k0 = n0;
          k1 = n1;
          if (!changed) break;
        }
#pragma unroll 1
        for (int w = 2 * ch + 2; w < words; ++w) {
          uint32_t v = (k0 ? sm.M[r0][w] : 0u) | (k1 ? sm.M[r1][w] : 0u);
          v = __reduce_or_sync(0xffffffffu, v);
          if (tid == 0) sm.supp[w] |= v;
        }
        bool m0 = k0, m1 = k1;
        if (ultra) {  // `i = i[:max_det]`: the first max_det_cap survivors, in score order
          m0 = m0 && acc_kept + __popcll(kept & lo_mask) < p.max_det_cap;
          m1 = m1 && acc_kept + __popcll(kept & hi_mask) < p.max_det_cap;
          acc_kept += __popcll(kept);
        }
        if (p.use_filter) {
          m0 = m0 && (double)key_conf(sm.keys[r0]) >= p.filter_thr;
          m1 = m1 && (double)key_conf(sm.keys[r1]) >= p.filter_thr;
        }
        const uint32_t w0 = __ballot_sync(0xffffffffu, m0), w1 = __ballot_sync(0xffffffffu, m1);
        if (tid == 0) {
          sm.keep_w[2 * ch] = w0;
          sm.keep_w[2 * ch + 1] = w1;
          sm.keep_off[ch] = acc_emit;
        }
        acc_emit += __popc(w0) + __popc(w1);
        __syncwarp();
      }
      if (tid == 0) {
        sm.keep_off[nchunks] = acc_emit;
        p.out_count[frame] = min(acc_emit, p.max_dets);
        if (acc_emit > p.max_dets) atomicOr(p.flags + FLAG_DET_OVERFLOW, 1);
        if (hand) hand->sh->s_prestaged = min(acc_emit, p.max_dets);  // the emit loop stages the first chunk
      }
    }
    PHASE_STAMP(p.dbg, 53);  // (the barrier before the emit loop below closes this phase)
  }
  PHASE_STAMP(p.dbg, 55);
  __syncthreads();
  PHASE_STAMP(p.dbg, 56);
  for (int i = tid; i < n; i += NT) {
    const unsigned long long w = ((unsigned long long)keep_w[2 * (i >> 6) + 1] << 32) | keep_w[2 * (i >> 6)];
    if ((w >> (i & 63)) & 1ull) {
      const int pos = keep_off[i >> 6] + __popcll(w & ((1ull << (i & 63)) - 1ull));
      if (pos < p.max_dets) {
        const size_t o = (size_t)frame * p.max_dets + pos;
        float4 b = box[i];
        const int slot = key_slot(keys[i]);
        if (ultra) b = ultra_scale_box(small ? sm.ubox[slot] : p.cand_box[cbase + slot], p.f[frame]);  // the un-shifted box
        else if (b.x != b.x) b = small ? sm.ubox[slot] : p.cand_box[cbase + slot];  // (nan_box_view: emit the box as decoded)
        const float cf = key_conf(keys[i]);
        const int cl = small ? sm.ucls[slot] : p.cand_cls[cbase + slot];  // the full int32 class id (scl[] holds 16 bits)
        reinterpret_cast<float4*>(p.out_box)[o] = b;
        p.out_conf[o] = cf;
        p.out_cls[o] = cl;
        if (hand && small && pos < kDetChunk) stage_detection(hand->sh->sd, pos, b, cf, cl, hand->scale, hand->has_scale != 0);
      }
    }
  }
  PHASE_STAMP(p.dbg, 21);
}

template <bool GRID>
__global__ void __launch_bounds__(kNmsThreads) k_sort_nms(const __grid_constant__ NmsParams p) {
  extern __shared__ __align__(16) uint8_t smem_raw[];
  griddep_launch_dependents();  // a tracker kernel behind this one may be scheduled; its griddep_wait() waits for this grid
  griddep_wait();
#ifdef B200VA_PHASE_TIMING
  // developer experiment (B200VA_DBG_REPS=n): run the frame n times in one launch; the stamps of the LAST pass show what
  // the same code costs once its instructions and data are warm in the SM
  for (int r = 1; r < p.dbg_reps; ++r) {
    const int saved = p.cand_count[blockIdx.x];
    __syncthreads();
    nms_frame<GRID, kNmsThreads, false, true>(p, blockIdx.x, smem_raw);
    __syncthreads();
    if (threadIdx.x == 0) p.cand_count[blockIdx.x] = saved;
    __syncthreads();
  }
#endif
  nms_frame<GRID, kNmsThreads, false, true>(p, blockIdx.x, smem_raw);
}

// Sparse scenes: sort + NMS + emit of frame i followed by the tracker update of stream i in ONE CTA of 256 threads.
// The detections never leave the SM's caches between the two halves, one launch and one kernel-to-kernel dependency
// disappear from the critical chain decode -> NMS -> tracker (what a tick of a few streams per GPU is made of), and
// 256-thread barriers replace 1024-thread ones.  Any candidate count is handled correctly (just more slowly than by
// the 1024-thread grid variant), so the host's choice between the two never changes a result.
template <bool ULTRA>
__global__ void __launch_bounds__(kNmsThreadsSmall) k_post_track(const __grid_constant__ NmsParams q,
                                                                  const __grid_constant__ TrkParams t) {
  extern __shared__ __align__(16) uint8_t smem_raw[];
  __shared__ TrkShared sh;
  // ---- before the decode kernel is done (this grid is its programmatic dependent): everything that does not read
  // its candidates.  The stream's live tracks go into a working table BEHIND the small-frame NMS layout, so the
  // tracker half finds them in shared memory (the general NMS path uses the whole buffer and voids that copy).
  const int trk_slot = t.slots[blockIdx.x];
  const int pre_cur = t.st.cur[trk_slot], pre_T0 = t.st.count[trk_slot];
  constexpr int kTabOff = (int)((sizeof(SmallNms) + 127) & ~(size_t)127);
  unsigned dyn_bytes;
  asm("mov.u32 %0, %%dynamic_smem_size;" : "=r"(dyn_bytes));
  const int staged_cap = (((int)dyn_bytes - kTabOff - kDetChunk * 4 - 32) / kTrkRowBytes) & ~7;  // rows (see tracker_smem_bytes)
  const bool stage_early = pre_T0 <= staged_cap - kDetChunk && pre_T0 <= kNmsThreadsSmall;
  TablePrefetch pf{0, 0, 0.0};
  if (stage_early) pf = stage_table(t, trk_slot, pre_cur, pre_T0, smem_raw + kTabOff, staged_cap, kNmsThreadsSmall);
  nms_small_init<kNmsThreadsSmall>(smem_raw);
  griddep_wait();
  TIMELINE_BEGIN(q.dbg, 44);
  const DetHandover hand{&sh, t.det_scale[blockIdx.x], t.has_scale};
  // the handover stages float32 detections; a skipped stream (host flag or device mask) takes none
  nms_frame<false, kNmsThreadsSmall, true, ULTRA>(q, blockIdx.x, smem_raw, t.f_box ? &hand : nullptr, true);
  __syncthreads();  // this frame's detections were written by this CTA: visible to all of its threads from here on
  TIMELINE_END(q.dbg, 44);
  TIMELINE_BEGIN(q.dbg, 46);
  const int prestaged = t.f_box ? sh.s_prestaged : -1;
  // (s_prestaged >= 0 also says that the small-frame NMS ran, i.e. the early copy of the table is intact)
  const bool table_ok = stage_early && prestaged >= 0;
  tracker_stream<true>(t, blockIdx.x, smem_raw, sh, prestaged, pre_cur, pre_T0, table_ok ? &pf : nullptr, smem_raw + kTabOff,
                       staged_cap);
  TIMELINE_END(q.dbg, 46);  // (threads the tracker retires early never get here; thread 0 always does)
}


// ---- dense scenes: NMS off "one CTA on one SM" -------------------------------------------------------------------
// k_sort_nms keeps a whole frame in one CTA; with ~1800 candidates it is issue-bound on ONE SM per frame (32 of 148 SMs
// busy, 113-130 us).  Greedy NMS is the unique solution of  kept_i = no kept j ahead of i (in score order) suppresses i,
// and that recurrence needs neither a sorted array nor a sequential sweep:
//   k_dense_pairs    every SM: the suppression predicate of ALL unordered pairs of a frame's candidates, in the order
//                    decode left them (slot order, no sort).  A work item is 128 rows x 32 columns of the upper
//                    triangle, handed to single warps (the first by warp number, the rest through an atomic counter
//                    fetched one item ahead); a thread owns four rows (a 16-byte column broadcast from shared memory
//                    costs four cycles of its pipe however many lanes want the same address, so it has to feed four
//                    tests); "the boxes overlap at all" is the sign of four differences, branch-free; the overlapping
//                    pairs of a warp (0.4 % of all in config 5) are queued in shared memory and the IoU formula then
//                    runs over the queue with every lane busy.  A hit appends the box with the larger key (the one
//                    greedy NMS meets first) to the suppressor list of the other one; hits are collected across items and
//                    recorded 128 at a time (their key loads and atomics are dependent round trips to L2).  Measured and
//                    dropped: 64- and 128-column items, two rows per thread, 10 / 12 CTAs per SM at 48 / 40 registers,
//                    rows and columns of the next item prefetched with cp.async into a second buffer (7 CTAs per SM).
//   k_dense_resolve  one CTA per frame: Jacobi iteration of the recurrence over the suppressor lists (a box of
//                    dependency depth d is final after d + 1 rounds; clusters of near-duplicates have depth 1-2), then
//                    only the KEPT boxes (~300 of 1800) are ordered by key -- rank among the kept = output position.
// A frame with a full suppressor list (more than kNbrCap boxes ahead of one candidate suppress it) or a dependency chain
// longer than kResolveRounds falls back to the single-CTA path inside k_dense_resolve (same results, slower).
// k_dense_resolve_track: the same resolution followed by the stream's tracker update in the same CTA (b200va_tick).
// Results are those of the single-kernel path bit for bit: same predicate (IEEE add / mul / min / max commute, so the
// predicate is symmetric in its two boxes), same greedy recurrence, same tie rule (the keys are unique).
struct DenseNms {
  int32_t* nbr_cnt;  // [frames][max_cand] suppressors found for a candidate; all zero between launches
  uint16_t* nbr;     // [frames][max_cand][kNbrCap] slots of the suppressors, in no particular order
  int32_t* work;     // next work item of k_dense_pairs; zero between launches (k_dense_resolve clears it)
  int max_cand;
  int ctas;          // grid of k_dense_pairs
};
constexpr int kDenseCandMax = 4096;   // candidates per frame the dense path is built for (k_dense_resolve: 4 rows per thread)
constexpr int kNbrCap = 32;
constexpr int kPairWarps = 4, kPairThreads = 32 * kPairWarps;  // the warps of a CTA work on their own items
constexpr int kPairGroups = 4;                               // a thread owns kPairGroups rows (32 apart)
constexpr int kPairRows = 32 * kPairGroups;                  // rows of a work item (one warp)
#ifndef B200VA_PAIR_COLS
#define B200VA_PAIR_COLS 32
#endif
constexpr int kPairCols = B200VA_PAIR_COLS;                  // columns of a work item (32, 64 or 128; 32 measured best: the
                                                             // kernel ends when the last item does, so items are kept short)
constexpr int kPairRC = kPairRows / kPairCols;               // column tiles per row tile
constexpr int kPairColBits = kPairCols == 32 ? 5 : (kPairCols == 64 ? 6 : 7);
constexpr int kPairQueue = 256;                              // overlapping pairs a warp queues per 32 columns
constexpr int kPairHits = 128;                               // suppressing pairs a warp collects before it records them
constexpr int kResolveThreads = 1024, kResolveRows = kDenseCandMax / kResolveThreads;
constexpr int kResolveRounds = 64;
constexpr int kRankMax = 512;         // more kept boxes than this are ordered by the bitonic sort instead of by rank

// Ultralytics' class-aware trick: boxes = x[:, :4] + x[:, 5:6] * max_wh in float32 (the rounding is part of the semantics)
__device__ __forceinline__ float4 nms_view_of_box(const NmsParams& p, float4 b, int cl) {
  if (!p.ultra) return nan_box_view(b);
  if (!p.ultra_agnostic) {
    const float c = __fmul_rn((float)cl, 7680.f);
    b = make_float4(__fadd_rn(b.x, c), __fadd_rn(b.y, c), __fadd_rn(b.z, c), __fadd_rn(b.w, c));
  }
  return b;
}

// Work items of a frame with n candidates: row tile r (kPairRows rows) x column tile c (kPairCols columns) with
// c >= kPairRC r (the upper triangle, diagonal tiles included).
__device__ __forceinline__ int dense_items_of(int n) {
  const int R = (n + kPairRows - 1) / kPairRows, Cn = (n + kPairCols - 1) / kPairCols;
  return n > 1 ? R * Cn - kPairRC * (R * (R - 1) / 2) : 0;
}
static_assert(kDenseCandMax <= 4096 && B200VA_LAUNCH_FRAMES <= 256, "a hit is packed into 32 bits");
static_assert(kPairRows == kPairRC * kPairCols && (kPairCols == 32 || kPairCols == 64 || kPairCols == 128), "bad work item shape");

struct PairWarp {  // a warp's staging area
  float4 row[kPairRows];
  float4 col[kPairCols];
  int rcl[kPairRows];
  int ccl[kPairCols];
  uint16_t queue[kPairQueue];
  uint32_t hits[kPairHits];  // frame << 24 | row << 12 | column (candidate slots)
};

__global__ void __launch_bounds__(kPairThreads, 8) k_dense_pairs(const __grid_constant__ NmsParams p, const DenseNms D, const int frames) {
  __shared__ PairWarp s_warp[kPairWarps];
  __shared__ int s_first[B200VA_LAUNCH_FRAMES + 1];  // first work item of each frame
  __shared__ int s_n[B200VA_LAUNCH_FRAMES];
  griddep_launch_dependents();
  griddep_wait();
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  // Every warp starts on the item of its own number; the rest are handed out through an atomic counter (diagonal tiles
  // are cheaper than the others), fetched one item ahead.
  const int n_warps = (int)gridDim.x * kPairWarps;
  int item = (int)blockIdx.x * kPairWarps + warp, next = 0;
  if (tid < 32) {
    int v[2];
#pragma unroll
    for (int h = 0; h < 2; ++h) {
      const int f = lane + 32 * h;
      int n = 0;
      if (f < frames && !(p.skip && p.skip[f])) n = min(p.cand_count[f], p.max_cand);
      s_n[f] = n;
      v[h] = dense_items_of(n);
    }
    int base = 0;
#pragma unroll
    for (int h = 0; h < 2; ++h) {
      int incl = v[h];
#pragma unroll
      for (int o = 1; o < 32; o <<= 1) {
        const int t = __shfl_up_sync(0xffffffffu, incl, o);
        if (lane >= o) incl += t;
      }
      s_first[1 + lane + 32 * h] = base + incl;
      base += __shfl_sync(0xffffffffu, incl, 31);
    }
    if (lane == 0) s_first[0] = 0;
  }
  __syncthreads();  // (the only block-wide barrier: from here on every warp is on its own)
  static_assert(B200VA_LAUNCH_FRAMES == 64, "the item scan covers two frames per lane");
  const int total = s_first[B200VA_LAUNCH_FRAMES];
  const bool aware = p.class_aware != 0, ultra = p.ultra != 0;
  const float thr = p.iou_thr;
  const bool thr_nonneg = ultra ? p.iou_thr64 >= 0.0 : thr >= 0.f;
  PairWarp& S = s_warp[warp];
  // a suppressing pair: the box greedy NMS meets first (the larger key) goes on the suppressor list of the other one
  auto record = [&](const uint32_t hit) {
    const int frame = (int)(hit >> 24), i = (int)((hit >> 12) & 0xfffu), j = (int)(hit & 0xfffu);
    const size_t cbase = (size_t)frame * p.max_cand;
    const bool i_first = p.cand_key[cbase + i] > p.cand_key[cbase + j];
    const int loser = i_first ? j : i, winner = i_first ? i : j;
    const size_t row = (size_t)frame * D.max_cand + loser;
    const int slot = atomicAdd(D.nbr_cnt + row, 1);
    if (slot < kNbrCap) D.nbr[row * kNbrCap + slot] = (uint16_t)winner;
  };
  // Hits are collected across items and recorded kPairHits at a time: the two key loads and the atomic of a hit are
  // dependent round trips to L2, paid once per batch this way instead of once per 32 queued pairs.
  int n_hits = 0;
  auto flush_hits = [&]() {
    __syncwarp();
    for (int e = lane; e < n_hits; e += 32) record(S.hits[e]);
    n_hits = 0;
    __syncwarp();
  };
  for (;; item = n_warps + __shfl_sync(0xffffffffu, next, 0)) {
    if (item >= total) break;
    if (lane == 0) next = atomicAdd(D.work, 1);  // (in flight while this item is worked on)
    // frame of the item: how many frames start at or before it
    const int frame = __popc(__ballot_sync(0xffffffffu, s_first[1 + lane] <= item)) +
                      __popc(__ballot_sync(0xffffffffu, s_first[33 + lane] <= item));
    const int n = s_n[frame];
    const int Cn = (n + kPairCols - 1) / kPairCols;
    int local = item - s_first[frame], r = 0;
    while (local >= Cn - kPairRC * r) {
      local -= Cn - kPairRC * r;
      ++r;
    }
    const int c = kPairRC * r + local;
    const size_t cbase = (size_t)frame * p.max_cand;
    const int jb = c * kPairCols, jn = min(kPairCols, n - jb);
    const int row0 = r * kPairRows;
    float4 bi[kPairGroups];
#pragma unroll
    for (int q = 0; q < kPairGroups; ++q) {
      const int rl = q * 32 + lane, i = row0 + rl;
      bi[q] = make_float4(0.f, 0.f, 0.f, 0.f);
      int ci = 0;
      if (i < n) {
        ci = p.cand_cls[cbase + i];
        bi[q] = nms_view_of_box(p, p.cand_box[cbase + i], ci);
      }
      S.row[rl] = bi[q];
      S.rcl[rl] = ci;
    }
#pragma unroll
    for (int h = 0; h < kPairCols / 32; ++h) {
      const int cl = 32 * h + lane;
      if (cl < jn) {
        const int cj = p.cand_cls[cbase + jb + cl];
        S.col[cl] = nms_view_of_box(p, p.cand_box[cbase + jb + cl], cj);
        S.ccl[cl] = cj;
      }
    }
    __syncwarp();
    // one overlapping pair, rows and columns by their position in the item: does either box suppress the other?
    auto test_pair = [&](const int rl, const int col) -> bool {
      if (aware && S.rcl[rl] != S.ccl[col]) return false;
      const float4 a = S.row[rl], b = S.col[col];
      return ultra ? suppresses_tv(a, b, p.iou_thr64) : suppresses(a, b, thr);
    };
    const uint32_t hit_base = ((uint32_t)frame << 24) | ((uint32_t)row0 << 12) | (uint32_t)jb;  // + (row << 12 | column) in the item
#pragma unroll 1
    for (int w = 0; w < kPairCols / 32; ++w) {
      const int j0 = jb + 32 * w, cnt = min(32, n - j0);
      if (cnt <= 0 || j0 + 31 <= row0) continue;  // (warp-uniform) no column of the word lies behind a row of the warp
      const float4* __restrict__ pc = S.col + 32 * w;
      uint32_t cand[kPairGroups];
#pragma unroll
      for (int q = 0; q < kPairGroups; ++q) cand[q] = thr_nonneg ? 0u : 0xffffffffu;  // a negative threshold: disjoint boxes suppress each other too
      if (thr_nonneg) {
        // Two boxes are apart when one ends before the other begins, on either axis: the sign of one of four
        // differences (subtractions on the FMA pipe; two LOP3 and a funnel shift -- sign bit into the accumulator --
        // on the ALU pipe).  Touching boxes (difference +0) and NaN coordinates (the canonical NaN is positive, and
        // nan_box_view made every coordinate of such a box NaN) stay in: the formula then decides.
#pragma unroll
        for (int b = 0; b < 32; ++b) {
          const float4 cb = pc[b];
#pragma unroll
          for (int q = 0; q < kPairGroups; ++q) {
            const int t = __float_as_int(__fsub_rn(cb.z, bi[q].x)) | __float_as_int(__fsub_rn(bi[q].z, cb.x)) |
                          __float_as_int(__fsub_rn(cb.w, bi[q].y)) | __float_as_int(__fsub_rn(bi[q].w, cb.y));
            cand[q] = __funnelshift_l((uint32_t)t, cand[q], 1);  // bit 31 - b: column b is apart from the row
          }
        }
#pragma unroll
        for (int q = 0; q < kPairGroups; ++q) cand[q] = ~__brev(cand[q]);
      }
      // columns of this frame that come after row i; queue what is left
      const uint32_t in_frame = cnt == 32 ? 0xffffffffu : ((1u << cnt) - 1u);
      int mine = 0;
#pragma unroll
      for (int q = 0; q < kPairGroups; ++q) {
        const int i = row0 + q * 32 + lane;
        uint32_t live = in_frame;
        if (i >= j0) live = (i - j0 >= 31) ? 0u : (live & ~((2u << (i - j0)) - 1u));
        cand[q] = i < n ? (cand[q] & live) : 0u;
        mine += __popc(cand[q]);
      }
      int incl = mine;
#pragma unroll
      for (int o = 1; o < 32; o <<= 1) {
        const int t = __shfl_up_sync(0xffffffffu, incl, o);
        if (lane >= o) incl += t;
      }
      const int queued = min(__shfl_sync(0xffffffffu, incl, 31), kPairQueue);
      int pos = incl - mine;
#pragma unroll
      for (int q = 0; q < kPairGroups; ++q) {
        uint32_t cq = cand[q];
        while (cq) {
          const int b = __ffs((int)cq) - 1;
          cq &= cq - 1u;
          if (pos < kPairQueue) S.queue[pos] = (uint16_t)(((q * 32 + lane) << kPairColBits) | (32 * w + b));
          else if (test_pair(q * 32 + lane, 32 * w + b)) record(hit_base + ((uint32_t)(q * 32 + lane) << 12) + (uint32_t)(32 * w + b));  // (queue full: on the spot)
          ++pos;
        }
      }
      __syncwarp();
      for (int e0 = 0; e0 < queued; e0 += 32) {
        if (n_hits > kPairHits - 32) flush_hits();
        const int e = e0 + lane;
        const int code = e < queued ? S.queue[e] : 0;
        const bool hit = e < queued && test_pair(code >> kPairColBits, code & (kPairCols - 1));
        const unsigned bal = __ballot_sync(0xffffffffu, hit);
        if (hit) S.hits[n_hits + __popc(bal & ((1u << lane) - 1u))] = hit_base + ((uint32_t)(code >> kPairColBits) << 12) + (uint32_t)(code & (kPairCols - 1));
        n_hits += __popc(bal);
      }
      __syncwarp();
    }
  }
  flush_hits();
}

__device__ __forceinline__ void dense_resolve_frame(const NmsParams& p, const DenseNms& D, uint8_t* const smem_raw) {
  __shared__ int s_m, s_out;
  const int tid = threadIdx.x, lane = tid & 31, frame = blockIdx.x;
  PHASE_STAMP(p.dbg, 36);
  const int n_raw = (p.skip && p.skip[frame]) ? 0 : p.cand_count[frame];
  const int n = min(n_raw, p.max_cand);
  const size_t cbase = (size_t)frame * p.max_cand, fbase = (size_t)frame * D.max_cand;
  // suppressor lists of this thread's rows: count, first eight entries (registers), the key
  int cnt[kResolveRows];
  uint4 nb[kResolveRows];
  unsigned long long key[kResolveRows];
  bool over = false;
#pragma unroll
  for (int q = 0; q < kResolveRows; ++q) {
    const int r = tid + q * kResolveThreads;
    cnt[q] = r < n ? D.nbr_cnt[fbase + r] : 0;
    key[q] = r < n ? p.cand_key[cbase + r] : 0ull;
    // (fetched in the same round trip as the count; entries past the count are stale and never looked at)
    nb[q] = r < n ? *reinterpret_cast<const uint4*>(D.nbr + (fbase + r) * kNbrCap) : make_uint4(0u, 0u, 0u, 0u);
  }
#pragma unroll
  for (int q = 0; q < kResolveRows; ++q) {
    const int r = tid + q * kResolveThreads;
    if (cnt[q] > 0) {
      D.nbr_cnt[fbase + r] = 0;  // left clean for the next launch
      over |= cnt[q] > kNbrCap;
    }
  }
  const int kstride = (D.max_cand + 15) & ~15;
  uint8_t* kept_a = smem_raw;           // [max_cand]
  uint8_t* kept_b = kept_a + kstride;   // [max_cand]
  unsigned long long* kkeys = reinterpret_cast<unsigned long long*>(smem_raw + 2 * (size_t)kstride);  // [pow2 >= max_cand]
#pragma unroll
  for (int q = 0; q < kResolveRows; ++q) {
    const int r = tid + q * kResolveThreads;
    if (r < n) kept_a[r] = kept_b[r] = cnt[q] == 0;  // nothing ahead suppresses it: kept, for good
  }
  if (tid == 0) {
    s_m = 0;
    s_out = 0;
  }
  const int fall_back = __syncthreads_or(over);  // (also: every thread has read the count)
  if (tid == 0) {
    if (p.stats && n > 256) *(volatile int*)p.stats = n;
    p.cand_count[frame] = 0;
    if (n_raw > p.max_cand) atomicOr(p.flags + FLAG_CAND_OVERFLOW, 1);
    if (frame == 0) *D.work = 0;  // (every CTA of k_dense_pairs has finished: griddep_wait / stream order)
  }
  if (n == 0) {
    if (tid == 0) p.out_count[frame] = 0;
    return;
  }
  PHASE_STAMP(p.dbg, 37);
  if (fall_back) {
    nms_general<true, kResolveThreads>(p, frame, smem_raw, n);
    return;
  }
  // kept_i = no kept suppressor, iterated from "only the unsuppressible boxes are kept" until nothing changes
  uint8_t *old = kept_a, *nw = kept_b;
  bool converged = false;
  for (int round = 0; round < kResolveRounds; ++round) {
    int changed = 0;
#pragma unroll
    for (int q = 0; q < kResolveRows; ++q) {
      if (cnt[q] > 0) {
        const int r = tid + q * kResolveThreads;
        const uint32_t w[4] = {nb[q].x, nb[q].y, nb[q].z, nb[q].w};
        bool k = true;
#pragma unroll
        for (int s = 0; s < 8; ++s)
          if (s < cnt[q]) k = k && !old[(w[s >> 1] >> (16 * (s & 1))) & 0xffffu];
        if (k && cnt[q] > 8) {
          const uint16_t* __restrict__ more = D.nbr + (fbase + r) * kNbrCap;
          for (int s = 8; s < cnt[q]; ++s)
            if (old[more[s]]) {
              k = false;
              break;
            }
        }
        changed |= (int)(k != (old[r] != 0));
        nw[r] = k;
      }
    }
    uint8_t* t = old;
    old = nw;
    nw = t;
    if (!__syncthreads_or(changed)) {
      converged = true;
      break;
    }
  }
  if (!converged) {  // a suppression chain deeper than kResolveRounds: let the sequential path walk it
    nms_general<true, kResolveThreads>(p, frame, smem_raw, n);
    return;
  }
  PHASE_STAMP(p.dbg, 38);
  // the kept keys, in no particular order
#pragma unroll
  for (int q = 0; q < kResolveRows; ++q) {
    const int r = tid + q * kResolveThreads;
    const bool k = r < n && old[r];
    const unsigned bal = __ballot_sync(0xffffffffu, k);
    int base = 0;
    if (lane == 0 && bal) base = atomicAdd(&s_m, __popc(bal));
    base = __shfl_sync(0xffffffffu, base, 0);
    if (k) kkeys[base + __popc(bal & ((1u << lane) - 1u))] = key[q];
  }
  __syncthreads();
  PHASE_STAMP(p.dbg, 39);
  const int m = s_m;
  const bool ultra = p.ultra != 0;
  // output position = rank among the kept keys.  ultralytics: `i = i[:max_det]` on the NMS survivors, before anything
  // else looks at them; filter_detections (detector.py:99-103): float64 compare on the kept boxes only (a threshold on
  // the score the keys are ordered by, so the boxes that pass are a prefix and their ranks do not move)
  auto emit = [&](const unsigned long long k, const int pos) {
    if (ultra && pos >= p.max_det_cap) return;
    const float conf = key_conf(k);
    if (p.use_filter && !((double)conf >= p.filter_thr)) return;
    atomicAdd(&s_out, 1);
    if (pos >= p.max_dets) return;
    const int slot = key_slot(k);
    const size_t o = (size_t)frame * p.max_dets + pos;
    float4 b = p.cand_box[cbase + slot];
    if (ultra) b = ultra_scale_box(b, p.f[frame]);
    reinterpret_cast<float4*>(p.out_box)[o] = b;
    p.out_conf[o] = conf;
    p.out_cls[o] = p.cand_cls[cbase + slot];
  };
  if (m <= kRankMax) {
    // eight lanes share four kept keys (registers) and split the scan of all kept keys between them: a 64-bit
    // shared-memory load feeds four compares (one compare per load is bound by the shared-memory pipe)
    static_assert(kRankMax == 4 * (kResolveThreads / 8), "four keys per group of eight lanes cover kRankMax");
    const int g = tid >> 3, part = tid & 7;
    unsigned long long ke[4];
    int ahead[4] = {0, 0, 0, 0};
#pragma unroll
    for (int k = 0; k < 4; ++k) ke[k] = g + k * (kResolveThreads / 8) < m ? kkeys[g + k * (kResolveThreads / 8)] : ~0ull;
    for (int t = part; t < m; t += 8) {
      const unsigned long long kt = kkeys[t];
#pragma unroll
      for (int k = 0; k < 4; ++k) ahead[k] += kt > ke[k];
    }
#pragma unroll
    for (int k = 0; k < 4; ++k) {
      ahead[k] += __shfl_xor_sync(0xffffffffu, ahead[k], 1);
      ahead[k] += __shfl_xor_sync(0xffffffffu, ahead[k], 2);
      ahead[k] += __shfl_xor_sync(0xffffffffu, ahead[k], 4);
    }
    // (lane k of a group emits key k: the stores of a warp spread over its lanes)
#pragma unroll
    for (int k = 0; k < 4; ++k)
      if (part == k && g + k * (kResolveThreads / 8) < m) emit(ke[k], ahead[k]);
  } else {
    int np2 = 64;
    while (np2 < m) np2 <<= 1;
    for (int t = m + tid; t < np2; t += kResolveThreads) kkeys[t] = 0ull;
    __syncthreads();
    block_bitonic_sort_desc<kResolveThreads>(kkeys, np2);
    for (int t = tid; t < m; t += kResolveThreads) emit(kkeys[t], t);
  }
  __syncthreads();
  PHASE_STAMP(p.dbg, 48);
  if (tid == 0) {
    p.out_count[frame] = min(s_out, p.max_dets);
    if (s_out > p.max_dets) atomicOr(p.flags + FLAG_DET_OVERFLOW, 1);
  }
}

static int next_pow2(int v) {
  int p = 64;
  while (p < v) p <<= 1;
  return p;
}

}  // namespace

static size_t nms_base_bytes(int max_cand) {
  const size_t cap = (size_t)next_pow2(max_cand);
  const size_t general = (cap * 24 + cap / 8 + cap / 8 + (cap / 64 + 1) * 4 + cap * 2 + 64 + 15) & ~(size_t)15;  // keys, boxes, supp, keep_w, keep_off, classes
  return std::max(general, (sizeof(SmallNms) + 15) & ~(size_t)15);  // frames of at most kSmallN candidates use their own layout
}
// the kept-box grid is carried when the candidate capacity leaves room for it (cap <= 4096: 106 KB + 21 KB)
static size_t nms_grid_offset(int max_cand) { return next_pow2(max_cand) <= 4096 ? nms_base_bytes(max_cand) : 0; }
size_t nms_smem_bytes(int max_cand) {
  const size_t cap = (size_t)next_pow2(max_cand);
  return nms_base_bytes(max_cand) + (nms_grid_offset(max_cand) ? sizeof(NmsGrid) + cap / 8 + cap * 2 : 0);
}
__global__ void __launch_bounds__(kResolveThreads) k_dense_resolve(const __grid_constant__ NmsParams p, const DenseNms D) {
  extern __shared__ __align__(16) uint8_t smem_raw[];
  griddep_launch_dependents();  // a tracker kernel behind this one may be scheduled; its griddep_wait() waits for this grid
  griddep_wait();
  dense_resolve_frame(p, D, smem_raw);
}

// Dense scenes with the tracker update in the same call: the resolution of frame i and the tracker update of stream i in
// ONE CTA (as k_post_track does for sparse scenes) -- one launch and one grid-to-grid dependency fewer on the chain
// decode -> pairs -> resolve -> tracker, which is what a dense tick waits for.
static_assert(kResolveThreads == kTrkThreadsMax, "the fused dense kernel runs both halves at the tracker's widest launch");
__global__ void __launch_bounds__(kResolveThreads) k_dense_resolve_track(const __grid_constant__ NmsParams q, const DenseNms D,
                                                                          const __grid_constant__ TrkParams t) {
  extern __shared__ __align__(16) uint8_t smem_raw[];
  __shared__ TrkShared sh;
  griddep_launch_dependents();
  griddep_wait();
  TIMELINE_BEGIN(q.dbg, 44);
  dense_resolve_frame(q, D, smem_raw);
  __syncthreads();  // this frame's detections were written by this CTA: visible to all of its threads from here on
  TIMELINE_END(q.dbg, 44);
  TIMELINE_BEGIN(q.dbg, 46);
  tracker_stream<false>(t, blockIdx.x, smem_raw, sh, -1);
  TIMELINE_END(q.dbg, 46);
}

static size_t dense_resolve_smem(int max_cand) {
  int np2 = 64;
  while (np2 < max_cand) np2 <<= 1;
  const size_t own = 2 * (((size_t)max_cand + 15) & ~(size_t)15) + (size_t)np2 * 8;
  return std::max(own, nms_smem_bytes(max_cand));
}



static const int kRingSmemMax = 96 * 1024;

// Tile width, stage shape and grid of k_decode_ring for `frames` heads of [C, A].  Every CTA must be resident
// (ctas_per_sm per SM) and should own the same number of tiles: the widest tile whose busiest CTA carries at most
// 2 % more than the mean wins.  B200VA_DECODE_TA / _ROWS / _STAGES / _CTAS_PER_SM override the choice
// (tools/bench_decode.py sweeps them).
static void ring_plan(const b200va_ctx* h, int frames, int C, int A, int cls0, RingCfg* rc, int* n_cta, size_t* smem) {
  const int per_sm = h->tune.decode_ctas_per_sm > 0 ? h->tune.decode_ctas_per_sm : 3;
  const int cap = h->num_sms * per_sm;
  auto eval = [&](int ta, int* ctas) {
    const long long tiles = (long long)((A + ta - 1) / ta) * frames;
    const long long tpc = (tiles + cap - 1) / cap;
    *ctas = (int)((tiles + tpc - 1) / tpc);
    return (double)frames * A / ((double)*ctas * (double)tpc * ta);
  };
  // a tile is one TMA box of up to 256 anchors, or two boxes; a box row is a multiple of 128 bytes so that every
  // box and stage starts 128-byte aligned in shared memory (a TMA requirement)
  auto valid = [](int t) { return t >= 64 && t <= 512 && (t <= 256 ? t % 32 == 0 : t % 64 == 0); };
  int ta = h->tune.decode_ta, ctas = 0;
  if (!valid(ta)) {
    double best = -1.0;
    ta = 128;
    for (int t = 256; t >= 128; t -= 32) {
      int c;
      const double e = eval(t, &c);
      if (e >= 0.98) {
        ta = t;
        break;
      }
      if (e > best) best = e, ta = t;
    }
  }
  eval(ta, &ctas);
  rc->ta = ta;
  rc->boxes = ta > 256 ? 2 : 1;
  rc->bw = ta / rc->boxes;
  rc->tiles_per_frame = (A + ta - 1) / ta;
  rc->n_tiles = rc->tiles_per_frame * frames;
  rc->warps = (ta / 4 + 31) / 32;
  // rows per stage: ~20 KB stages by default, as equal as possible over the C rows, never fewer than the box rows +
  // objectness + one class row (the consumers expect them in a tile's first stage)
  int rows = h->tune.decode_rows;
  if (rows <= 0) {
    const int want = (20 * 1024) / (ta * 4);
    const int n_stage = (C + want - 1) / (want > 0 ? want : 1);
    rows = (C + n_stage - 1) / n_stage;
  }
  if (rows < cls0 + 1) rows = cls0 + 1;
  if (rows > 256) rows = 256;
  if (rows > C) rows = C;
  rc->rows = rows;
  const size_t stage = (size_t)rows * ta * 4;
  int stages = h->tune.decode_stages > 0 ? h->tune.decode_stages : (int)((size_t)(64 * 1024) / stage);
  if (stages < 2) stages = 2;
  if (stages > kRingMaxStages) stages = kRingMaxStages;
  while (stages > 2 && stages * stage > (size_t)kRingSmemMax) --stages;
  rc->stages = stages;
  *n_cta = ctas;
  *smem = stages * stage;
}

// cuTensorMapEncodeTiled through the runtime (no link-time dependency on libcuda)
typedef CUresult (*EncodeTiledFn)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*, const cuuint64_t*,
                                  const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave, CUtensorMapSwizzle,
                                  CUtensorMapL2promotion, CUtensorMapFloatOOBfill);
static EncodeTiledFn encode_tiled_fn() {
  static EncodeTiledFn fn = [] {
    void* p = nullptr;
    cudaDriverEntryPointQueryResult q;
    if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &p, cudaEnableDefault, &q) != cudaSuccess || q != cudaDriverEntryPointSuccess) {
      cudaGetLastError();
      p = nullptr;
    }
    return (EncodeTiledFn)p;
  }();
  return fn;
}

// tensor map over a head [B, C, A] float32 with boxes of `bw` anchors x `rows` channel rows of one frame
static bool head_tensor_map(const float* head, int B, int C, int A, int bw, int rows, CUtensorMap* out) {
  EncodeTiledFn enc = encode_tiled_fn();
  if (!enc) return false;
  const cuuint64_t dims[3] = {(cuuint64_t)A, (cuuint64_t)C, (cuuint64_t)B};
  const cuuint64_t strides[2] = {(cuuint64_t)A * 4, (cuuint64_t)A * 4 * (cuuint64_t)C};
  const cuuint32_t box[3] = {(cuuint32_t)bw, (cuuint32_t)rows, 1};
  const cuuint32_t estr[3] = {1, 1, 1};
  return enc(out, CU_TENSOR_MAP_DATA_TYPE_FLOAT32, 3, const_cast<float*>(head), dims, strides, box, estr,
             CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_NONE, CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
             CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE) == CUDA_SUCCESS;
}

int postprocess_configure(b200va_ctx* h) {
  CUDA_TRY(h, cudaFuncSetAttribute(k_decode_ring, cudaFuncAttributeMaxDynamicSharedMemorySize, kRingSmemMax));
  if (h->tune.uniform_carveout) {  // B200VA_UNIFORM_CARVEOUT=1 (experiment, see prefer_max_shared)
    CUDA_TRY(h, prefer_max_shared(k_decode_cm<4>));
    CUDA_TRY(h, prefer_max_shared(k_decode_cm<1>));
    CUDA_TRY(h, prefer_max_shared(k_decode_cm_split<8, 12>));
    CUDA_TRY(h, prefer_max_shared(k_decode_am));
    CUDA_TRY(h, prefer_max_shared(k_decode_ring));
    CUDA_TRY(h, prefer_max_shared(k_decode16_cm<8>));
    CUDA_TRY(h, prefer_max_shared(k_decode16_cm<1>));
    CUDA_TRY(h, prefer_max_shared(k_decode16_cm_split));
    CUDA_TRY(h, prefer_max_shared(k_decode16_am));
    CUDA_TRY(h, prefer_max_shared(k_sort_nms<false>));
    CUDA_TRY(h, prefer_max_shared(k_sort_nms<true>));
    CUDA_TRY(h, prefer_max_shared(k_post_track<false>));
    CUDA_TRY(h, prefer_max_shared(k_post_track<true>));
  }
  const size_t smem = nms_smem_bytes(h->cfg.max_candidates);
  if (smem > 220 * 1024) return set_error(h, B200VA_ERR_INVALID, "max_candidates %d needs %zu bytes of shared memory", h->cfg.max_candidates, smem);
  {
    const size_t fused = std::min<size_t>(200 * 1024, std::max(smem, tracker_smem_bytes(std::min(h->cfg.max_tracks, kTrkSmemRowsMax))));
    CUDA_TRY(h, raise_dyn_smem(k_post_track<false>, fused));
    CUDA_TRY(h, raise_dyn_smem(k_post_track<true>, fused));
    // k_post_track runs beside the letterbox in b200va_tick, and an SM only hosts kernels that agree on its L1 /
    // shared-memory split (see prefer_max_shared): ask for the split the letterbox launches get -- all of it: six
    // 34 KB CTAs at 1080p (preprocess.cu: the shared-memory floor that keeps it at six), two or three 50-100 KB CTAs at
    // 4K -- instead of the one the driver would derive from this kernel's own occupancy.  Measured on the 32 x 1080p
    // tick: 63.5 us with 100 %, 64.3 us with 86 %, 65.5 us with the 71 % that matched the letterbox of round 1 (six
    // 24.5 KB CTAs): with a split that differs, the 32 SMs that host this kernel are closed to letterbox CTAs.
    const int pct = h->tune.post_carveout >= 0 ? h->tune.post_carveout : 100;
    if (pct > 0) {
      CUDA_TRY(h, cudaFuncSetAttribute(k_post_track<false>, cudaFuncAttributePreferredSharedMemoryCarveout, pct));
      CUDA_TRY(h, cudaFuncSetAttribute(k_post_track<true>, cudaFuncAttributePreferredSharedMemoryCarveout, pct));
    }
  }
  CUDA_TRY(h, raise_dyn_smem(k_sort_nms<false>, smem));
  CUDA_TRY(h, raise_dyn_smem(k_sort_nms<true>, smem));
  // dense-scene path (k_dense_pairs / k_dense_resolve): suppressor lists of every candidate
  if (h->cfg.max_candidates <= kDenseCandMax && h->tune.dense_impl != 1) {
    DenseNms* D = new DenseNms();
    memset(D, 0, sizeof(*D));
    h->dense_nms = D;
    D->max_cand = h->cfg.max_candidates;
    D->ctas = h->num_sms * (h->tune.dense_ctas_per_sm > 0 ? h->tune.dense_ctas_per_sm : 8);
    const size_t rows = (size_t)h->cand_set_frames * D->max_cand;
    CUDA_TRY(h, cudaMalloc(&D->nbr_cnt, rows * sizeof(int32_t)));
    CUDA_TRY(h, cudaMalloc(&D->nbr, rows * kNbrCap * sizeof(uint16_t)));
    CUDA_TRY(h, cudaMemset(D->nbr_cnt, 0, rows * sizeof(int32_t)));
    CUDA_TRY(h, cudaMalloc(&D->work, sizeof(int32_t)));
    CUDA_TRY(h, cudaMemset(D->work, 0, sizeof(int32_t)));
    CUDA_TRY(h, raise_dyn_smem(k_dense_resolve, dense_resolve_smem(D->max_cand)));
    if (h->tune.dense_carveout >= 0) {  // B200VA_DENSE_CARVEOUT=pct (see the note on k_post_track's carve-out above)
      CUDA_TRY(h, cudaFuncSetAttribute(k_dense_pairs, cudaFuncAttributePreferredSharedMemoryCarveout, h->tune.dense_carveout));
      CUDA_TRY(h, cudaFuncSetAttribute(k_dense_resolve, cudaFuncAttributePreferredSharedMemoryCarveout, h->tune.dense_carveout));
      CUDA_TRY(h, cudaFuncSetAttribute(k_dense_resolve_track, cudaFuncAttributePreferredSharedMemoryCarveout, h->tune.dense_carveout));
    }
    CUDA_TRY(h, raise_dyn_smem(k_dense_resolve_track,
                               std::min<size_t>(200 * 1024, std::max(dense_resolve_smem(D->max_cand),
                                                                     tracker_smem_bytes(std::min(h->cfg.max_tracks, kTrkSmemRowsMax))))));
  }
  return B200VA_OK;
}

namespace {
// b200va_tick: the tracker update that follows this post-process on the same stream.  When the launch qualifies, NMS
// and tracker run as one kernel (k_post_track) and `done` is set; otherwise the caller launches the tracker itself.
struct FuseReq {
  const int* stream_slots;
  int batch, max_dets;
  const double* det_scale;
  const uint8_t* skip;
  const b200va_tracker_cfg* cfg;
  const int64_t* id_base;
  const b200va_tracks* out;
  int32_t* new_counts;
  bool done;
  bool tail_on_side;  // schedule 3: NMS (and the fused tracker) went to the handle's tail stream
  bool defer;         // schedule 4: only decode now; NMS + tracker are stashed in the handle and launched by the next tick
};

// schedule 4: the NMS (+ tracker) launch a decode still owes, with everything it needs held by value
struct PendingChain {
  NmsParams q;
  TrkParams t;
  bool has_trk;  // t is filled: the tracker update of the same rows follows the NMS
  int n;         // frames
};

struct UltraOpts {  // b200va_postprocess_ultralytics
  const int* src_h;
  const int* src_w;
  int in_h, in_w, agnostic, max_det;
};
}  // namespace

static int postprocess_impl(b200va_handle h, const void* head, int layout, int batch, int channels, int anchors,
                                  const b200va_letterbox* meta, double conf_thr, double iou_thr,
                                  const int32_t* classes, int n_classes, int score_mode, int nms_mode,
                                  double filter_conf_thr_f64, int use_filter, const b200va_dets* out, void* stream,
                                  const UltraOpts* ultra, FuseReq* fuse = nullptr) {
  if (!h) return B200VA_ERR_INVALID;
  std::lock_guard<std::recursive_mutex> lock(h->mu);
  DeviceGuard guard(h->cfg.device);
  cudaStream_t st = (cudaStream_t)stream;
  REQUIRE(h, head && (meta || ultra) && out && out->bbox_xyxy && out->conf && out->cls && out->count, "NULL argument");
  if (ultra) {
    REQUIRE(h, ultra->src_h && ultra->src_w && ultra->in_h > 0 && ultra->in_w > 0, "bad frame / input shapes");
    REQUIRE(h, ultra->max_det >= 1, "max_det must be positive");
  }
  REQUIRE(h, batch >= 0 && batch <= h->cfg.max_batch, "batch %d outside [0, %d]", batch, h->cfg.max_batch);
  const bool f16 = (layout & B200VA_HEAD_F16) != 0;
  const int order = layout & ~B200VA_HEAD_F16;
  REQUIRE(h, order == B200VA_HEAD_CHANNEL_MAJOR || order == B200VA_HEAD_ANCHOR_MAJOR, "unknown layout %d", layout);
  layout = order;
  REQUIRE(h, score_mode == B200VA_SCORE_REF_COMPAT || score_mode == B200VA_SCORE_V8_NATIVE, "unknown score mode %d", score_mode);
  REQUIRE(h, nms_mode == B200VA_NMS_AGNOSTIC || nms_mode == B200VA_NMS_CLASS_AWARE, "unknown nms mode %d", nms_mode);
  REQUIRE(h, nms_mode == B200VA_NMS_AGNOSTIC || channels - 4 <= 65535, "class-aware NMS supports at most 65535 classes");
  REQUIRE(h, anchors >= 0 && anchors <= h->cfg.max_anchors, "anchors %d outside [0, %d]", anchors, h->cfg.max_anchors);
  // detector.py:285-287: fewer than 5 channels is "unexpected shape" -> no detections
  if (batch == 0) return B200VA_OK;
  if (channels < 5 || anchors == 0) {
    CUDA_TRY(h, cudaMemsetAsync(out->count, 0, sizeof(int32_t) * batch, st));
    return B200VA_OK;
  }
  REQUIRE(h, n_classes >= 0 && (n_classes == 0 || classes), "class whitelist is NULL");
  // the whitelist is a bitmap over class ids 0..2047 in the kernel parameters; a larger id that the head can produce is
  // refused rather than silently never matched (ids < 0 or >= the class count match nothing, as in np.isin)
  const int n_cls_rows = channels - ((score_mode == B200VA_SCORE_REF_COMPAT && channels > 5) ? 5 : 4);
  for (int k = 0; k < n_classes; ++k)
    REQUIRE(h, classes[k] < kClassMaskIds || classes[k] >= n_cls_rows,
            "class whitelist id %d: ids >= %d are not supported", classes[k], kClassMaskIds);

  for (int base = 0; base < batch; base += B200VA_LAUNCH_FRAMES) {
    const int n = batch - base < B200VA_LAUNCH_FRAMES ? batch - base : B200VA_LAUNCH_FRAMES;
    PostParams p;
    memset(&p, 0, sizeof(p));
    for (int i = 0; i < n; ++i) {
      if (ultra) {
        // ultralytics scale_boxes (utils/ops.py): gain = min(h1/h0, w1/w0); pad = round((s1 - s0*gain)/2 - 0.1)
        // (Python round = round-half-even = nearbyint); boxes /= gain; clamp to [0, w0] x [0, h0]
        const int h0 = ultra->src_h[base + i], w0 = ultra->src_w[base + i];
        REQUIRE(h, h0 > 0 && w0 > 0, "frame %d has bad size", base + i);
        const double g0 = (double)ultra->in_h / h0, g1 = (double)ultra->in_w / w0;
        const double gain = g0 < g1 ? g0 : g1;
        p.f[i].left = (float)nearbyint(((double)ultra->in_w - (double)w0 * gain) / 2 - 0.1);
        p.f[i].top = (float)nearbyint(((double)ultra->in_h - (double)h0 * gain) / 2 - 0.1);
        p.f[i].scale = (float)gain;
        p.f[i].xmax = (float)w0;
        p.f[i].ymax = (float)h0;
        continue;
      }
      const b200va_letterbox& m = meta[base + i];
      p.f[i].left = (float)m.pad_left;
      p.f[i].top = (float)m.pad_top;
      p.f[i].scale = (float)m.scale;  // NumPy rounds the Python float to float32 for `boxes /= scale`
      p.f[i].xmax = (float)(m.src_w - 1);
      p.f[i].ymax = (float)(m.src_h - 1);
    }
    if (n_classes > 0) {  // an empty list means "no filter" (detector.py:313: `if self.config.classes`)
      p.use_mask = 1;
      for (int k = 0; k < n_classes; ++k)
        if (classes[k] >= 0 && classes[k] < kClassMaskIds) p.class_mask[classes[k] >> 5] |= 1u << (classes[k] & 31);
    }
    const bool defer = fuse && fuse->defer && base == 0 && n == batch;
    const int set = defer ? h->cand_set : 0;  // ordinary calls always use set 0 (decode and NMS in the same call)
    p.head = head;
    p.cand_key = h->cand_key + (size_t)set * h->cand_set_elems;
    p.cand_box = h->cand_box + (size_t)set * h->cand_set_elems;
    p.cand_cls = h->cand_cls + (size_t)set * h->cand_set_elems;
    p.cand_count = h->cand_count + (size_t)set * h->cand_set_frames;
    p.C = channels;
    p.A = anchors;
    p.max_cand = h->cfg.max_candidates;
    p.dbg = h->dbg;
    // REF_COMPAT (detector.py:294-307): C > 5 -> class columns 5.. times column 4; C == 5 -> pred[:, 4:].
    // V8_NATIVE: class columns 4.. as they are (what a YOLOv8 export actually contains).
    p.use_obj = (score_mode == B200VA_SCORE_REF_COMPAT && channels > 5) ? 1 : 0;
    p.cls0 = p.use_obj ? 5 : 4;
    p.conf_thr = (float)conf_thr;  // NEP-50 weak scalar: compared in float32 (detector.py:312)
    p.ultra = ultra ? 1 : 0;
    p.skip = h->skip_dev;
    {
    PhaseScope phase(h, B200VA_PHASE_DECODE, st);
    const int impl = h->tune.decode_impl;  // 0 auto, 1 registers (k_decode_cm), 2 ring, 3 split
    if (f16) {
      // the float16 kernels: the same selection with 16-byte loads of 8 anchors, the split variant with 8-byte loads of
      // 4, and no ring (it buys nothing in float32 either, see below)
      const uintptr_t addr = (uintptr_t)head;
      const int n_cls_rows = channels - p.cls0;
      const bool vec8 = anchors % 8 == 0 && addr % 16 == 0;
      const bool split_ok = anchors % 4 == 0 && addr % 8 == 0 && n_cls_rows >= 16 && n_cls_rows <= 96;
      if (layout == B200VA_HEAD_ANCHOR_MAJOR) {
        k_decode16_am<<<dim3((anchors + 7) / 8, n), 256, 0, st>>>(p, base);
      } else if (split_ok && (impl == 3 || (impl == 0 && n <= 8))) {
        k_decode16_cm_split<<<dim3((anchors / 4 + 31) / 32, n), 256, 0, st>>>(p, base);
      } else if (vec8) {
        k_decode16_cm<8><<<dim3((anchors / 8 + 63) / 64, n), 64, 0, st>>>(p, base);
      } else {
        k_decode16_cm<1><<<dim3((anchors + 63) / 64, n), 64, 0, st>>>(p, base);
      }
    } else if (layout == B200VA_HEAD_CHANNEL_MAJOR) {
      // 16-byte loads need every channel row (A floats) and the tensor base 16-byte aligned
      // (a TMA-staged variant -- all C rows of a 128-anchor tile bulk-copied to shared memory -- measured
      // 24.6 us against 21.5 us for this register version on [32,84,8400]: the 512-byte row pieces at a
      // 33.6 KB stride bound both; block sizes 64..256 are equivalent, 512 is slower)
      const int n_cls_rows = channels - p.cls0;
      const bool vec4 = anchors % 4 == 0 && ((uintptr_t)head % 16 == 0);
      // few frames: latency-bound, split the class rows over 8 warps; many frames: HBM-bound, the TMA-fed persistent ring
      const bool split_ok = vec4 && n_cls_rows >= 16 && n_cls_rows <= 96;
      // The ring kernel is opt-in (B200VA_DECODE_IMPL=2): measured on [32, 84, 8400] it is no faster than the register
      // kernel, and neither can be -- a pure 90 MB read of this tensor takes 19.4 us on a B200 whatever fetches it
      // (linear LDG, 1-D bulk copies with enough issuing warps, tensor-map boxes: tools/readbw.cu,
      // profiles/r2_readbw.log), and k_decode_cm<4> needs 20.1 us.
      bool ring_ok = vec4 && anchors >= 128 && impl == 2 && !h->skip_dev;
      RingCfg rc;
      int ring_ctas = 0;
      size_t ring_smem = 0;
      alignas(64) CUtensorMap tmap;
      if (ring_ok) {
        ring_plan(h, n, channels, anchors, p.cls0, &rc, &ring_ctas, &ring_smem);
        // the map spans the frames of this launch only (coordinate 2 = frame index inside the launch)
        ring_ok = ring_smem <= (size_t)kRingSmemMax &&
                  head_tensor_map(static_cast<const float*>(head) + (size_t)base * channels * anchors, n, channels, anchors, rc.bw, rc.rows, &tmap);
      }
      if (split_ok && (impl == 3 || (impl == 0 && n <= 8))) {
        dim3 grid((anchors / 4 + 31) / 32, n);
        k_decode_cm_split<8, 12><<<grid, 256, 0, st>>>(p, base);
      } else if (ring_ok) {
        k_decode_ring<<<ring_ctas, 32 * (kRingWarps + 1), ring_smem, st>>>(p, base, rc, tmap);
      } else if (vec4) {
        dim3 grid((anchors / 4 + 63) / 64, n);
        k_decode_cm<4><<<grid, 64, 0, st>>>(p, base);
      } else {
        dim3 grid((anchors + 63) / 64, n);
        k_decode_cm<1><<<grid, 64, 0, st>>>(p, base);
      }
    } else {
      dim3 grid((anchors + 7) / 8, n);
      k_decode_am<<<grid, 256, 0, st>>>(p, base);
    }
    LAUNCH_CHECK(h);
    }
    // b200va_tick, schedule 1: the letterbox on the caller's stream starts when the (HBM-bound) decode is done
    if (h->hook_after_decode && base + n >= batch) {
      CUDA_TRY(h, cudaEventRecord(h->hook_after_decode, st));
      h->hook_recorded = true;
    }
    // schedule 3 of b200va_tick (single launch group only): the rest of the post-process moves to the tail stream
    cudaStream_t decode_st = st;
    const bool split_streams = h->post_tail_stream && h->hook_recorded && base == 0 && n == batch;
    if (split_streams) {
      CUDA_TRY(h, cudaStreamWaitEvent(h->post_tail_stream, h->hook_after_decode, 0));
      st = h->post_tail_stream;
    }
    (void)decode_st;

    NmsParams q;
    memset(&q, 0, sizeof(q));
    q.cand_key = p.cand_key;
    q.cand_box = p.cand_box;
    q.cand_cls = p.cand_cls;
    q.cand_count = p.cand_count;
    q.flags = h->status_flags;
    q.out_box = out->bbox_xyxy + (size_t)base * h->cfg.max_dets * 4;
    q.out_conf = out->conf + (size_t)base * h->cfg.max_dets;
    q.out_cls = out->cls + (size_t)base * h->cfg.max_dets;
    q.out_count = out->count + base;
    q.max_cand = h->cfg.max_candidates;
    q.max_dets = h->cfg.max_dets;
    q.cap_pow2 = next_pow2(h->cfg.max_candidates);
    q.iou_thr = (float)iou_thr;  // detector.py:373 compares float32 IoUs with the weak Python scalar
    q.filter_thr = filter_conf_thr_f64;
    q.use_filter = use_filter;
    q.class_aware = nms_mode == B200VA_NMS_CLASS_AWARE;
    q.dbg = h->dbg;
    q.dbg_reps = getenv("B200VA_DBG_REPS") ? atoi(getenv("B200VA_DBG_REPS")) : 1;
    q.ultra = ultra ? 1 : 0;
    q.ultra_agnostic = ultra ? ultra->agnostic : 0;
    q.max_det_cap = ultra ? ultra->max_det : 0;
    q.grid_off = (int)nms_grid_offset(h->cfg.max_candidates);
    q.skip = h->skip_dev ? h->skip_dev + base : nullptr;
    q.iou_thr64 = iou_thr;  // torchvision's CPU kernel compares the float32 IoU with the double threshold
    memcpy(q.f, p.f, sizeof(q.f));
    // dense scenes (more than 256 candidates in some frame of the previous launch) take the grid variant; the
    // statistic is a host-mapped word that dense frames overwrite with a posted store: no synchronisation, at worst
    // one launch late (both variants give identical results)
    q.stats = h->nms_stats_dev;
    bool dense = false;
    if (h->nms_stats_host) {
      // the host runs several launches ahead of the GPU, so one sighting keeps the grid variant for the next 64 launches
      cudaStreamCaptureStatus cap = cudaStreamCaptureStatusNone;
      cudaStreamIsCapturing(st, &cap);
      if (*(volatile int*)h->nms_stats_host > 256) {
        h->nms_dense_ttl = 64;
        if (cap == cudaStreamCaptureStatusNone) *(volatile int*)h->nms_stats_host = 0;
      }
      dense = h->nms_dense_ttl > 0;
      if (dense && cap == cudaStreamCaptureStatusNone) --h->nms_dense_ttl;
    }
    if (h->tune.dense_impl == 2 && h->dense_nms) dense = true;  // tests: every launch takes the dense-scene kernels
    if (defer) {
      // stash the chain: the next b200va_tick launches it beside its own decode and letterbox
      PendingChain* pc = (PendingChain*)h->pending_chain;
      if (!pc) h->pending_chain = pc = new PendingChain();
      pc->q = q;
      pc->n = n;
      pc->has_trk = false;
      if (fuse->stream_slots && fuse->cfg && fuse->batch == batch) {
        memset(&pc->t, 0, sizeof(pc->t));
        pc->t.f_box = out->bbox_xyxy;
        pc->t.f_conf = out->conf;
        pc->t.d_cls = out->cls;
        pc->t.d_count = out->count;
        pc->t.max_dets = fuse->max_dets;
        const int rc = tracker_fill_params(h, pc->t, fuse->stream_slots, fuse->batch, fuse->det_scale, fuse->skip, fuse->cfg,
                                           fuse->id_base, fuse->out, fuse->new_counts);
        if (rc != B200VA_OK) return rc;
        pc->has_trk = true;
        fuse->done = true;  // the tracker update is owed together with the NMS
      }
      h->cand_set ^= 1;
      return B200VA_OK;
    }
    PhaseScope phase(h, B200VA_PHASE_NMS, st);
    const size_t nms_smem = nms_smem_bytes(h->cfg.max_candidates);
    const bool pdl = h->tune.pdl != 0 && !split_streams;  // across streams the event carries the dependency
    // sparse scene, one launch group, detection rows = this handle's tables: NMS + tracker in one 256-thread CTA
    // (the tracker's working table gets tracker_pick_smem_tracks rows of shared memory, 512 in a sparse scene: the CTA
    // leaves most of its SM to the letterbox CTAs it runs beside)
    const bool fusable = fuse && fuse->stream_slots && fuse->cfg && !dense && h->tune.fuse_post_track != 0 && base == 0 &&
                         n == batch && fuse->batch == batch && fuse->max_dets == h->cfg.max_dets;
    const int trk_rows = fusable ? tracker_pick_smem_tracks(h, st) : 0;
    const size_t nms_plain = nms_base_bytes(h->cfg.max_candidates);  // the variants without the kept-box grid
    const size_t fused_smem = std::max(nms_plain, tracker_smem_bytes(trk_rows));
    if (fusable && fused_smem <= 200 * 1024) {
      TrkParams t;
      memset(&t, 0, sizeof(t));
      t.f_box = out->bbox_xyxy;
      t.f_conf = out->conf;
      t.d_cls = out->cls;
      t.d_count = out->count;
      t.max_dets = fuse->max_dets;
      const int rc = tracker_fill_params(h, t, fuse->stream_slots, fuse->batch, fuse->det_scale, fuse->skip, fuse->cfg,
                                         fuse->id_base, fuse->out, fuse->new_counts);
      if (rc != B200VA_OK) return rc;
      t.smem_tracks = trk_rows;
      if (q.ultra) CUDA_TRY(h, launch_pdl(k_post_track<true>, dim3(n), dim3(kNmsThreadsSmall), fused_smem, st, pdl, q, t));
      else CUDA_TRY(h, launch_pdl(k_post_track<false>, dim3(n), dim3(kNmsThreadsSmall), fused_smem, st, pdl, q, t));
      fuse->done = true;
    } else if (dense && h->dense_nms) {
      const DenseNms& D = *(const DenseNms*)h->dense_nms;
      CUDA_TRY(h, launch_pdl(k_dense_pairs, dim3(D.ctas), dim3(kPairThreads), 0, st, pdl, q, D, n));
      h->launches.fetch_add(1, std::memory_order_relaxed);
      // the tracker update of the same rows rides in the resolving CTA when the call carries one
      const bool fuse_trk = fuse && fuse->stream_slots && fuse->cfg && h->tune.fuse_post_track != 0 && base == 0 && n == batch &&
                            fuse->batch == batch && fuse->max_dets == h->cfg.max_dets;
      const int rows = fuse_trk ? tracker_pick_smem_tracks(h, st) : 0;
      const size_t both = std::max(dense_resolve_smem(D.max_cand), tracker_smem_bytes(rows));
      if (fuse_trk && both <= 200 * 1024) {
        TrkParams t;
        memset(&t, 0, sizeof(t));
        t.f_box = out->bbox_xyxy;
        t.f_conf = out->conf;
        t.d_cls = out->cls;
        t.d_count = out->count;
        t.max_dets = fuse->max_dets;
        const int rc = tracker_fill_params(h, t, fuse->stream_slots, fuse->batch, fuse->det_scale, fuse->skip, fuse->cfg,
                                           fuse->id_base, fuse->out, fuse->new_counts);
        if (rc != B200VA_OK) return rc;
        t.smem_tracks = rows;
        CUDA_TRY(h, launch_pdl(k_dense_resolve_track, dim3(n), dim3(kResolveThreads), both, st, h->tune.pdl != 0, q, D, t));
        fuse->done = true;
      } else {
        CUDA_TRY(h, launch_pdl(k_dense_resolve, dim3(n), dim3(kResolveThreads), dense_resolve_smem(D.max_cand), st, h->tune.pdl != 0, q, D));
      }
    } else if (dense && q.grid_off) {
      CUDA_TRY(h, launch_pdl(k_sort_nms<true>, dim3(n), dim3(kNmsThreads), nms_smem, st, pdl, q));
    } else {
      CUDA_TRY(h, launch_pdl(k_sort_nms<false>, dim3(n), dim3(kNmsThreads), nms_plain, st, pdl, q));
    }
    LAUNCH_CHECK(h);
    if (fuse) fuse->tail_on_side = split_streams;
  }
  return B200VA_OK;
}

extern "C" int b200va_postprocess(b200va_handle h, const void* head, int layout, int batch, int channels, int anchors,
                                  const b200va_letterbox* meta, double conf_thr, double iou_thr,
                                  const int32_t* classes, int n_classes, int score_mode, int nms_mode,
                                  double filter_conf_thr_f64, int use_filter, const b200va_dets* out, void* stream) {
  return postprocess_impl(h, head, layout, batch, channels, anchors, meta, conf_thr, iou_thr, classes, n_classes, score_mode,
                          nms_mode, filter_conf_thr_f64, use_filter, out, stream, nullptr);
}

extern "C" int b200va_postprocess_ultralytics(b200va_handle h, const void* head, int layout, int batch, int channels,
                                              int anchors, const int* src_h, const int* src_w, int in_h, int in_w,
                                              double conf_thr, double iou_thr, const int32_t* classes, int n_classes,
                                              int agnostic, int max_det, double filter_conf_thr_f64, int use_filter,
                                              const b200va_dets* out, void* stream) {
  const UltraOpts u{src_h, src_w, in_h, in_w, agnostic ? 1 : 0, max_det};
  return postprocess_impl(h, head, layout, batch, channels, anchors, nullptr, conf_thr, iou_thr, classes, n_classes,
                          B200VA_SCORE_V8_NATIVE, B200VA_NMS_AGNOSTIC, filter_conf_thr_f64, use_filter, out, stream, &u);
}

// schedule 4: launch the NMS (+ tracker) a previous tick's decode left behind, on `stream`
int postprocess_run_pending(b200va_handle h, void* stream) {
  PendingChain* pc = (PendingChain*)h->pending_chain;
  if (!pc || pc->n == 0) return B200VA_OK;
  cudaStream_t st = (cudaStream_t)stream;
  const int n = pc->n;
  pc->n = 0;
  bool dense = false;
  if (h->nms_stats_host) {
    cudaStreamCaptureStatus cap = cudaStreamCaptureStatusNone;
    cudaStreamIsCapturing(st, &cap);
    if (*(volatile int*)h->nms_stats_host > 256) {
      h->nms_dense_ttl = 64;
      if (cap == cudaStreamCaptureStatusNone) *(volatile int*)h->nms_stats_host = 0;
    }
    dense = h->nms_dense_ttl > 0;
    if (dense && cap == cudaStreamCaptureStatusNone) --h->nms_dense_ttl;
  }
  if (h->tune.dense_impl == 2 && h->dense_nms) dense = true;
  const size_t nms_smem = nms_smem_bytes(h->cfg.max_candidates);
  const bool fusable = pc->has_trk && !dense && h->tune.fuse_post_track != 0 && pc->t.max_dets == h->cfg.max_dets;
  const int trk_rows = fusable ? tracker_pick_smem_tracks(h, st) : 0;
  const size_t nms_plain = nms_base_bytes(h->cfg.max_candidates);
  const size_t fused_smem = std::max(nms_plain, tracker_smem_bytes(trk_rows));
  {
    PhaseScope phase(h, B200VA_PHASE_NMS, st);
    if (fusable && fused_smem <= 200 * 1024) {
      pc->t.smem_tracks = trk_rows;
      if (pc->q.ultra) CUDA_TRY(h, launch_pdl(k_post_track<true>, dim3(n), dim3(kNmsThreadsSmall), fused_smem, st, false, pc->q, pc->t));
      else CUDA_TRY(h, launch_pdl(k_post_track<false>, dim3(n), dim3(kNmsThreadsSmall), fused_smem, st, false, pc->q, pc->t));
      LAUNCH_CHECK(h);
      return B200VA_OK;
    }
    if (dense && h->dense_nms) {
      const DenseNms& D = *(const DenseNms*)h->dense_nms;
      CUDA_TRY(h, launch_pdl(k_dense_pairs, dim3(D.ctas), dim3(kPairThreads), 0, st, false, pc->q, D, n));
      h->launches.fetch_add(1, std::memory_order_relaxed);
      const bool fuse_trk = pc->has_trk && h->tune.fuse_post_track != 0 && pc->t.max_dets == h->cfg.max_dets;
      const int rows = fuse_trk ? tracker_pick_smem_tracks(h, st) : 0;
      const size_t both = std::max(dense_resolve_smem(D.max_cand), tracker_smem_bytes(rows));
      if (fuse_trk && both <= 200 * 1024) {
        pc->t.smem_tracks = rows;
        CUDA_TRY(h, launch_pdl(k_dense_resolve_track, dim3(n), dim3(kResolveThreads), both, st, h->tune.pdl != 0, pc->q, D, pc->t));
        LAUNCH_CHECK(h);
        return B200VA_OK;
      }
      CUDA_TRY(h, launch_pdl(k_dense_resolve, dim3(n), dim3(kResolveThreads), dense_resolve_smem(D.max_cand), st, h->tune.pdl != 0, pc->q, D));
    } else if (dense && pc->q.grid_off) CUDA_TRY(h, launch_pdl(k_sort_nms<true>, dim3(n), dim3(kNmsThreads), nms_smem, st, false, pc->q));
    else CUDA_TRY(h, launch_pdl(k_sort_nms<false>, dim3(n), dim3(kNmsThreads), nms_plain, st, false, pc->q));
    LAUNCH_CHECK(h);
  }
  if (pc->has_trk) return tracker_launch_params(h, pc->t, n, st);
  return B200VA_OK;
}

bool postprocess_has_pending(b200va_handle h) {
  const PendingChain* pc = (const PendingChain*)h->pending_chain;
  return pc && pc->n > 0;
}

void postprocess_release(b200va_ctx* h) {
  delete (PendingChain*)h->pending_chain;
  h->pending_chain = nullptr;
  if (DenseNms* D = (DenseNms*)h->dense_nms) {
    if (D->nbr_cnt) cudaFree(D->nbr_cnt);
    if (D->nbr) cudaFree(D->nbr);
    if (D->work) cudaFree(D->work);
    delete D;
    h->dense_nms = nullptr;
  }
}

// b200va_tick: post-process followed by the tracker update of the same rows; *fused tells the caller whether the
// tracker already ran inside the post-process's second kernel.
int postprocess_then_track(b200va_handle h, const b200va_tick_args* a, void* stream, bool* fused, bool* tail_on_side, bool defer) {
  FuseReq f{a->stream_slots, a->trk_batch, a->max_dets, a->det_scale, a->skip, a->trk_cfg, a->id_base, a->tracks, a->new_counts, false, false, defer};
  const bool want = a->stream_slots != nullptr && a->trk_batch > 0 && a->trk_batch == a->head_batch && a->trk_cfg != nullptr;
  const int rc = postprocess_impl(h, a->head, a->layout, a->head_batch, a->channels, a->anchors, a->meta, a->conf_thr, a->iou_thr,
                                  a->classes, a->n_classes, a->score_mode, a->nms_mode, a->filter_conf_thr_f64, a->use_filter,
                                  a->dets, stream, nullptr, &f);
  *fused = f.done;
  *tail_on_side = f.tail_on_side;
  (void)want;
  return rc;
}