// The per-stream body of the IoU tracker (tracker.py:50-126 restated for one CTA), shared by k_tracker (tracker.cu)
// and the fused post-process + tracker kernel (postprocess.cu).  See tracker.cu for the algorithm notes.
#pragma once
#include <type_traits>
#include "common.cuh"

struct TrackerState {
  // ping-pong buffers, each [max_streams, max_tracks]
  long long* id[2];
  int32_t* cls[2];
  double* conf[2];
  double* box[2];  // [.., 4]
  int32_t* age[2];
  int32_t* hits[2];
  uint8_t* touched;   // [max_streams, max_tracks]
  int32_t* count;     // [max_streams]
  int32_t* cur;       // [max_streams] current buffer index
  long long* next_id; // shared counter
  uint32_t* ticket;   // last-CTA election
  int32_t* new_count; // [max_batch] scratch
  int32_t* need_max;  // largest table a stream of the running launch needed (live tracks + detections)
  uint8_t* scratch;   // [max_batch][scratch_stride]: the working table of a stream that does not fit the launch's shared memory
  size_t scratch_stride;
  void* base = nullptr;
};

struct TrkParams {
  TrackerState st;
  int slots[B200VA_MAX_BATCH];
  double det_scale[B200VA_MAX_BATCH];
  long long id_base[B200VA_MAX_BATCH];
  uint8_t skip[B200VA_MAX_BATCH];
  const uint8_t* skip_dev;  // device-side gates: [batch] flags decided on the device (b200va_set_skip_mask), OR-ed with skip[]
  int max_threads;          // 0: the whole CTA; else the widest a stream's update runs (the surplus warps leave at once)
  // detections (one of the two sources)
  const float* f_box;
  const float* f_conf;
  const double* d_box;
  const double* d_conf;
  const int32_t* d_cls;
  const int32_t* d_count;
  int max_dets, max_tracks, batch;
  int max_age, min_hits;
  double thr;
  int has_id_base, has_scale;
  // outputs (optional)
  long long* o_id;
  int32_t* o_cls;
  double* o_conf;
  double* o_box;
  int32_t* o_age;
  int32_t* o_hits;
  int32_t* o_count;
  int32_t* o_new;
  int o_rows;  // rows per stream of the output arrays
  int32_t* flags;
  long long* dbg;
  // The working table (boxes, classes, hits, claims, last detection, overlap keys: 62 bytes per track) of a stream lives in shared
  // memory when `live tracks + detections <= smem_tracks`, in the stream's global scratch otherwise (same code, exact,
  // slower).  The launch sizes its dynamic shared memory for smem_tracks, not for max_tracks: a CTA that asks for
  // 188 KB closes its SM to the letterbox CTAs it runs beside in b200va_tick (measured: 32 x 1080p letterbox 36 us
  // alone, 41.5 us beside 32 such CTAs).  The host picks smem_tracks from what earlier launches needed (`stats`).
  int smem_tracks;
  int* stats;  // host-mapped words (b200va_ctx::nms_stats_dev): [1] = largest need of the last launch, posted by its last CTA
};

namespace {


// Python's builtin min / max on two floats: the first argument unless the second compares strictly below / above it.
// So a NaN second argument gives the first, a NaN first argument gives NaN (fmin / fmax return the non-NaN operand
// either way).  The tracker calls them with the track's coordinate first (tracker.py:129-147): a NaN coordinate of the
// detection is replaced by the track's in the intersection, a NaN coordinate of the track makes the intersection 0.
__device__ __forceinline__ double py_min(double a, double b) { return b < a ? b : a; }
__device__ __forceinline__ double py_max(double a, double b) { return b > a ? b : a; }
__device__ __forceinline__ double py_relu(double x) { return x > 0.0 ? x : 0.0; }  // max(0.0, x)

// tracker.py:129-147, IEEE double, no contraction; a = the track, b = the detection.
__device__ __forceinline__ double iou64(double ax1, double ay1, double ax2, double ay2, double bx1, double by1,
                                        double bx2, double by2) {
  const double iw = py_relu(__dsub_rn(py_min(ax2, bx2), py_max(ax1, bx1)));
  const double ih = py_relu(__dsub_rn(py_min(ay2, by2), py_max(ay1, by1)));
  const double inter = __dmul_rn(iw, ih);
  const double area_a = __dmul_rn(py_relu(__dsub_rn(ax2, ax1)), py_relu(__dsub_rn(ay2, ay1)));
  const double area_b = __dmul_rn(py_relu(__dsub_rn(bx2, bx1)), py_relu(__dsub_rn(by2, by1)));
  const double uni = __dsub_rn(__dadd_rn(area_a, area_b), inter);
  if (uni <= 0.0) return 0.0;
  return __ddiv_rn(inter, uni);
}

// launched; a stream with few detections and tracks keeps only kTrkThreadsMin of them.  512 by default, not 1024: a 1024-thread
// CTA owns the whole register file of its SM until it retires, and in b200va_tick the tracker runs underneath the
// letterbox -- 32 SMs closed to letterbox CTAs for 14 us cost the 32 x 1080p tick 3 us (dense tracker: 84 us at 512, 63 at 1024)
constexpr int kTrkThreadsMax = 1024;   // widest launch (dense scenes, see tracker_launch)
constexpr int kTrkThreadsWide = 512;   // default launch width
constexpr int kTrkThreadsMin = 256;
constexpr int kDetChunk = 64;  // detections staged in shared memory at a time (two warps cover a chunk)
constexpr int kTrkPairs = 2048;  // phase A, few pairs: capacity of the overlapping-pair list (= the most pairs that path takes)
constexpr int kCand = 6;        // candidate slots per detection and kind; more -> exact brute-force scan

struct DetStage {
  double4 box[kDetChunk];
  double conf[kDetChunk];
  int cls[kDetChunk];
};
struct Cand {
  double iou;
  int idx;  // track index (c_trk) or chunk-local detection index (c_det)
  int pad_;
};

// One detection into the chunk staging area, converted the way the tracker consumes it (float32 rows of the
// post-process: exact widening, then StreamWorker._rescale_detections' float64 multiply, pipeline.py:224-240).
__device__ __forceinline__ void stage_detection(DetStage& sd, int i, float4 f4, float conf, int cls, double scale, bool has_scale) {
  double4 b = make_double4(f4.x, f4.y, f4.z, f4.w);
  if (has_scale) {
    b.x = __dmul_rn(b.x, scale);
    b.y = __dmul_rn(b.y, scale);
    b.z = __dmul_rn(b.z, scale);
    b.w = __dmul_rn(b.w, scale);
  }
  sd.box[i] = b;
  sd.conf[i] = (double)conf;
  sd.cls[i] = cls;
}

// Boxes whose intersection is empty have IoU 0, which can never beat best_iou = 0.0 (tracker.py:100-106).
// A cheap superset of overlaps(): the same eight comparisons on order-preserving integer keys of the doubles' HIGH
// words (x > y implies key(x) >= key(y), whatever the signs), as `>=`.  It may pass pairs that do not overlap (their
// IoU then comes out as 0 and is discarded like before) but never rejects one that does.  Non-finite coordinates:
// a NaN of the DETECTION does not empty the intersection (iou64 puts the track's coordinate in its place), so the
// detection's keys (det_keys) give a NaN or infinite lower coordinate (x1, y1) key 0 and an upper one (x2, y2) key
// 0xFFFFFFFF, which pass every comparison.  A NaN of the TRACK makes the IoU 0 whatever the detection is, so the
// track's keys (box_keys) are the plain hi_key and may reject such a pair arbitrarily.  Integer compares instead of a
// chain of eight dependent float64 compares: the pre-filter runs once per (detection, track) pair on the
// latency-bound path.
__device__ __forceinline__ uint32_t hi_key(double v) {
  const int hi = __double2hiint(v);
  return (uint32_t)hi ^ ((uint32_t)(hi >> 31) | 0x80000000u);
}
__device__ __forceinline__ uint32_t nonfinite_mask(double v) {
  return ((uint32_t)__double2hiint(v) & 0x7ff00000u) == 0x7ff00000u ? 0xffffffffu : 0u;
}
__device__ __forceinline__ uint32_t lower_key(double v) { return hi_key(v) & ~nonfinite_mask(v); }
__device__ __forceinline__ uint32_t upper_key(double v) { return hi_key(v) | nonfinite_mask(v); }
__device__ __forceinline__ bool may_overlap(const double4 a, const double4 b) {
  const uint32_t ax = hi_key(a.x), ay = hi_key(a.y), az = hi_key(a.z), aw = hi_key(a.w);
  const uint32_t bx = lower_key(b.x), by = lower_key(b.y), bz = upper_key(b.z), bw = upper_key(b.w);
  return (az >= bx) & (bz >= ax) & (az >= ax) & (bz >= bx) & (aw >= by) & (bw >= ay) & (aw >= ay) & (bw >= by);
}

// Row bytes of a stream's working table: box 32, class 4, hits 4, claims 4, last detection 2, overlap keys 16.
constexpr int kTrkRowBytes = 62;
// The last detection of a row is an int16_t index into the frame's detections, so a call takes at most this many
// detection rows per stream (b200va_tracker_update[_f64] refuse more; the tick's rows are max_dets <= 8192).
constexpr int kTrkMaxDets = 32768;
// The overlap keys of a row: hi_key of (x1, y1, x2, y2), 16 bytes (det_keys for the chunk's detections).  Phase A of
// a dense stream tests every (detection, track) pair; reading the track's four doubles for that costs 8 shared-memory
// wavefronts per warp step (32-byte lane stride) and eight float64 compares, the keys cost 4 wavefronts and four
// integer compares -- and only a pair that passes them (a superset of the overlapping ones, see may_overlap) looks at
// the doubles.
__device__ __forceinline__ uint4 box_keys(const double4 b) {
  return make_uint4(hi_key(b.x), hi_key(b.y), hi_key(b.z), hi_key(b.w));
}
__device__ __forceinline__ uint4 det_keys(const double4 b) {
  return make_uint4(lower_key(b.x), lower_key(b.y), upper_key(b.z), upper_key(b.w));
}
__device__ __forceinline__ uint4* trk_key_table(uint8_t* tab, int cap) {
  return reinterpret_cast<uint4*>(tab + (((size_t)cap * 46 + kDetChunk * 4 + 15) & ~(size_t)15));
}

// The intersection of track (or earlier detection) `a` and detection `b` is not empty.  The terms with a coordinate of
// `b` are negated comparisons, so a NaN there passes them (see iou64); a NaN of `a` fails `a.z > a.x` or `a.w > a.y`.
__device__ __forceinline__ bool overlaps(const double4 a, const double4 b) {
  return !(b.x >= a.z) & !(a.x >= b.z) & (a.z > a.x) & !(b.x >= b.z) & !(b.y >= a.w) & !(a.y >= b.w) & (a.w > a.y) &
         !(b.y >= b.w);
}

// Best track for one detection among tracks t = first, first + stride, ... (tracker.py:97-109).
__device__ __forceinline__ void scan_tracks(const double* __restrict__ sbox, const int32_t* __restrict__ scls, int T,
                                            int first, int stride, const double4 db, int dcls, double thr,
                                            double& best, int& best_t) {
  best = 0.0;  // best_iou starts at 0.0 and must be beaten strictly
  best_t = 0x7fffffff;
  for (int t = first; t < T; t += stride) {
    if (scls[t] != dcls) continue;
    const double4 tb = reinterpret_cast<const double4*>(sbox)[t];
    if (!overlaps(tb, db)) continue;
    const double v = iou64(tb.x, tb.y, tb.z, tb.w, db.x, db.y, db.z, db.w);
    if (v >= thr && v > best) {
      best = v;
      best_t = t;
    }
  }
}

__device__ __forceinline__ void warp_argmax(double& best, int& best_t) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) {
    const double ob = __shfl_xor_sync(0xffffffffu, best, o);
    const int ot = __shfl_xor_sync(0xffffffffu, best_t, o);
    if (ob > best || (ob == best && ot < best_t)) {  // ties: earliest-inserted track
      best = ob;
      best_t = ot;
    }
  }
}

// The matching is sequential in the reference, but every IoU it can ever ask for within one chunk of
// detections is known up front: detection i against a track as it stood at the start of the chunk,
// or against an earlier detection of the chunk (a matched or new track carries exactly that box).
//
//   phase A   all threads: those float64 IoUs; per detection keep the few that pass the threshold
//             (c_trk: vs tracks, c_det: vs earlier detections) and count how many detections claim
//             each track.
//   phase A2  a thread per detection: a detection is SIMPLE when it has no detection-detection edge
//             and every track it could match is claimed by it alone -- nothing another detection does
//             can change its outcome, so it is resolved right away (arg-max over its own list).
//   phase B   one warp walks the remaining CONFLICTED detections in order, look-ups only:
//             aux[key] = last conflicted detection that took the track `key`; a track created by
//             detection j of the chunk has the virtual key Tc + j until phase C numbers it.
//   phase C   all threads: number the new tracks in detection order (prefix sum), add the hits, and
//             let the last detection matched to each track write its box.
//   A chunk in which some detection has more than kCand candidates falls back to the plain
//   sequential scan (exact, slower).  Nothing in the sequential parts touches global memory:
//   confidence, age and id of a touched track are derived from last_det[] at write-back.
// TAB_GLOBAL only tells the two instantiations apart: `tab` is shared memory in one and global memory in the other, and
// the compiler specialises the loads and stores of each inlined copy from the pointer's provenance.
struct TrkShared {
  DetStage sd;
  Cand c_trk[kDetChunk][kCand], c_det[kDetChunk][kCand];
  int n_trk[kDetChunk], n_det[kDetChunk], key[kDetChunk], conflicted[kDetChunk], clist[kDetChunk];
  int s_T, s_new, s_is_last, s_fallback, s_nconf;
  int n_plist;      // phase A, few pairs: number of listed (overlapping, same class) pairs
  uint32_t plist[kTrkPairs];  // idx | detection << 16 | (vs track) << 31
  uint4 dkey[kDetChunk];      // phase A, many pairs: overlap keys of the chunk's detections (det_keys)
  int s_prestaged;  // fused kernel: detections of this frame (count) whose first chunk the NMS half left in `sd`; -1 = none
  int wsum[kTrkThreadsMax / 32];
  int warp_cnt[kTrkThreadsMax / 32];
  int s_base;
  int f_new[B200VA_MAX_BATCH], f_cur[B200VA_MAX_BATCH], f_cnt[B200VA_MAX_BATCH], f_pre[B200VA_MAX_BATCH];
  long long f_next;
};

// A crowded chunk (some detection with more than kCand candidates): the plain sequential scan of the live table by
// one warp, exact (tracker.py:50-109).  Not inlined: rare, and its code would otherwise sit in the middle of the
// instruction stream every ordinary chunk runs through.
__device__ __forceinline__ void chunk_fallback_scan_body(const TrkParams& p, TrkShared& sh, double* sbox, uint4* skey, int32_t* scls, int32_t* shits,
                                                         int16_t* last_det, const int d0, const int nd) {
  DetStage& sd = sh.sd;
  int& s_T = sh.s_T;
  int& s_new = sh.s_new;
  const int lane = threadIdx.x & 31;
  {
        for (int i = 0; i < nd; ++i) {
          const int T = s_T;
          const int dcls = sd.cls[i];
          double best;
          int best_t;
          scan_tracks(sbox, scls, T, lane, 32, sd.box[i], dcls, p.thr, best, best_t);
          const unsigned cand = __ballot_sync(0xffffffffu, best_t != 0x7fffffff);
          int match = 0x7fffffff;
          if (cand) {
            warp_argmax(best, best_t);
            match = best_t;
          }
          if (lane == 0) {
            int t = match;
            if (t == 0x7fffffff) {
              t = T;
              if (t < p.max_tracks) {
                scls[t] = dcls;
                shits[t] = 1;
                s_new = s_new + 1;
                s_T = T + 1;
              } else {
                atomicOr(p.flags + FLAG_TRACK_OVERFLOW, 1);
                t = -1;
              }
            } else {
              shits[t] += 1;
            }
            if (t >= 0) {
              last_det[t] = (int16_t)(d0 + i);
              reinterpret_cast<double4*>(sbox)[t] = sd.box[i];
              skey[t] = box_keys(sd.box[i]);
            }
          }
          __syncwarp();
        }
      }
}

__device__ __noinline__ void chunk_fallback_scan(const TrkParams& p, TrkShared& sh, double* sbox, uint4* skey, int32_t* scls, int32_t* shits,
                                                 int16_t* last_det, const int d0, const int nd) {
  chunk_fallback_scan_body(p, sh, sbox, skey, scls, shits, last_det, d0, nd);
}

// What the prune step needs of a stream's first rows (row = threadIdx.x), fetched while the table is staged: its
// loads would otherwise start a global round trip at the very end of the critical path.
struct TablePrefetch {
  int age;
  long long id;
  double conf;
};

// Copy the live rows of a stream's table (buffer `cur`, T0 rows) into the working table at `tab` (capacity `cap` rows).
__device__ __forceinline__ TablePrefetch stage_table(const TrkParams& p, const int slot, const int cur, const int T0,
                                                     uint8_t* const tab, const int cap, const int nthreads) {
  double* sbox = reinterpret_cast<double*>(tab);
  int32_t* scls = reinterpret_cast<int32_t*>(sbox + (size_t)cap * 4);
  int32_t* shits = scls + cap;
  int16_t* last_det = reinterpret_cast<int16_t*>(shits + cap + cap + kDetChunk);
  uint4* skey = trk_key_table(tab, cap);
  const TrackerState& S = p.st;
  const size_t sb = (size_t)slot * p.max_tracks;
  const int tid = threadIdx.x;
  TablePrefetch pf{0, 0, 0.0};
  if (tid < T0) {
    pf.age = S.age[cur][sb + tid];
    pf.id = S.id[cur][sb + tid];
    pf.conf = S.conf[cur][sb + tid];
  }
  for (int t = tid; t < T0; t += nthreads) {
    const double4 b = reinterpret_cast<const double4*>(S.box[cur] + sb * 4)[t];
    reinterpret_cast<double4*>(sbox)[t] = b;
    skey[t] = box_keys(b);
    scls[t] = S.cls[cur][sb + t];
    shits[t] = S.hits[cur][sb + t];
    last_det[t] = -1;
  }
  return pf;
}

template <bool TAB_GLOBAL, bool SMALL>
__device__ __forceinline__ void tracker_stream_impl(const TrkParams& p, const int bi, uint8_t* const tab, const int cap,
                                                    TrkShared& sh, const int D, const bool prestaged, const int cur,
                                                    const int T0, const TablePrefetch* const staged_table = nullptr) {
  double* sbox = reinterpret_cast<double*>(tab);                           // [cap][4]
  int32_t* scls = reinterpret_cast<int32_t*>(sbox + (size_t)cap * 4);      // [cap]
  int32_t* shits = scls + cap;                                             // [cap]
  int32_t* aux = shits + cap;                                              // [cap + kDetChunk] claims, then phase-B state
  int16_t* last_det = reinterpret_cast<int16_t*>(aux + cap + kDetChunk);   // [cap] detection holding the track's box now, -1 untouched
  uint4* skey = trk_key_table(tab, cap);                                   // [cap] overlap keys of sbox (kept in step with it)
  // one set of statically allocated shared variables for both instantiations (declared by tracker_stream)
  DetStage& sd = sh.sd;
  auto& c_trk = sh.c_trk;
  auto& c_det = sh.c_det;
  auto& n_trk = sh.n_trk;
  auto& n_det = sh.n_det;
  auto& key = sh.key;
  auto& conflicted = sh.conflicted;
  auto& clist = sh.clist;
  int& s_T = sh.s_T;
  int& s_new = sh.s_new;
  int& s_is_last = sh.s_is_last;
  int& s_fallback = sh.s_fallback;
  int& s_nconf = sh.s_nconf;
  auto& wsum = sh.wsum;
  auto& warp_cnt = sh.warp_cnt;
  int& s_base = sh.s_base;
  auto& f_new = sh.f_new;
  auto& f_cur = sh.f_cur;
  auto& f_cnt = sh.f_cnt;
  auto& f_pre = sh.f_pre;
  long long& f_next = sh.f_next;

  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  PHASE_STAMP(p.dbg, 0);
  const int slot = p.slots[bi];
  const TrackerState& S = p.st;
  const size_t sb = (size_t)slot * p.max_tracks;
  long long* id_c = S.id[cur] + sb;
  int32_t* cls_c = S.cls[cur] + sb;
  double* conf_c = S.conf[cur] + sb;
  double* box_c = S.box[cur] + sb * 4;
  int32_t* age_c = S.age[cur] + sb;
  int32_t* hits_c = S.hits[cur] + sb;
  // phase A is bound by dependent shared-memory latency on one SM and scales with the warp count (dense config,
  // 313 detections x 365 tracks: 131 us with 256 threads, 84 us with 512, 63 us with 1024), while a small stream
  // (25 x 25) only pays for the wider barriers (19 us with 256, 22 us with 1024): the surplus warps of a small
  // stream leave at once (a barrier counts the warps that are still alive); see kTrkThreadsMax for the width launched
  // SMALL (one chunk, few pairs: what tracker_stream checks before it picks this instantiation) always runs 256 wide
  const int wide = p.max_threads > 0 ? min((int)blockDim.x, p.max_threads) : (int)blockDim.x;
  const int kTrkThreads = SMALL ? kTrkThreadsMin : ((T0 > 96 || D > 64) ? wide : kTrkThreadsMin);
  if (tid >= kTrkThreads) return;

  // (`staged_table`: the fused kernel copied the table into `tab` before it even waited for the decode kernel)
  const TablePrefetch pf = staged_table ? *staged_table : stage_table(p, slot, cur, T0, tab, cap, kTrkThreads);
  const int pf_age = pf.age;
  const long long pf_id = pf.id;
  const double pf_conf = pf.conf;
  if (tid == 0) {
    s_T = T0;
    s_new = 0;
  }

  const size_t db = (size_t)bi * p.max_dets;
  const double scale = p.det_scale[bi];

  PHASE_STAMP(p.dbg, 1);
  for (int d0 = 0; d0 < D; d0 += kDetChunk) {
    const int nd = min(kDetChunk, D - d0);
    if (d0) __syncthreads();  // previous chunk fully consumed
    const bool staged = prestaged && d0 == 0;  // fused kernel: the NMS half left the first chunk in `sd`
    for (int i = tid; i < nd; i += kTrkThreads) {
      const int d = d0 + i;
      if (staged) {
      } else if (p.f_box) {
        stage_detection(sd, i, reinterpret_cast<const float4*>(p.f_box)[db + d], p.f_conf[db + d], p.d_cls[db + d], scale,
                        p.has_scale != 0);
      } else {
        sd.box[i] = reinterpret_cast<const double4*>(p.d_box)[db + d];
        sd.conf[i] = p.d_conf[db + d];
        sd.cls[i] = p.d_cls[db + d];
      }
      n_trk[i] = 0;
      n_det[i] = 0;
    }
    if (tid == 0) {
      s_fallback = 0;
      s_nconf = 0;
      sh.n_plist = 0;
    }
    __syncthreads();
    PHASE_STAMP(p.dbg, 2);

    // ---- phase A: every IoU the chunk can need.  Warp w takes detections w, w+8, ..; lanes take tracks ----
    const int Tc = s_T;
    for (int t = tid; t < Tc + kDetChunk; t += kTrkThreads) aux[t] = 0;  // claims per track
    if (!SMALL && tid < nd) sh.dkey[tid] = det_keys(sd.box[tid]);
    __syncthreads();
    const int pairs_t = nd * Tc, pairs = pairs_t + nd * nd;
    static_assert(kTrkPairs >= 8 * kTrkThreadsMin, "the pair list must hold every pair of the small path");
    // one listed pair: the float64 IoU, and the candidate lists / claim counts it feeds
    auto score = [&](int i, int idx, bool vs_track) {
      const double4 bx = sd.box[i];
      const double4 ob = vs_track ? reinterpret_cast<const double4*>(sbox)[idx] : sd.box[idx];
      const double v = iou64(ob.x, ob.y, ob.z, ob.w, bx.x, bx.y, bx.z, bx.w);
      if (v >= p.thr && v > 0.0) {
        if (vs_track) {
          const int k = atomicAdd(&n_trk[i], 1);
          if (k < kCand) {
            c_trk[i][k].iou = v;
            c_trk[i][k].idx = idx;
          }
          atomicAdd(&aux[idx], 1);
        } else {
          const int k = atomicAdd(&n_det[i], 1);
          if (k < kCand) {
            c_det[i][k].iou = v;
            c_det[i][k].idx = idx;
          }
        }
      }
    };
    if (SMALL || pairs <= min(kTrkPairs, 8 * kTrkThreads)) {
      // Few pairs.  The CTA is latency-bound: a warp in which ONE lane meets an overlapping pair walks all 32 lanes
      // through the float64 IoU (a dependent chain of ~170 instructions), and the warp that owns a detection does
      // that once per 32 tracks and again for the earlier detections.  So pass 1 spreads ALL (detection, track) and
      // (detection, earlier detection) pairs over the threads and only lists those of equal class whose boxes overlap;
      // pass 2 evaluates one listed pair per thread, lanes converged (25 x 25: 5.6 k -> ~1.6 k SM cycles).  The
      // candidate lists come out in a different order, which nothing downstream depends on (arg-max with index ties).
      PHASE_STAMP(p.dbg, 58);
      const float inv_T = 1.0f / (float)max(Tc, 1), inv_n = 1.0f / (float)nd;
      // which of this thread's pairs q = tid + it * kTrkThreads are listed (at most 8 rounds: pairs <= 8 * kTrkThreads)
      auto unpack = [&](int q, int& i, int& idx) -> bool {
        const bool vs_track = q < pairs_t;
        const int r = vs_track ? q : q - pairs_t;
        i = (int)(((float)r + 0.5f) * (vs_track ? inv_T : inv_n));  // r / Tc, r / nd for these small integers
        idx = r - i * (vs_track ? Tc : nd);
        return vs_track;
      };
      unsigned cmask = 0u;
      {
        int it = 0;
#pragma unroll 1
        for (int q = tid; q < pairs; q += kTrkThreads, ++it) {
          int i, idx;
          if (unpack(q, i, idx)) {
            if (scls[idx] != sd.cls[i]) continue;
            if (!may_overlap(reinterpret_cast<const double4*>(sbox)[idx], sd.box[i])) continue;
          } else {
            if (idx >= i || sd.cls[idx] != sd.cls[i]) continue;
            if (!may_overlap(sd.box[idx], sd.box[i])) continue;
          }
          cmask |= 1u << it;
        }
      }
      // one list reservation per warp (exclusive prefix of the lanes' counts; lane 31 draws the block)
      {
        const int mine = __popc(cmask);
        int incl = mine;
#pragma unroll
        for (int o = 1; o < 32; o <<= 1) {
          const int v = __shfl_up_sync(0xffffffffu, incl, o);
          if (lane >= o) incl += v;
        }
        int base = 0;
        if (lane == 31 && incl > 0) base = atomicAdd(&sh.n_plist, incl);
        base = __shfl_sync(0xffffffffu, base, 31);
        int slot = base + incl - mine;
        while (cmask) {
          const int it = __ffs((int)cmask) - 1;
          cmask &= cmask - 1u;
          int i, idx;
          const bool vs_track = unpack(tid + it * kTrkThreads, i, idx);
          sh.plist[slot] = (uint32_t)idx | ((uint32_t)i << 16) | (vs_track ? 0x80000000u : 0u);  // (slot < pairs <= kTrkPairs)
          ++slot;
        }
      }
      PHASE_STAMP(p.dbg, 59);
      __syncthreads();
      PHASE_STAMP(p.dbg, 60);
      const int listed = sh.n_plist;
#pragma unroll 1
      for (int q = tid; q < listed; q += kTrkThreads) {
        const uint32_t e = sh.plist[q];
        score((int)((e >> 16) & 0x7fffu), (int)(e & 0xffffu), (e >> 31) != 0u);
      }
      PHASE_STAMP(p.dbg, 61);
    } else {
      // Many pairs (a dense stream).  Pass 1: warp w scans detections w, w + warps, ..: lanes over the tracks (integer
      // overlap keys first, see box_keys) and over the earlier detections of the chunk; a pair of equal class whose
      // boxes overlap is LISTED, not evaluated -- the float64 IoU is a dependent chain of ~170 instructions, and a warp
      // that meets such pairs in different steps of its scan would walk through it once per step.  Pass 2: one listed
      // pair per thread, all of them in flight together.  (Pairs past the end of the list are evaluated on the spot.)
      auto list_pair = [&](int i, int idx, bool vs_track) {
        const int slot = atomicAdd(&sh.n_plist, 1);
        if (slot < kTrkPairs) sh.plist[slot] = (uint32_t)idx | ((uint32_t)i << 16) | (vs_track ? 0x80000000u : 0u);
        else score(i, idx, vs_track);
      };
      PHASE_STAMP(p.dbg, 58);
      // A unit of pass 1 = 64 rows (lane l owns rows l and l + 32 of the block: keys and class in registers) x one
      // group of the chunk's detections, whose keys are broadcast from shared memory one by one (a 16-byte broadcast
      // occupies the shared-memory pipe for four cycles whatever the lanes do with it, hence two rows per lane).  The
      // rows are the live tracks followed by the chunk's own detections (row e of that block pairs with the later
      // detections i > e only).  The CTA is issue-bound on its one SM: a (row, detection) visit costs ~8 instructions
      // this way (ALU pipe, two cycles each), ~25 as a scan of the tracks per detection.
      const int nblk_t = (Tc + 63) >> 6, nblk = nblk_t + 1;
      const int G = nblk >= 16 ? 2 : (nblk >= 8 ? 4 : 8);  // detection groups: enough units for every warp
      // (the group size is a compile-time constant of the unit: the loop over its detections is unrolled, the bit a
      // visit sets is an immediate, and the five compares of a visit chain into one predicate)
      auto unit = [&](auto gs_c, const int u) {
        constexpr int GS = decltype(gs_c)::value;
        constexpr int kGroups = kDetChunk / GS;
        const int blk = u / kGroups, i0 = (u - blk * kGroups) * GS, i1 = min(nd, i0 + GS);
        if (i0 >= i1) return;
        const bool vs_track = blk < nblk_t;
        const int r0 = (vs_track ? blk * 64 : 0) + lane, r1 = r0 + 32;
        const int rows = vs_track ? Tc : nd;
        // (a row past the end gets keys that no finite box meets; a detection with non-finite coordinates can meet
        // them, since det_keys widens those, so the `r0 >= rows` masks below are what drops such rows)
        uint4 k0 = make_uint4(0xffffffffu, 0xffffffffu, 0u, 0u), k1 = k0;
        int c0 = 0, c1 = 0;
        if (r0 < rows) {
          k0 = vs_track ? skey[r0] : sh.dkey[r0];
          c0 = vs_track ? scls[r0] : sd.cls[r0];
        }
        if (r1 < rows) {
          k1 = vs_track ? skey[r1] : sh.dkey[r1];
          c1 = vs_track ? scls[r1] : sd.cls[r1];
        }
        uint32_t pass0 = 0u, pass1 = 0u;
#pragma unroll
        for (int b = 0; b < GS; ++b) {  // (entries past nd are stale; their bits are masked below)
          const uint4 dk = sh.dkey[i0 + b];
          const int dc = sd.cls[i0 + b];
          // same class, and the key intervals meet on both axes (cf. may_overlap)
          asm("{\n\t.reg .pred t;\n\t"
              "setp.eq.s32 t, %1, %2;\n\t"
              "setp.ge.and.u32 t, %3, %4, t;\n\t"
              "setp.ge.and.u32 t, %5, %6, t;\n\t"
              "setp.ge.and.u32 t, %7, %8, t;\n\t"
              "setp.ge.and.u32 t, %9, %10, t;\n\t"
              "@t or.b32 %0, %0, %11;\n\t}"
              : "+r"(pass0)
              : "r"(c0), "r"(dc), "r"(k0.z), "r"(dk.x), "r"(dk.z), "r"(k0.x), "r"(k0.w), "r"(dk.y), "r"(dk.w), "r"(k0.y), "r"(1u << b));
          asm("{\n\t.reg .pred t;\n\t"
              "setp.eq.s32 t, %1, %2;\n\t"
              "setp.ge.and.u32 t, %3, %4, t;\n\t"
              "setp.ge.and.u32 t, %5, %6, t;\n\t"
              "setp.ge.and.u32 t, %7, %8, t;\n\t"
              "setp.ge.and.u32 t, %9, %10, t;\n\t"
              "@t or.b32 %0, %0, %11;\n\t}"
              : "+r"(pass1)
              : "r"(c1), "r"(dc), "r"(k1.z), "r"(dk.x), "r"(dk.z), "r"(k1.x), "r"(k1.w), "r"(dk.y), "r"(dk.w), "r"(k1.y), "r"(1u << b));
        }
        const uint32_t in_chunk = i1 - i0 >= 32 ? 0xffffffffu : ((1u << (i1 - i0)) - 1u);
        pass0 &= in_chunk;
        pass1 &= in_chunk;
        if (!vs_track) {  // detection rows: only the detections after the row
          pass0 = r0 < i0 ? pass0 : (r0 - i0 >= 31 ? 0u : (pass0 & ~((2u << (r0 - i0)) - 1u)));
          pass1 = r1 < i0 ? pass1 : (r1 - i0 >= 31 ? 0u : (pass1 & ~((2u << (r1 - i0)) - 1u)));
        }
        if (r0 >= rows) pass0 = 0u;
        if (r1 >= rows) pass1 = 0u;
#pragma unroll
        for (int h = 0; h < 2; ++h) {
          uint32_t pass = h ? pass1 : pass0;
          const int r = h ? r1 : r0;
          while (pass) {
            const int i = i0 + __ffs((int)pass) - 1;
            pass &= pass - 1u;
            const double4 rb = vs_track ? reinterpret_cast<const double4*>(sbox)[r] : sd.box[r];
            if (overlaps(rb, sd.box[i])) list_pair(i, r, vs_track);
          }
        }
      };
      for (int u = warp; u < nblk * G; u += kTrkThreads / 32) {
        if (G == 2) unit(std::integral_constant<int, 32>{}, u);
        else if (G == 4) unit(std::integral_constant<int, 16>{}, u);
        else unit(std::integral_constant<int, 8>{}, u);
      }
      PHASE_STAMP(p.dbg, 59);
      __syncthreads();
      PHASE_STAMP(p.dbg, 60);
      const int listed = min(sh.n_plist, kTrkPairs);
#pragma unroll 1
      for (int q = tid; q < listed; q += kTrkThreads) {
        const uint32_t e = sh.plist[q];
        score((int)((e >> 16) & 0x7fffu), (int)(e & 0xffffu), (e >> 31) != 0u);
      }
      PHASE_STAMP(p.dbg, 61);
    }
    __syncthreads();

    PHASE_STAMP(p.dbg, 62);
    // ---- phase A2: classify; simple detections are resolved here ----
    {
      bool conf = false;
      if (tid < nd) {
        const int i = tid;
        const int nt = n_trk[i], ne = n_det[i];
        if (nt > kCand || ne > kCand) atomicOr(&s_fallback, 1);
        conf = ne > 0;
        double best = 0.0;
        int best_t = 0x7fffffff;
        for (int k = 0; k < min(nt, kCand); ++k) {
          const Cand c = c_trk[i][k];
          conf |= aux[c.idx] > 1;
          if (c.iou > best || (c.iou == best && c.idx < best_t)) {
            best = c.iou;
            best_t = c.idx;
          }
        }
        conflicted[i] = conf;
        key[i] = conf ? -1 : (best_t == 0x7fffffff ? Tc + i : best_t);
      }
      // ordered list of the conflicted detections (kDetChunk <= 64: two warps cover the chunk)
      const unsigned bal = __ballot_sync(0xffffffffu, conf);
      if (warp < 2 && lane == 0) wsum[warp] = __popc(bal);
      __syncthreads();
      if (tid < nd && conf) clist[(warp ? wsum[0] : 0) + __popc(bal & ((1u << lane) - 1u))] = tid;
      if (tid == 0) s_nconf = wsum[0] + (nd > 32 ? wsum[1] : 0);
      // phase-B state: aux[key] = last conflicted detection that took `key` (-1: none)
      __syncthreads();
      for (int t = tid; t < Tc + kDetChunk; t += kTrkThreads) aux[t] = -1;
      __syncthreads();
    }
    PHASE_STAMP(p.dbg, 7);

    if (s_fallback) {
      // ---- crowded chunk: plain sequential scan of the live table, exact (tracker.py:50-109) ----
      if (warp == 0) {
        if (SMALL) chunk_fallback_scan(p, sh, sbox, skey, scls, shits, last_det, d0, nd);
        else chunk_fallback_scan_body(p, sh, sbox, skey, scls, shits, last_det, d0, nd);
      }
    } else {
      // ---- phase B: conflicted detections, in order, look-ups only ----
      if (warp == 0) {
        const int nconf = s_nconf;
        for (int q = 0; q < nconf; ++q) {
          const int i = clist[q];
          const int nt = n_trk[i], ne = n_det[i];
          double best = 0.0;
          int best_t = 0x7fffffff;
          if (lane < nt) {
            const Cand c = c_trk[i][lane];
            if (aux[c.idx] < 0) {  // nobody re-boxed this track yet in the chunk
              best = c.iou;
              best_t = c.idx;
            }
          } else if (lane >= kCand && lane - kCand < ne) {
            const Cand c = c_det[i][lane - kCand];
            const int e = c.idx, k = key[e];  // the track detection e was given (k >= 0: e precedes i)
            // still carrying e's box: e was the last to take it (conflicted e), or nobody took it after a simple e
            if (k >= 0 && (conflicted[e] ? aux[k] == e : aux[k] < 0)) {
              best = c.iou;
              best_t = k;
            }
          }
          const unsigned cand = __ballot_sync(0xffffffffu, best_t != 0x7fffffff);
          int match = Tc + i;  // no match: new track (virtual key)
          if (cand) {
            if (cand & (cand - 1)) {
              warp_argmax(best, best_t);
              match = best_t;
            } else {
              match = __shfl_sync(0xffffffffu, best_t, __ffs(cand) - 1);
            }
          }
          if (lane == 0) {
            key[i] = match;
            aux[match] = i;
          }
          __syncwarp();
        }
      }
      __syncthreads();

      // ---- phase C: number the new tracks in detection order, count hits, write the final boxes ----
      {
        const int i = tid;
        const int k = i < nd ? key[i] : -1;
        const bool is_new = i < nd && k == Tc + i;
        const unsigned bal = __ballot_sync(0xffffffffu, is_new);
        if (warp < 2 && lane == 0) wsum[warp] = __popc(bal);
        __syncthreads();
        const int total_new = wsum[0] + (nd > 32 ? wsum[1] : 0);
        const int room = p.max_tracks - Tc;
        if (is_new) {
          const int rank = (warp ? wsum[0] : 0) + __popc(bal & ((1u << lane) - 1u));
          clist[i] = rank;  // clist is free again: rank of the track created by detection i
          if (rank < room) {
            scls[Tc + rank] = sd.cls[i];
            shits[Tc + rank] = 0;
            last_det[Tc + rank] = -1;
          }
        }
        __syncthreads();
        if (i < nd) {
          const int r = k < Tc ? k : Tc + clist[k - Tc];
          if (r < p.max_tracks) {
            atomicAdd(&shits[r], 1);
            // the last detection matched to a track leaves its box there
            const bool last = conflicted[i] ? aux[k] == i : aux[k] < 0;
            if (last) {
              last_det[r] = (int16_t)(d0 + i);
              reinterpret_cast<double4*>(sbox)[r] = sd.box[i];
              skey[r] = box_keys(sd.box[i]);
            }
          }
        }
        if (tid == 0) {
          const int made = min(total_new, room);
          if (total_new > room) atomicOr(p.flags + FLAG_TRACK_OVERFLOW, 1);
          s_new += made;
          s_T = Tc + made;
        }
      }
    }
  }
  __syncthreads();
  PHASE_STAMP(p.dbg, 3);

  // ---- prune + stable compaction into the other buffer (tracker.py:111-126) ----
  const int T = s_T;
  const int nxt = cur ^ 1;
  long long* id_n = S.id[nxt] + sb;
  int32_t* cls_n = S.cls[nxt] + sb;
  double* conf_n = S.conf[nxt] + sb;
  double* box_n = S.box[nxt] + sb * 4;
  int32_t* age_n = S.age[nxt] + sb;
  int32_t* hits_n = S.hits[nxt] + sb;
  const size_t ob = (size_t)bi * p.o_rows;
  if (tid == 0) s_base = 0;
  __syncthreads();
  int kept_total = 0;  // (thread 0) rows that survive; stays 0 for an empty table
  for (int t0 = 0; t0 < T; t0 += kTrkThreads) {
    const int t = t0 + tid;
    bool keep = false;
    int age = 0, hits = 0;
    int ld = -1;
    if (t < T) {
      ld = last_det[t];
      hits = shits[t];
      if (ld >= 0) {  // matched or created this frame: age = 0 (tracker.py:85)
        keep = true;
      } else {
        age = (t0 == 0 ? pf_age : age_c[t]) + 1;
        keep = !(age > p.max_age || hits < p.min_hits);
      }
    }
    const unsigned bal = __ballot_sync(0xffffffffu, keep);
    if (lane == 0) warp_cnt[warp] = __popc(bal);
    __syncthreads();
    int off = s_base;
    for (int w = 0; w < warp; ++w) off += warp_cnt[w];
    if (keep) {
      const int dst = off + __popc(bal & ((1u << lane) - 1u));
      // tracks appended this frame sit at t >= T0 in creation order: provisional id = -(ordinal + 1)
      const long long idv = t < T0 ? (t0 == 0 ? pf_id : id_c[t])
                                   : (p.has_id_base ? p.id_base[bi] + (t - T0) : -(long long)(t - T0 + 1));
      double cf;
      if (ld < 0) cf = t0 == 0 ? pf_conf : conf_c[t];
      else if (p.f_box) cf = (double)p.f_conf[db + ld];
      else cf = p.d_conf[db + ld];
      const double4 b = reinterpret_cast<const double4*>(sbox)[t];
      id_n[dst] = idv;
      cls_n[dst] = scls[t];
      conf_n[dst] = cf;
      reinterpret_cast<double4*>(box_n)[dst] = b;
      age_n[dst] = age;
      hits_n[dst] = hits;
      if (p.o_id && dst < p.o_rows) {
        p.o_id[ob + dst] = idv;
        p.o_cls[ob + dst] = scls[t];
        p.o_conf[ob + dst] = cf;
        reinterpret_cast<double4*>(p.o_box)[ob + dst] = b;
        p.o_age[ob + dst] = age;
        p.o_hits[ob + dst] = hits;
      }
    }
    if (t0 + kTrkThreads >= T) {  // last round (the only one of a small table): no further barrier needed
      if (tid == 0) {
        int tot = s_base;
        for (int w = 0; w < kTrkThreads / 32; ++w) tot += warp_cnt[w];
        kept_total = tot;
      }
      break;
    }
    __syncthreads();
    if (tid == 0) {
      int tot = 0;
      for (int w = 0; w < kTrkThreads / 32; ++w) tot += warp_cnt[w];
      s_base += tot;
    }
    __syncthreads();
  }
  if (tid == 0) {
    S.count[slot] = kept_total;
    S.cur[slot] = nxt;
    S.new_count[bi] = s_new;
    if (p.o_count) p.o_count[bi] = kept_total;
    if (p.o_id && kept_total > p.o_rows) atomicOr(p.flags + FLAG_TRACK_ROWS, 1);
    if (p.o_new) p.o_new[bi] = s_new;
  }

  // ---- shared id counter: last CTA converts provisional ordinals to ids in batch order ----
  PHASE_STAMP(p.dbg, 4);
  if (p.has_id_base) return;
  __threadfence();
  __syncthreads();
  PHASE_STAMP(p.dbg, 5);
  if (tid == 0) {
    const unsigned tk = atomicAdd(S.ticket, 1u);
    s_is_last = (tk == (unsigned)p.batch - 1u);
  }
  __syncthreads();
  PHASE_STAMP(p.dbg, 6);
  if (!s_is_last) return;
  __threadfence();
  // every stream's new-track count, buffer index and length are fetched in parallel (one thread
  // per stream), prefix-summed in batch order, then only streams that created tracks are patched
  if (tid < p.batch) {
    const int sl = p.slots[tid];
    f_new[tid] = ((volatile int32_t*)S.new_count)[tid];
    f_cur[tid] = ((volatile int32_t*)S.cur)[sl];
    f_cnt[tid] = ((volatile int32_t*)S.count)[sl];
  }
  if (tid == kTrkThreads - 1) f_next = *((volatile long long*)S.next_id);
  __syncthreads();
  if (tid == 0) {
    int acc = 0;
    for (int i = 0; i < p.batch; ++i) {
      f_pre[i] = acc;
      acc += f_new[i];
    }
    *S.next_id = f_next + acc;
    *S.ticket = 0u;
    // every stream of the launch has posted its need by now: report the largest to the host (one posted write; it is
    // only a hint for the next launch's shared-memory size) and re-arm the device word
    const int need = *((volatile int32_t*)S.need_max);
    *S.need_max = 0;
    if (p.stats && (need > 256 || need > p.smem_tracks)) ((volatile int*)p.stats)[1] = need;
  }
  __syncthreads();
  const long long next = f_next;
  // a warp per stream: new tracks sit at the tail of the table (creation order)
  for (int i = warp; i < p.batch; i += kTrkThreads / 32) {
    const int nnew = f_new[i];
    if (nnew == 0) continue;
    const int sl = p.slots[i];
    long long* ids = S.id[f_cur[i]] + (size_t)sl * p.max_tracks;
    const int cnt = f_cnt[i];
    for (int t = lane; t < cnt; t += 32) {
      const long long v = ((volatile long long*)ids)[t];
      if (v < 0) {
        const long long real = next + f_pre[i] + (-v - 1);
        ids[t] = real;
        if (p.o_id && t < p.o_rows) p.o_id[(size_t)i * p.o_rows + t] = real;
      }
    }
  }
}


__device__ __noinline__ void tracker_stream_general(const TrkParams& p, const int bi, uint8_t* const smem_raw, TrkShared& sh,
                                                    const int D, const bool prestaged, const int cur, const int T0,
                                                    const int need) {
  if (need <= p.smem_tracks) tracker_stream_impl<false, false>(p, bi, smem_raw, p.smem_tracks, sh, D, prestaged, cur, T0);
  else tracker_stream_impl<true, false>(p, bi, p.st.scratch + (size_t)bi * p.st.scratch_stride, p.max_tracks, sh, D, prestaged, cur, T0);
}

// One stream's tracker update.  The table never grows past `live tracks + detections` within the call, so that sum
// decides (uniformly for the CTA) whether the working table fits the shared memory this launch was given.
// `prestaged` >= 0 (fused kernel only): the detection count of this frame, whose first chunk already sits in sh.sd.
// `pre_cur` / `pre_T0` >= 0: the slot's buffer index and track count, read by the caller ahead of time.
// HOT_SMALL (the fused sparse-scene kernel): the common small case runs a compact instantiation inline and everything
// else sits behind one call; otherwise (k_tracker, which the host launches on its own for dense scenes and for plain
// b200va_tracker_update calls) the general code is inlined as it always was.
template <bool HOT_SMALL>
__device__ __forceinline__ void tracker_stream(const TrkParams& p, const int bi, uint8_t* const smem_raw, TrkShared& sh,
                                               const int prestaged, const int pre_cur = -1, const int pre_T0 = -1,
                                               const TablePrefetch* const staged_table = nullptr,
                                               uint8_t* const staged_tab = nullptr, const int staged_cap = 0) {
  const int slot = p.slots[bi];
  const int cur = pre_cur >= 0 ? pre_cur : p.st.cur[slot];
  const int T0 = pre_T0 >= 0 ? pre_T0 : p.st.count[slot];
  const bool skipped = p.skip[bi] || (p.skip_dev && p.skip_dev[bi]);
  const int D = skipped ? 0 : (prestaged >= 0 ? prestaged : min(p.d_count[bi], p.max_dets));
  const int need = T0 + D;
  if (threadIdx.x == 0 && need > 256) atomicMax(p.st.need_max, need);
  // the common case -- the table fits shared memory, one chunk of detections, few pairs -- runs a compact
  // instantiation inline; everything else goes through one call to the general code, kept out of the hot
  // instruction stream (these CTAs stall on instruction fetch more than on anything else)
  if (!HOT_SMALL) {
    if (need <= p.smem_tracks) tracker_stream_impl<false, false>(p, bi, smem_raw, p.smem_tracks, sh, D, prestaged >= 0, cur, T0);
    else tracker_stream_impl<true, false>(p, bi, p.st.scratch + (size_t)bi * p.st.scratch_stride, p.max_tracks, sh, D, prestaged >= 0, cur, T0);
  } else if (staged_table && need <= staged_cap && D <= kDetChunk && D * (T0 + D) <= 8 * kTrkThreadsMin) {
    tracker_stream_impl<false, true>(p, bi, staged_tab, staged_cap, sh, D, prestaged >= 0, cur, T0, staged_table);
  } else if (need <= p.smem_tracks && D <= kDetChunk && D * (T0 + D) <= 8 * kTrkThreadsMin) {
    tracker_stream_impl<false, true>(p, bi, smem_raw, p.smem_tracks, sh, D, prestaged >= 0, cur, T0);
  } else {
    tracker_stream_general(p, bi, smem_raw, sh, D, prestaged >= 0, cur, T0, need);
  }
}

}  // namespace

// shared-memory bytes tracker_stream needs for a working table of `tracks` rows
inline size_t tracker_smem_bytes(int tracks) { return (size_t)tracks * kTrkRowBytes + kDetChunk * 4 + 32; }
// rows a shared-memory working table can have at most (190 KB of dynamic shared memory); bigger streams use the global scratch
constexpr int kTrkSmemRowsMax = 3072;
// rows of the shared-memory working table the next launch gets (host side, tracker.cu)
int tracker_pick_smem_tracks(b200va_ctx* h, cudaStream_t st);
// validates the host arguments of a tracker update and fills the launch parameters (tracker.cu)
int tracker_fill_params(b200va_ctx* h, TrkParams& p, const int* stream_slots, int batch, const double* det_scale,
                        const uint8_t* skip, const b200va_tracker_cfg* cfg, const int64_t* id_base,
                        const b200va_tracks* out, int32_t* new_counts);
int tracker_launch_params(b200va_ctx* h, const TrkParams& p, int batch, cudaStream_t st);
