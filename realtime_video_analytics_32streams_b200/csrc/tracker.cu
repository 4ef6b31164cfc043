// a8: the IoU tracker for a batch of streams, state resident in HBM.
//
// Replaces IouTracker.update (tracker.py:50-95), _match_detection (:97-109), _prune_tracks
// (:111-126) and _iou (:129-147).  The reference is sequential and order dependent: detections
// are matched one after another, a matched track's box is overwritten at once, a new track is
// matchable by later detections of the same frame, and ties go to the earliest-inserted track.
// One CTA owns one stream: detections are visited in order, and for each one all threads score
// the live tracks in parallel (float64, Python's operation order) followed by a block arg-max
// with the reference's tie rule.  Pruning is a stable block compaction into the slot's second
// buffer, which preserves dict insertion order.  Track ids come from one counter shared by all
// streams (tracker.py:47): CTAs hand out provisional ordinals and the last CTA to finish turns
// them into ids in batch order -- the order one shared IouTracker would have been called in.
#include "tracker_body.cuh"

namespace {

__global__ void __launch_bounds__(kTrkThreadsMax) k_tracker(const __grid_constant__ TrkParams p) {
  extern __shared__ __align__(16) uint8_t smem_raw[];
  __shared__ TrkShared sh;
  griddep_wait();  // launched as a programmatic dependent of the NMS kernel: everything above overlapped its tail
  tracker_stream<false>(p, blockIdx.x, smem_raw, sh, -1);
}

__global__ void k_tracker_reset(TrackerState S, int slot) {
  S.count[slot] = 0;
}
__global__ void k_tracker_set_next(TrackerState S, long long v) { *S.next_id = v; }

}  // namespace

int tracker_state_create(b200va_ctx* h) {
  TrackerState* S = new TrackerState();
  h->tracker = S;
  const size_t n = (size_t)h->cfg.max_streams * h->cfg.max_tracks;
  // one arena: 2 x (id 8 + cls 4 + conf 8 + box 32 + age 4 + hits 4) + touched 1, plus the small arrays
  size_t bytes = 0;
  auto take = [&](size_t b) {
    size_t o = bytes;
    bytes += (b + 255) & ~(size_t)255;
    return o;
  };
  size_t o_id[2], o_cls[2], o_conf[2], o_box[2], o_age[2], o_hits[2];
  for (int k = 0; k < 2; ++k) {
    o_box[k] = take(n * 32);
    o_id[k] = take(n * 8);
    o_conf[k] = take(n * 8);
    o_cls[k] = take(n * 4);
    o_age[k] = take(n * 4);
    o_hits[k] = take(n * 4);
  }
  size_t o_touched = take(n);
  size_t o_count = take((size_t)h->cfg.max_streams * 4);
  size_t o_cur = take((size_t)h->cfg.max_streams * 4);
  size_t o_next = take(8);
  size_t o_ticket = take(4);
  size_t o_new = take((size_t)B200VA_MAX_BATCH * 4);
  size_t o_need = take(4);
  const size_t scratch_stride = (tracker_smem_bytes(h->cfg.max_tracks) + 255) & ~(size_t)255;
  size_t o_scratch = take((size_t)std::min(h->cfg.max_batch, B200VA_MAX_BATCH) * scratch_stride);
  CUDA_TRY(h, cudaMalloc(&S->base, bytes));
  CUDA_TRY(h, cudaMemset(S->base, 0, bytes));
  uint8_t* b = (uint8_t*)S->base;
  for (int k = 0; k < 2; ++k) {
    S->box[k] = (double*)(b + o_box[k]);
    S->id[k] = (long long*)(b + o_id[k]);
    S->conf[k] = (double*)(b + o_conf[k]);
    S->cls[k] = (int32_t*)(b + o_cls[k]);
    S->age[k] = (int32_t*)(b + o_age[k]);
    S->hits[k] = (int32_t*)(b + o_hits[k]);
  }
  S->touched = b + o_touched;
  S->count = (int32_t*)(b + o_count);
  S->cur = (int32_t*)(b + o_cur);
  S->next_id = (long long*)(b + o_next);
  S->ticket = (uint32_t*)(b + o_ticket);
  S->new_count = (int32_t*)(b + o_new);
  S->need_max = (int32_t*)(b + o_need);
  S->scratch = b + o_scratch;
  S->scratch_stride = scratch_stride;
  const long long one = 1;  // itertools.count(1), tracker.py:47
  CUDA_TRY(h, cudaMemcpy(S->next_id, &one, 8, cudaMemcpyHostToDevice));
  if (h->cfg.max_tracks > 4096) return set_error(h, B200VA_ERR_INVALID, "max_tracks %d too large (<= 4096)", h->cfg.max_tracks);
  const size_t smem = tracker_smem_bytes(std::min(h->cfg.max_tracks, kTrkSmemRowsMax));
  CUDA_TRY(h, raise_dyn_smem(k_tracker, smem));
  if (h->tune.uniform_carveout) CUDA_TRY(h, prefer_max_shared(k_tracker));
  return B200VA_OK;
}

void tracker_state_destroy(b200va_ctx* h) {
  if (!h->tracker) return;
  if (h->tracker->base) cudaFree(h->tracker->base);
  delete h->tracker;
  h->tracker = nullptr;
}

int tracker_fill_params(b200va_ctx* h, TrkParams& p, const int* stream_slots, int batch, const double* det_scale,
                        const uint8_t* skip, const b200va_tracker_cfg* cfg, const int64_t* id_base,
                        const b200va_tracks* out, int32_t* new_counts) {
  REQUIRE(h, stream_slots && cfg, "NULL argument");
  REQUIRE(h, batch >= 0 && batch <= h->cfg.max_batch && batch <= B200VA_MAX_BATCH, "batch %d outside [0, %d]", batch, h->cfg.max_batch);
  uint8_t seen[4096 / 8] = {0};
  for (int i = 0; i < batch; ++i) {
    const int s = stream_slots[i];
    REQUIRE(h, s >= 0 && s < h->cfg.max_streams, "stream slot %d outside [0, %d)", s, h->cfg.max_streams);
    if (s < 4096) {
      REQUIRE(h, !(seen[s >> 3] & (1 << (s & 7))), "stream slot %d appears twice in one call", s);
      seen[s >> 3] |= 1 << (s & 7);
    }
    p.slots[i] = s;
    p.det_scale[i] = det_scale ? det_scale[i] : 1.0;
    p.id_base[i] = id_base ? id_base[i] : 0;
    p.skip[i] = skip ? skip[i] : 0;
  }
  p.st = *h->tracker;
  p.max_threads = h->tune.trk_max_threads;
  p.max_tracks = h->cfg.max_tracks;
  p.batch = batch;
  p.max_age = cfg->max_age;
  p.min_hits = cfg->min_hits;
  p.thr = cfg->max_iou_distance;
  p.has_id_base = id_base != nullptr;
  p.has_scale = det_scale != nullptr;
  if (out) {
    REQUIRE(h, out->track_id && out->cls && out->conf && out->bbox_xyxy && out->age && out->hits && out->count, "NULL output array");
    p.o_id = (long long*)out->track_id;
    p.o_cls = out->cls;
    p.o_conf = out->conf;
    p.o_box = out->bbox_xyxy;
    p.o_age = out->age;
    p.o_hits = out->hits;
    p.o_count = out->count;
    REQUIRE(h, out->rows >= 0 && out->rows <= h->cfg.max_tracks, "b200va_tracks.rows %d outside [0, max_tracks]", out->rows);
    p.o_rows = out->rows > 0 ? out->rows : h->cfg.max_tracks;
  }
  p.o_new = new_counts;
  p.flags = h->status_flags;
  p.dbg = h->dbg;
  p.stats = h->nms_stats_dev;
  p.skip_dev = h->skip_dev;
  return B200VA_OK;
}

// Rows of the shared-memory working table for the next tracker launch.  512 rows (24 KB) unless a recent launch
// reported a stream that needed more (TrkParams::stats, posted by the launch's last CTA): then twice that need, rounded
// up to 1024 / 2048 / max_tracks, for the next 64 launches.  A stream that still does not fit runs from its global
// scratch -- the choice only moves time, never results.  Under stream capture the size is frozen into the graph.
int tracker_pick_smem_tracks(b200va_ctx* h, cudaStream_t st) {
  const int cap = std::min(h->cfg.max_tracks, kTrkSmemRowsMax);  // (a stream that needs more rows works in the global scratch)
  if (h->tune.trk_smem_tracks > 0) return std::min(cap, h->tune.trk_smem_tracks);  // B200VA_TRK_SMEM_TRACKS (tests)
  if (h->nms_stats_host) {
    cudaStreamCaptureStatus capt = cudaStreamCaptureStatusNone;
    cudaStreamIsCapturing(st, &capt);
    const int need = ((volatile int*)h->nms_stats_host)[1];
    if (need > 0) {
      int rows = 512;
      while (rows < 2 * need && rows < cap) rows <<= 1;
      if (rows >= h->trk_rows || h->trk_rows_ttl <= 0) h->trk_rows = rows;
      h->trk_rows_ttl = 64;
      if (capt == cudaStreamCaptureStatusNone) ((volatile int*)h->nms_stats_host)[1] = 0;
    } else if (h->trk_rows_ttl > 0 && capt == cudaStreamCaptureStatusNone) {
      if (--h->trk_rows_ttl == 0) h->trk_rows = 512;
    }
  }
  return std::min(cap, std::max(h->trk_rows, 512));
}

static int tracker_launch(b200va_ctx* h, TrkParams& p, const int* stream_slots, int batch, const double* det_scale,
                          const uint8_t* skip, const b200va_tracker_cfg* cfg, const int64_t* id_base,
                          const b200va_tracks* out, int32_t* new_counts, cudaStream_t st) {
  const int rc = tracker_fill_params(h, p, stream_slots, batch, det_scale, skip, cfg, id_base, out, new_counts);
  if (rc != B200VA_OK || batch == 0) return rc;
  PhaseScope phase(h, B200VA_PHASE_TRACKER, st);
  // dense scenes (the post-process saw more than 256 candidates in a frame lately) are worth a CTA that owns its SM
  const int width = h->nms_dense_ttl > 0 ? kTrkThreadsMax : kTrkThreadsWide;
  p.smem_tracks = tracker_pick_smem_tracks(h, st);
  CUDA_TRY(h, launch_pdl(k_tracker, dim3(batch), dim3(width), tracker_smem_bytes(p.smem_tracks), st, h->tune.pdl != 0, p));
  LAUNCH_CHECK(h);
  return B200VA_OK;
}

// launch k_tracker for parameters filled earlier (schedule 4 of b200va_tick)
int tracker_launch_params(b200va_ctx* h, const TrkParams& p0, int batch, cudaStream_t st) {
  PhaseScope phase(h, B200VA_PHASE_TRACKER, st);
  const int width = h->nms_dense_ttl > 0 ? kTrkThreadsMax : kTrkThreadsWide;
  TrkParams p = p0;
  p.smem_tracks = tracker_pick_smem_tracks(h, st);
  CUDA_TRY(h, launch_pdl(k_tracker, dim3(batch), dim3(width), tracker_smem_bytes(p.smem_tracks), st, h->tune.pdl != 0, p));
  LAUNCH_CHECK(h);
  return B200VA_OK;
}

extern "C" int b200va_tracker_update(b200va_handle h, const int* stream_slots, int batch, const b200va_dets* dets,
                                     int max_dets, const double* det_scale, const uint8_t* skip,
                                     const b200va_tracker_cfg* cfg, const int64_t* id_base, const b200va_tracks* out,
                                     int32_t* new_counts, void* stream) {
  if (!h) return B200VA_ERR_INVALID;
  std::lock_guard<std::recursive_mutex> lock(h->mu);
  DeviceGuard guard(h->cfg.device);
  REQUIRE(h, dets && dets->bbox_xyxy && dets->conf && dets->cls && dets->count, "NULL detections");
  REQUIRE(h, max_dets > 0 && max_dets <= kTrkMaxDets, "max_dets %d outside [1, %d]", max_dets, kTrkMaxDets);
  TrkParams p;
  memset(&p, 0, sizeof(p));
  p.f_box = dets->bbox_xyxy;
  p.f_conf = dets->conf;
  p.d_cls = dets->cls;
  p.d_count = dets->count;
  p.max_dets = max_dets;
  return tracker_launch(h, p, stream_slots, batch, det_scale, skip, cfg, id_base, out, new_counts, (cudaStream_t)stream);
}

extern "C" int b200va_tracker_update_f64(b200va_handle h, const int* stream_slots, int batch, const b200va_dets64* dets,
                                         int max_dets, const uint8_t* skip, const b200va_tracker_cfg* cfg,
                                         const int64_t* id_base, const b200va_tracks* out, int32_t* new_counts,
                                         void* stream) {
  if (!h) return B200VA_ERR_INVALID;
  std::lock_guard<std::recursive_mutex> lock(h->mu);
  DeviceGuard guard(h->cfg.device);
  REQUIRE(h, dets && dets->bbox_xyxy && dets->conf && dets->cls && dets->count, "NULL detections");
  REQUIRE(h, max_dets > 0 && max_dets <= kTrkMaxDets, "max_dets %d outside [1, %d]", max_dets, kTrkMaxDets);
  TrkParams p;
  memset(&p, 0, sizeof(p));
  p.d_box = dets->bbox_xyxy;
  p.d_conf = dets->conf;
  p.d_cls = dets->cls;
  p.d_count = dets->count;
  p.max_dets = max_dets;
  return tracker_launch(h, p, stream_slots, batch, nullptr, skip, cfg, id_base, out, new_counts, (cudaStream_t)stream);
}

extern "C" int b200va_tracker_reset(b200va_handle h, int stream_slot, void* stream) {
  if (!h) return B200VA_ERR_INVALID;
  std::lock_guard<std::recursive_mutex> lock(h->mu);
  DeviceGuard guard(h->cfg.device);
  REQUIRE(h, stream_slot >= 0 && stream_slot < h->cfg.max_streams, "stream slot %d outside [0, %d)", stream_slot, h->cfg.max_streams);
  k_tracker_reset<<<1, 1, 0, (cudaStream_t)stream>>>(*h->tracker, stream_slot);
  LAUNCH_CHECK(h);
  return B200VA_OK;
}

extern "C" int b200va_tracker_set_next_id(b200va_handle h, int64_t next_id, void* stream) {
  if (!h) return B200VA_ERR_INVALID;
  std::lock_guard<std::recursive_mutex> lock(h->mu);
  DeviceGuard guard(h->cfg.device);
  k_tracker_set_next<<<1, 1, 0, (cudaStream_t)stream>>>(*h->tracker, (long long)next_id);
  LAUNCH_CHECK(h);
  return B200VA_OK;
}
