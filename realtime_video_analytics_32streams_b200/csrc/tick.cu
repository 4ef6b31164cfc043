// b200va_tick: the letterbox of the next detector batch and the post-process + tracker update of
// the last head tensor as two branches of one call (fork / join on events, capturable in a graph).
#include "common.cuh"

int postprocess_then_track(b200va_handle h, const b200va_tick_args* a, const UltraOpts* ultra, void* stream, bool* fused,
                           bool* tail_on_side, bool defer);            // postprocess.cu
int postprocess_run_pending(b200va_handle h, void* stream);            // postprocess.cu
bool postprocess_has_pending(b200va_handle h);                         // postprocess.cu

// The letterbox of one tick: BGR frames (a->frames) or, when `nv12` is given, NV12 frames; with the caller's geometry
// when `geom` is given (b200va_tick_ultralytics).
static int tick_letterbox(b200va_handle h, const b200va_tick_args* a, const b200va_nv12_frame* nv12,
                          const b200va_letterbox* geom, cudaStream_t st) {
  if (geom && nv12)
    return b200va_preprocess_geom_nv12(h, nv12, a->src_h, a->src_w, a->batch, a->roi_masks, geom, a->net_out, a->dst_h,
                                       a->dst_w, a->out_format, st);
  if (geom)
    return b200va_preprocess_geom(h, a->frames, a->src_h, a->src_w, a->src_pitch, a->batch, a->roi_masks, geom, a->net_out,
                                  a->dst_h, a->dst_w, a->out_format, st);
  if (nv12)
    return b200va_preprocess_nv12(h, nv12, a->src_h, a->src_w, a->batch, a->roi_masks, a->net_out, a->dst_h, a->dst_w,
                                  a->out_format, a->meta_out, st);
  return b200va_preprocess(h, a->frames, a->src_h, a->src_w, a->src_pitch, a->batch, a->roi_masks, a->net_out, a->dst_h,
                           a->dst_w, a->out_format, a->meta_out, st);
}

// ultra / geom: b200va_tick_ultralytics (NULL for b200va_tick*).
static int tick_impl(b200va_handle h, const b200va_tick_args* a, const b200va_nv12_frame* nv12, const UltraOpts* ultra,
                     const b200va_letterbox* geom, void* stream) {
  std::lock_guard<std::recursive_mutex> lock(h->mu);
  DeviceGuard guard(h->cfg.device);
  REQUIRE(h, a->schedule >= 0 && a->schedule <= 6, "unknown schedule %d", a->schedule);
  // schedule 6 (auto).  Large sparse batches take 3: the letterbox is the long pole, and launched as a programmatic
  // dependent of the decode kernel it fills the SMs as that drains (60.6 against 63.5 us on the 32 x 1080p tick).  Up to
  // ~16 streams the chain decode -> NMS + tracker is as long as the letterbox, and schedule 3 starts it 2-4 us later (it
  // moves to the second stream behind an event): 1 there (4 streams: 20.2 against 21.3 us, 1 stream: 15.3 against
  // 16.5).  Dense frames (the post-process saw more than 256 candidates lately) take 1 as well: the chain decode ->
  // pairs -> resolve + tracker is the tick, and letterbox CTAs launched early take SMs from k_dense_pairs (0.142
  // against 0.129 ms).
  const int schedule = a->schedule == 6 ? ((h->nms_dense_ttl > 0 || a->batch < 24) ? 1 : 3) : a->schedule;
  cudaStream_t main_st = (cudaStream_t)stream;
  const bool has_pre = (nv12 != nullptr || a->frames != nullptr) && a->batch > 0;
  const bool has_post = a->head != nullptr && a->head_batch > 0;
  const bool has_trk = a->stream_slots != nullptr && a->trk_batch > 0;
  // schedule 4, the software-pipelined tick: this call only DECODES its head; NMS + tracker of the head decoded by the
  // previous call run beside it (they share nothing with this call's decode and letterbox: two candidate sets).  The
  // latency-bound chain decode -> NMS -> tracker, which is what bounds schedules 1-3 (tools/timeline.py: 23 us of
  // decode, then 38 us of NMS + tracker slowed down by the letterbox CTAs they share SMs with), leaves the critical path.
  // Results lag one call: the tables of tick k are complete after call k + 1 (or a final call without a head).
  const bool sched4 = schedule == 4 && (!has_post || (a->head_batch <= B200VA_LAUNCH_FRAMES && a->channels >= 5 && a->anchors > 0));
  const bool pending = postprocess_has_pending(h);
  PhaseScope phase(h, B200VA_PHASE_TICK, main_st);
  int rc = B200VA_OK;
  auto note = [&](cudaError_t e, const char* what) {
    if (e != cudaSuccess && rc == B200VA_OK) rc = set_error(h, B200VA_ERR_CUDA, "%s failed: %s", what, cudaGetErrorString(e));
  };
  if (pending && !sched4) {
    // a caller that leaves schedule 4 still gets the chain it is owed, in stream order, before anything else
    rc = postprocess_run_pending(h, main_st);
    if (rc != B200VA_OK) return rc;
  }
  if (sched4) {
    const bool side = pending && (has_post || has_pre);
    if (side) {
      CUDA_TRY(h, cudaEventRecord(h->ev_fork, main_st));
      CUDA_TRY(h, cudaStreamWaitEvent(h->side_stream, h->ev_fork, 0));
    }
    // from here on the side stream may be forked: collect errors, always join
    if (pending) {
      const int r = postprocess_run_pending(h, side ? h->side_stream : main_st);
      if (rc == B200VA_OK) rc = r;
    }
    if (side) note(cudaEventRecord(h->ev_join, h->side_stream), "cudaEventRecord(join)");
    bool tracked = false, tail = false;
    if (rc == B200VA_OK && has_post) rc = postprocess_then_track(h, a, ultra, main_st, &tracked, &tail, true);
    if (rc == B200VA_OK && has_trk && !has_post)
      rc = b200va_tracker_update(h, a->stream_slots, a->trk_batch, a->dets, a->max_dets, a->det_scale, a->skip, a->trk_cfg,
                                 a->id_base, a->tracks, a->new_counts, main_st);
    if (rc == B200VA_OK && has_pre) {
      if (a->ev_pre_begin) note(cudaEventRecord((cudaEvent_t)a->ev_pre_begin, main_st), "cudaEventRecord(pre_begin)");
      if (rc == B200VA_OK) rc = tick_letterbox(h, a, nv12, geom, main_st);
      if (rc == B200VA_OK && a->ev_pre_end) note(cudaEventRecord((cudaEvent_t)a->ev_pre_end, main_st), "cudaEventRecord(pre_end)");
    }
    if (side) note(cudaStreamWaitEvent(main_st, h->ev_join, 0), "cudaStreamWaitEvent(join)");
    return rc;
  }

  const bool fork = schedule != 0 && has_pre && (has_post || has_trk);
  // schedule 3: the decode kernel stays on the caller's stream and the letterbox follows it there as a programmatic
  // dependent that never waits: its CTAs start as soon as SM resources allow (see prefer_max_shared in common.cuh for
  // why that is only the decode's tail today); NMS + tracker move to the side stream behind an event recorded right
  // after the decode.
  // schedule 5: the same launch, but the letterbox executes griddepcontrol.wait before its first load: the two HBM
  // kernels never share the bus (their mix is slower than their sequence, tools/membw.cu) and no launch latency
  // separates them.
  const bool sched3 = (schedule == 3 || schedule == 5) && fork && has_post && a->head_batch <= B200VA_LAUNCH_FRAMES;
  cudaStream_t post_st = (fork && !sched3) ? h->side_stream : main_st;
  if (fork && !sched3) {
    CUDA_TRY(h, cudaEventRecord(h->ev_fork, main_st));
    CUDA_TRY(h, cudaStreamWaitEvent(post_st, h->ev_fork, 0));
  }
  // From here on the side stream is forked: every path, errors included, must reach the join below (an unjoined
  // stream invalidates a CUDA-graph capture), so failures are collected in `rc` instead of returning early.
  bool tracked = false, tail_on_side = false;
  if (has_post) {
    h->hook_after_decode = (fork && (schedule == 1 || sched3)) ? h->ev_decoded : nullptr;
    h->hook_recorded = false;
    h->post_tail_stream = sched3 ? h->side_stream : nullptr;
    // sparse scenes: NMS and the tracker update of the same rows run as ONE kernel (k_post_track)
    rc = postprocess_then_track(h, a, ultra, post_st, &tracked, &tail_on_side, false);
    h->hook_after_decode = nullptr;
    h->post_tail_stream = nullptr;
    // the post-process reports whether it recorded the hook (it does not for empty or malformed heads)
    if (h->hook_recorded && !sched3) note(cudaStreamWaitEvent(main_st, h->ev_decoded, 0), "cudaStreamWaitEvent(decoded)");
    if (tail_on_side) post_st = h->side_stream;
  }
  if (rc == B200VA_OK && has_trk && !tracked)
    rc = b200va_tracker_update(h, a->stream_slots, a->trk_batch, a->dets, a->max_dets, a->det_scale, a->skip, a->trk_cfg,
                               a->id_base, a->tracks, a->new_counts, post_st);
  const bool joined = fork && post_st == h->side_stream;
  if (joined) note(cudaEventRecord(h->ev_join, post_st), "cudaEventRecord(join)");
  h->pdl_preprocess = sched3 && tail_on_side;
  h->pdl_preprocess_wait = schedule == 5;
  if (rc == B200VA_OK && has_pre) {
    if (a->ev_pre_begin) note(cudaEventRecord((cudaEvent_t)a->ev_pre_begin, main_st), "cudaEventRecord(pre_begin)");
    if (rc == B200VA_OK) rc = tick_letterbox(h, a, nv12, geom, main_st);
    if (rc == B200VA_OK && a->ev_pre_end) note(cudaEventRecord((cudaEvent_t)a->ev_pre_end, main_st), "cudaEventRecord(pre_end)");
  }
  h->pdl_preprocess = false;
  h->pdl_preprocess_wait = false;
  if (joined) note(cudaStreamWaitEvent(main_st, h->ev_join, 0), "cudaStreamWaitEvent(join)");
  return rc;
}

extern "C" int b200va_tick(b200va_handle h, const b200va_tick_args* a, void* stream) {
  if (!h || !a) return B200VA_ERR_INVALID;
  return tick_impl(h, a, nullptr, nullptr, nullptr, stream);
}

extern "C" int b200va_tick_nv12(b200va_handle h, const b200va_tick_args* a, const b200va_nv12_frame* frames, void* stream) {
  if (!h || !a) return B200VA_ERR_INVALID;
  if (!frames && a->batch > 0) {
    std::lock_guard<std::recursive_mutex> lock(h->mu);
    return set_error(h, B200VA_ERR_INVALID, "b200va_tick_nv12: NULL frames for a batch of %d", a->batch);
  }
  return tick_impl(h, a, frames, nullptr, nullptr, stream);
}

extern "C" int b200va_tick_ultralytics(b200va_handle h, const b200va_tick_args* a, const b200va_tick_ultra* u,
                                       const b200va_nv12_frame* frames, void* stream) {
  if (!h || !a || !u) return B200VA_ERR_INVALID;
  if (a->batch > 0 && (!u->geom || (!frames && !a->frames))) {
    std::lock_guard<std::recursive_mutex> lock(h->mu);
    return set_error(h, B200VA_ERR_INVALID, "b200va_tick_ultralytics: NULL frames or geometry for a batch of %d", a->batch);
  }
  const UltraOpts ultra{u->src_h, u->src_w, u->in_h, u->in_w, u->agnostic ? 1 : 0, u->max_det};
  return tick_impl(h, a, frames, &ultra, u->geom, stream);
}
