/*
 * b200va.h -- C ABI of the B200-native video-analytics hot path (libb200va.so).
 *
 * Drop-in boundary for the per-frame data-parallel path of
 * skygazer42/realtime-video-analytics-32streams.  Every entry point cites the reference
 * interface it replaces (paths relative to the reference root).  The reference is pure
 * Python; a maintainer binds these with ctypes (see INTEGRATION.md) behind the reference's
 * own classes/functions, so the YAML config keeps working.
 *
 * Conventions
 *   - extern "C", plain pointers and sizes only; no C++/torch types.
 *   - Pointers marked DEVICE point to CUDA device memory on the handle's device; pointers
 *     marked HOST are ordinary host memory read synchronously during the call (they are
 *     small per-frame descriptors, never pixel data).
 *   - `stream` is a cudaStream_t passed as void* (NULL = legacy default stream).  All work
 *     is enqueued asynchronously on it; nothing synchronises unless stated.
 *   - Return value: 0 = B200VA_OK, negative = error (b200va_error_string).  Nothing throws.
 *     b200va_last_error(handle) returns a detailed message for the last failing call.
 *   - No hidden device allocation after b200va_create(): all scratch and all tracker state
 *     are carved from arenas sized by b200va_config.
 *   - There is NO CPU fallback: every compute entry point launches sm_100a kernels.
 */
#ifndef B200VA_H_
#define B200VA_H_

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define B200VA_VERSION 200 /* 0.2.0 */

#if defined(__GNUC__)
#define B200VA_API __attribute__((visibility("default")))
#else
#define B200VA_API
#endif

enum b200va_status {
  B200VA_OK = 0,
  B200VA_ERR_INVALID = -1,  /* bad argument */
  B200VA_ERR_CUDA = -2,     /* a CUDA runtime call failed; see b200va_last_error */
  B200VA_ERR_CAPACITY = -3, /* a configured capacity (batch, candidates, tracks...) was exceeded */
  B200VA_ERR_STATE = -4     /* call order violated (e.g. pending track ids not assigned) */
};

/* Output tensor formats of b200va_preprocess. */
enum b200va_out_format {
  B200VA_OUT_F32_RGB_NCHW = 0, /* detector.py:245-257, half=False: float32, RGB planes, x*(1/255)        */
  B200VA_OUT_F16_RGB_NCHW = 1, /* detector.py:248-251, half=True : float16(x) * float16(1/255)           */
  B200VA_OUT_U8_BGR_NCHW = 2,  /* detector.py:777-839 RKNN variant, use_nhwc=False: letterboxed BGR uint8  */
  B200VA_OUT_U8_BGR_NHWC = 3   /* detector.py:777-839 RKNN variant, use_nhwc=True; also plain resize       */
};

/* OR-ed into out_format: the caller guarantees that the full-width pad rows of `out` (the 114-valued bands above
 * and below the resized image) still hold what an earlier call with the same geometry and format wrote there, so
 * the kernel does not write them again.  A letterboxed 16:9 frame in a 640 x 640 input is 44 % padding: with a
 * persistent network-input buffer (what a batched tick driver uses anyway) those 69 MB per 32 frames are written
 * once instead of every tick.  The tensor contents are identical either way. */
#define B200VA_OUT_FLAG_PADS_VALID 0x100

/* Head tensor layouts accepted by b200va_postprocess (detector.py:278-283 transposes
 * [C,A] exports to [A,C]; both are read in place here, no transpose pass). */
enum b200va_head_layout {
  B200VA_HEAD_CHANNEL_MAJOR = 0, /* [B, C, A]  e.g. YOLOv8 [B,84,8400]   */
  B200VA_HEAD_ANCHOR_MAJOR = 1   /* [B, A, C]  e.g. YOLOv5 [B,25200,85]  */
};

/* OR-ed into `layout` (b200va_postprocess, b200va_postprocess_ultralytics, b200va_tick_args.layout): the head is
 * IEEE binary16 in the same [B, C, A] / [B, A, C] layout, as a model exported for fp16 input returns it, and is
 * read in place -- half the bytes of the float32 head, and no conversion pass before the call.  Every element is
 * widened to float32 exactly where it is loaded (float16 -> float32 is exact, subnormals included) and all
 * arithmetic after that is the float32 code: the results are bit-for-bit those of the same call on the head
 * converted to float32.  An fp16 head never takes the TMA ring decode (B200VA_DECODE_IMPL=2 selects the register
 * kernels for it).  Any other bit in `layout` is refused with B200VA_ERR_INVALID. */
#define B200VA_HEAD_F16 0x200

/* Scoring rule.  REF_COMPAT is what detector.py:294-307 computes for BOTH model types:
 * C>5: score_k = head[5+k] * head[4];  C==5: score_0 = head[4]. */
enum b200va_score_mode {
  B200VA_SCORE_REF_COMPAT = 0, /* the reference's rule, bit-exact with detector.py:294-310                    */
  B200VA_SCORE_V8_NATIVE = 1   /* score_k = head[4+k]: what a YOLOv8 [84, A] export holds (additive mode)     */
};

/* NMS flavour.  The reference's _nms (detector.py:361-375) is class-agnostic; CLASS_AWARE is the
 * additive mode named by the north star: a kept box suppresses only boxes of its own class. */
enum b200va_nms_mode { B200VA_NMS_AGNOSTIC = 0, B200VA_NMS_CLASS_AWARE = 1 };

typedef struct b200va_ctx* b200va_handle;

typedef struct b200va_config {
  int device;         /* CUDA device ordinal                                                     */
  int max_batch;      /* frames per call (<= 128)                                                */
  int max_anchors;    /* A upper bound (8400 for 640x640 YOLOv8, 25200 for YOLOv5; <= 262144)    */
  int max_candidates; /* per-frame candidates surviving the confidence filter (<= 8192)          */
  int max_dets;       /* per-frame detections kept after NMS (output row capacity)               */
  int max_streams;    /* tracker stream slots (<= 4096)                                          */
  int max_tracks;     /* live tracks per stream slot (<= 4096)                                   */
} b200va_config;

/* Letterbox geometry, the `meta` dict of detector.py:259-263 plus the resized size. */
typedef struct b200va_letterbox {
  int src_h, src_w; /* meta["orig_shape"]                            */
  int new_h, new_w; /* int(h*scale), int(w*scale)  (detector.py:214) */
  int pad_left, pad_top; /* meta["pad"]                              */
  double scale;     /* meta["scale"] (float64)                       */
} b200va_letterbox;

/* Detections, structure-of-arrays, row-major [batch, max_dets].  DEVICE pointers.
 * Mirrors Detection(class_id, confidence, bbox_xyxy) of detector.py:32-40. */
typedef struct b200va_dets {
  float* bbox_xyxy; /* [B, max_dets, 4] float32 (frame pixels)  */
  float* conf;      /* [B, max_dets]                            */
  int32_t* cls;     /* [B, max_dets]                            */
  int32_t* count;   /* [B]                                      */
} b200va_dets;

/* Float64 detections for callers that hold Python-float Detection objects (tracker.py:50 takes
 * arbitrary doubles).  Same layout as b200va_dets with double boxes / confidences. */
typedef struct b200va_dets64 {
  const double* bbox_xyxy; /* [B, max_dets, 4] */
  const double* conf;      /* [B, max_dets]    */
  const int32_t* cls;      /* [B, max_dets]    */
  const int32_t* count;    /* [B]              */
} b200va_dets64;

/* Tracker parameters, TrackerConfig of config.py:194-209. */
typedef struct b200va_tracker_cfg {
  int max_age;
  int min_hits;
  double max_iou_distance;
} b200va_tracker_cfg;

/* Track rows, structure-of-arrays [batch, max_tracks].  DEVICE pointers.
 * Mirrors Track(track_id, class_id, confidence, bbox_xyxy, age, hits) of tracker.py:18-33. */
typedef struct b200va_tracks {
  int64_t* track_id; /* [B, max_tracks] */
  int32_t* cls;      /* [B, max_tracks] */
  double* conf;      /* [B, max_tracks] */
  double* bbox_xyxy; /* [B, max_tracks, 4] */
  int32_t* age;      /* [B, max_tracks] */
  int32_t* hits;     /* [B, max_tracks] */
  int32_t* count;    /* [B] */
  int32_t rows;      /* rows per stream of the arrays above; 0 = max_tracks.  A caller that copies the tables to the host
                      * every tick allocates fewer rows than the state can hold: `count` always reports the true number
                      * of tracks, rows beyond `rows` are not written and status word [3] is raised.  (New in 0.2.0:
                      * zero-initialise the struct.) */
} b200va_tracks;

/* ---- library ------------------------------------------------------------------------ */
B200VA_API int b200va_version(void);
B200VA_API const char* b200va_error_string(int status);
B200VA_API int b200va_create(const b200va_config* cfg, b200va_handle* out);
B200VA_API int b200va_destroy(b200va_handle h);
B200VA_API const char* b200va_last_error(b200va_handle h);
/* Number of kernels this handle has launched since creation (for launch accounting). */
B200VA_API int64_t b200va_launch_count(b200va_handle h);
/* Kernels never block on capacity problems; they raise device-side flags instead.  This call
 * synchronises `stream`, returns B200VA_ERR_CAPACITY (and clears the flags) if any frame since the
 * last poll exceeded max_candidates / max_dets / max_tracks (the surplus rows were dropped), else
 * B200VA_OK.  The reference has no such limits; size the config so that this never fires. */
B200VA_API int b200va_poll_status(b200va_handle h, void* stream);

/* Asynchronous form for callers that already copy results back every tick: enqueues a copy of the status words
 * (B200VA_STATUS_WORDS int32: [0] candidates > max_candidates, [1] detections > max_dets, [2] tracks > max_tracks,
 * [3] tracks > b200va_tracks.rows (state intact, output truncated), rest reserved) into host_out (HOST, pinned memory for a truly asynchronous copy) and, when clear != 0, resets them
 * on the device afterwards, all on `stream`; nothing synchronises.  The words are valid once the caller has
 * synchronised `stream` (e.g. with the event that guards its result tables). */
#define B200VA_STATUS_WORDS 8
B200VA_API int b200va_read_status_async(b200va_handle h, int32_t* host_out, int clear, void* stream);

/* ---- per-phase device times and NVTX ranges ------------------------------------------------
 * The reference times each packet on the host (`start = time.perf_counter()` ... `health.update_success(dt)`,
 * pipeline.py:145, 200-201).  With the work on the GPU the caller needs device times instead: after
 * b200va_set_profiling(h, 1) every entry point brackets its kernels with CUDA events (one pair per phase, on the
 * stream the kernels run on; skipped while the stream is being captured into a CUDA graph), and
 * b200va_get_phase_times waits for the pairs recorded since the last query and returns their durations in
 * milliseconds (ms[phase] = -1 when the phase did not run).  Independently of that switch every entry point
 * opens an NVTX range named "b200va:<phase>" around its launches (free when no tool is attached). */
enum b200va_phase {
  B200VA_PHASE_UPLOAD = 0,     /* b200va_upload_frames                                   */
  B200VA_PHASE_ROI = 1,        /* b200va_roi_rasterize / b200va_apply_mask               */
  B200VA_PHASE_RESIZE = 2,     /* b200va_resize_linear_u8                                */
  B200VA_PHASE_MOTION = 3,     /* b200va_motion / b200va_motion_preprocess               */
  B200VA_PHASE_PREPROCESS = 4, /* b200va_preprocess / b200va_preprocess_geom             */
  B200VA_PHASE_DECODE = 5,     /* head decode + confidence filter (b200va_postprocess*)  */
  B200VA_PHASE_NMS = 6,        /* sort + NMS + emit (b200va_postprocess*)                */
  B200VA_PHASE_TRACKER = 7,    /* b200va_tracker_update*                                 */
  B200VA_PHASE_DFL = 8,        /* b200va_dfl_decode                                      */
  B200VA_PHASE_TICK = 9,       /* the whole b200va_tick call, fork to join               */
  B200VA_PHASE_EGRESS = 10,    /* b200va_resize_area_u8 / b200va_draw_rects              */
  B200VA_PHASE_COUNT = 11
};
B200VA_API int b200va_set_profiling(b200va_handle h, int enable);
B200VA_API int b200va_get_phase_times(b200va_handle h, float* ms /* HOST [B200VA_PHASE_COUNT] */);

/* ---- a1: letterbox preprocess --------------------------------------------------------
 * Replaces _TensorRTBaseDetector._preprocess (detector.py:198-264) and
 * RKNNDetector._preprocess (detector.py:777-839) for a batch of frames.
 * Host-only geometry helper: fills `out` exactly like detector.py:209-230. */
B200VA_API int b200va_letterbox_meta(int src_h, int src_w, int dst_h, int dst_w, b200va_letterbox* out);

/* frames    HOST array [batch] of DEVICE pointers to BGR uint8 HWC frames
 * src_h/w   HOST [batch]; src_pitch HOST [batch] row pitch in bytes (>= 3*w)
 * roi_masks HOST array [batch] of DEVICE pointers to uint8 [src_h, src_w] masks (0 = outside),
 *           entries may be NULL; the array itself may be NULL.  Fuses apply_roi
 *           (frame_filter.py:43-50) into the resize taps.
 * out       DEVICE tensor [batch, 3, dst_h, dst_w] (NCHW formats) or [batch, dst_h, dst_w, 3]
 * meta_out  HOST [batch], may be NULL */
B200VA_API int b200va_preprocess(b200va_handle h, const uint8_t* const* frames, const int* src_h, const int* src_w,
                      const int64_t* src_pitch, int batch, const uint8_t* const* roi_masks, void* out,
                      int dst_h, int dst_w, int out_format, b200va_letterbox* meta_out, void* stream);

/* ---- host -> device staging of decoded frames -------------------------------------------
 * The reference hands host ndarrays to predict() (detector.py:193, pipeline.py:172-179); this is
 * the upload half of that call.  host_frames HOST array [batch] of HOST pointers (pinned memory
 * for asynchronous copies), dev_frames HOST array [batch] of DEVICE pointers to full-size frame
 * buffers, pitches in bytes (NULL = 3*w).  rows_mode 0 copies every row; rows_mode 1 copies only
 * the rows that b200va_preprocess to dst_h x dst_w reads (non-zero vertical tap weight), into
 * their original positions -- e.g. one row in three for 1080p -> 640x360 -- so the device frame
 * is valid for b200va_preprocess but NOT for b200va_motion / b200va_resize_linear_u8.
 * bytes_copied (HOST, may be NULL) receives the number of bytes put on the bus. */
B200VA_API int b200va_upload_frames(b200va_handle h, const uint8_t* const* host_frames, uint8_t* const* dev_frames,
                                    const int* src_h, const int* src_w, const int64_t* host_pitch,
                                    const int64_t* dev_pitch, int batch, int dst_h, int dst_w, int rows_mode,
                                    int64_t* bytes_copied, void* stream);

/* ---- a10: downsample -----------------------------------------------------------------
 * Replaces utils.downsample (frame_filter.py:53-57): cv2.resize INTER_LINEAR, BGR uint8 HWC in,
 * BGR uint8 HWC out (dst pitch = 3*dst_w).  dst HOST array [batch] of DEVICE pointers.
 * roi_masks as in b200va_preprocess (may be NULL): the reference applies the ROI to the full
 * frame BEFORE downsampling (pipeline.py:149-154), so the mask is fused into the taps here too. */
B200VA_API int b200va_resize_linear_u8(b200va_handle h, const uint8_t* const* frames, const int* src_h, const int* src_w,
                            const int64_t* src_pitch, int batch, const uint8_t* const* roi_masks,
                            uint8_t* const* dst, const int* dst_h, const int* dst_w, void* stream);

/* ---- NV12 frames (what video decoders produce) ---------------------------------------------
 * NVDEC / PyNvVideoCodec / DALI surfaces and FFmpeg's `-pix_fmt nv12` hold a frame as src_h rows of src_w luma bytes
 * and a separate plane of src_h / 2 rows of src_w bytes, the interleaved Cb, Cr pair of each 2 x 2 pixel block.  Each
 * plane has its own base and pitch (decoder surfaces keep the chroma plane at pitch * aligned_height).  The entry
 * points below take such frames directly, with the colour conversion folded into the letterbox / resize taps (no
 * conversion pass, no BGR frame in memory): every result is BYTE-IDENTICAL to the BGR entry point of the same name
 * run on cv2.cvtColor(frame, cv2.COLOR_YUV2BGR_NV12) -- OpenCV's BT.601 limited-range fixed point with nearest
 * chroma:  y' = max(0, Y - 16) * 1220542 + (1 << 19), u = Cb - 128, v = Cr - 128,
 *          R = sat_u8((y' + 1673527 v) >> 20), G = sat_u8((y' - 852492 v - 409993 u) >> 20), B = sat_u8((y' + 2116026 u) >> 20).
 * ROI masks are uint8 [src_h, src_w] (luma size); geometry, output formats, flags and the skip mask are those of the
 * BGR calls.  Odd src_h / src_w and NULL planes are refused with B200VA_ERR_INVALID.  The chroma plane is read at
 * row y >> 1 for luma row y; only NV12 (not I420, not BT.709, not full range) is accepted. */
typedef struct b200va_nv12_frame {
  const uint8_t* y;  /* DEVICE (HOST for the source side of b200va_upload_frames_nv12) luma plane [src_h, y_pitch]   */
  const uint8_t* uv; /* chroma plane [src_h / 2, uv_pitch]: Cb, Cr byte pairs                                        */
  int64_t y_pitch;   /* bytes between luma rows   (>= src_w) */
  int64_t uv_pitch;  /* bytes between chroma rows (>= src_w) */
} b200va_nv12_frame;

/* b200va_preprocess for NV12 frames.  frames: HOST array [batch] of plane descriptors (DEVICE planes); every other
 * argument as in b200va_preprocess. */
B200VA_API int b200va_preprocess_nv12(b200va_handle h, const b200va_nv12_frame* frames, const int* src_h, const int* src_w,
                                      int batch, const uint8_t* const* roi_masks, void* out, int dst_h, int dst_w,
                                      int out_format, b200va_letterbox* meta_out, void* stream);
/* b200va_resize_linear_u8 for NV12 frames: BGR uint8 HWC out (dst pitch = 3 * dst_w).  With dst == src size this is
 * cv2.cvtColor(frame, COLOR_YUV2BGR_NV12) itself (masked pixels zeroed when a mask is given). */
B200VA_API int b200va_resize_linear_u8_nv12(b200va_handle h, const b200va_nv12_frame* frames, const int* src_h,
                                            const int* src_w, int batch, const uint8_t* const* roi_masks,
                                            uint8_t* const* dst, const int* dst_h, const int* dst_w, void* stream);
/* b200va_resize_area_u8 (the 8f-3 preview downscale, below) for NV12 frames: BGR uint8 HWC out (dst pitch = 3 * dst_w),
 * byte-identical to cv2.resize(cv2.cvtColor(frame, COLOR_YUV2BGR_NV12), (dst_w, dst_h), interpolation=cv2.INTER_AREA);
 * every source pixel is converted and saturated before it is summed.  With dst == src size this is cv2.cvtColor itself.
 * Frames are grouped by (source, destination) size, at most 64 per launch, under B200VA_PHASE_EGRESS.  Shrinking only;
 * odd source sizes, NULL planes, plane pitches below src_w and enlarging are refused with B200VA_ERR_INVALID. */
B200VA_API int b200va_resize_area_u8_nv12(b200va_handle h, const b200va_nv12_frame* frames, const int* src_h,
                                          const int* src_w, int batch, uint8_t* const* dst, const int* dst_h,
                                          const int* dst_w, void* stream);
/* b200va_upload_frames for NV12 frames: host[i] (HOST planes, pinned for asynchronous copies) -> dev[i] (DEVICE
 * planes, written through the const pointers).  rows_mode 0 copies both planes whole; rows_mode 1 copies only the
 * luma rows b200va_preprocess_nv12 to dst_h x dst_w reads and the chroma rows those use (each once) -- e.g. 1,382,400
 * bytes of a 1080p frame for 640 x 640 instead of 3,110,400 -- and the device frame is then valid for the letterbox
 * only.  bytes_copied (HOST, may be NULL) receives the bytes put on the bus. */
B200VA_API int b200va_upload_frames_nv12(b200va_handle h, const b200va_nv12_frame* host, const b200va_nv12_frame* dev,
                                         const int* src_h, const int* src_w, int batch, int dst_h, int dst_w, int rows_mode,
                                         int64_t* bytes_copied, void* stream);

/* ---- a9: ROI polygons ----------------------------------------------------------------
 * Replaces the mask construction of utils.apply_roi (frame_filter.py:46-49): one cv2.fillPoly
 * per polygon (LINE_8, shift 0), union.  pts HOST [sum(poly_sizes), 2] int32 (x, y);
 * poly_sizes HOST [n_polys]; mask_out DEVICE uint8 [h, w] (255 inside, 0 outside). */
B200VA_API int b200va_roi_rasterize(b200va_handle h, const int32_t* pts, const int* poly_sizes, int n_polys, int height,
                         int width, uint8_t* mask_out, void* stream);
/* Replaces cv2.bitwise_and(frame, frame, mask=mask) (frame_filter.py:50): dst = mask ? src : 0. */
B200VA_API int b200va_apply_mask(b200va_handle h, const uint8_t* src, int64_t src_pitch, const uint8_t* mask, int height,
                      int width, uint8_t* dst, int64_t dst_pitch, void* stream);

/* ---- a11: motion filter --------------------------------------------------------------
 * Replaces MotionFilter.should_process (frame_filter.py:26-40) for a batch:
 * BGR2GRAY -> GaussianBlur 5x5 -> |new - prev| > 25 -> count; always stores the new blurred gray.
 * prev_gray    HOST array [batch] of DEVICE uint8 [h, w] state buffers (read, unless has_prev==0)
 * next_gray    HOST array [batch] of DEVICE uint8 [h, w] buffers receiving the new state
 *              (must differ from prev_gray[i]: the stencil reads neighbours)
 * has_prev     HOST [batch]; 0 = first frame of the stream (count is written as -1)
 * changed_out  DEVICE int32 [batch]: number of pixels with |diff| > 25
 * The caller decides `count / (h*w) >= threshold` in float64 (frame_filter.py:38-40). */
B200VA_API int b200va_motion(b200va_handle h, const uint8_t* const* frames, const int* src_h, const int* src_w,
                  const int64_t* src_pitch, int batch, const uint8_t* const* roi_masks,
                  const uint8_t* const* prev_gray, uint8_t* const* next_gray, const int* has_prev,
                  int32_t* changed_out, void* stream);

/* ---- a11 + a1 in one pass: motion gate and letterbox from the same staged rows ------------------
 * b200va_motion and b200va_preprocess (reference letterbox geometry) on the same frames in ONE pass over each
 * frame: the motion gate reads every pixel anyway, so the network input is interpolated from the rows it has
 * staged in shared memory instead of reading the tapped rows and their ROI-mask rows from HBM a second time.
 * Arguments as in b200va_motion followed by those of b200va_preprocess; out_format is
 * B200VA_OUT_F32_RGB_NCHW or B200VA_OUT_F16_RGB_NCHW (optionally | B200VA_OUT_FLAG_PADS_VALID).  Results are
 * identical to the two separate calls.  Frames the fused kernel cannot take (unaligned base / pitch, width
 * not a multiple of 16, up-scaling geometry) run through the two separate kernels inside this call.
 * The letterbox of a frame the motion gate then rejects is wasted work (4.9 MB of writes per frame). */
B200VA_API int b200va_motion_preprocess(b200va_handle h, const uint8_t* const* frames, const int* src_h, const int* src_w,
                                        const int64_t* src_pitch, int batch, const uint8_t* const* roi_masks,
                                        const uint8_t* const* prev_gray, uint8_t* const* next_gray, const int* has_prev,
                                        int32_t* changed_out, void* out, int dst_h, int dst_w, int out_format,
                                        b200va_letterbox* meta_out, void* stream);

/* ---- a3-a7: head post-process --------------------------------------------------------
 * Replaces _TensorRTBaseDetector._postprocess (detector.py:266-338), _xywh2xyxy (:352-359),
 * _scale_boxes (:340-350), _nms (:361-375) + _iou (:469-481), and folds in
 * filter_detections (detector.py:99-103, called at pipeline.py:182) when use_filter != 0:
 * kept boxes whose float64 confidence is below filter_conf_thr_f64 still suppress others but
 * are not emitted.
 * head       DEVICE float32 (float16 with B200VA_HEAD_F16 in `layout`), layout per `layout`; B frames, C channels,
 *            A anchors
 * meta       HOST [batch] letterbox geometry of each frame
 * conf_thr / iou_thr  the Python floats of DetectorConfig; rounded to float32 exactly where
 *            NumPy does (detector.py:312, :373)
 * classes    HOST int32 [n_classes] whitelist (detector.py:313-314) or NULL; ids below 0 or at or above the
 *            head's class count match nothing (np.isin); an id in [2048, class count) is refused with
 *            B200VA_ERR_INVALID (the kernels hold the whitelist as a 2048-bit map)
 * out        kept detections in keep order (score descending), at most max_dets per frame
 * Equal scores are ordered higher-candidate-index first (stable argsort reversed); -0.0 and +0.0 are
 * equal scores, and each detection keeps the sign of its own score. */
B200VA_API int b200va_postprocess(b200va_handle h, const void* head, int layout, int batch, int channels, int anchors,
                       const b200va_letterbox* meta, double conf_thr, double iou_thr, const int32_t* classes,
                       int n_classes, int score_mode, int nms_mode, double filter_conf_thr_f64, int use_filter,
                       const b200va_dets* out, void* stream);

/* ---- a14: DFL decode of a raw YOLOv8 Detect head --------------------------------------
 * Not part of /root/reference (its _postprocess consumes decoded tensors); restates the published
 * Ultralytics Detect decode so that a raw export can feed b200va_postprocess.  raw DEVICE float32
 * [batch, 4*reg_max + num_classes, A]; level_hw HOST [n_levels][2] grid sizes (80x80, 40x40, 20x20 at
 * 640x640), level_stride HOST [n_levels] (8, 16, 32); out DEVICE float32 [batch, 4 + num_classes, A]
 * with A = sum(h*w): rows 0-3 = (cx, cy, w, h) in input pixels, rows 4.. = sigmoid(class logits).
 * Floating point (exp), not bit-exact: every output is within a bound derived from the float32 operation
 * order of the float64 decode of the same inputs (tests/dfl_bound.py).  A side with a NaN or +inf bin, or
 * only -inf bins, decodes to NaN in its two outputs (l, r: cx and w; t, b: cy and h).
 * Refuses (B200VA_ERR_INVALID) NULL pointers, batch or num_classes < 0, reg_max outside [1, 64], n_levels
 * outside [1, 8], a level with h or w <= 0, and more than INT_MAX anchors in all. */
B200VA_API int b200va_dfl_decode(b200va_handle h, const float* raw, int batch, int num_classes, int reg_max,
                                 const int* level_hw, const float* level_stride, int n_levels, float* out,
                                 void* stream);

/* ---- a8: IoU tracker -----------------------------------------------------------------
 * Replaces IouTracker.update (tracker.py:50-95), _match_detection (:97-109), _prune_tracks
 * (:111-126), _iou (:129-147) for a batch of streams; state lives in the handle per slot.
 * stream_slots HOST [batch] slot ids in [0, max_streams), distinct within a call
 * dets         detections per frame ([batch, max_dets] SoA as produced by b200va_postprocess);
 *              max_dets in [1, 32768] (a track row remembers its detection in 16 bits), else
 *              B200VA_ERR_INVALID;
 *              det_scale HOST double [batch] or NULL: pipeline.py:224-240 rescale (1/ratio), applied
 *              in float64 to the boxes before matching
 * skip         HOST uint8 [batch] or NULL: 1 = tracker.update(stream, []) (pipeline.py:214-215)
 * id_base      HOST int64 [batch] or NULL.  New tracks get ids id_base[i], id_base[i]+1, ... in
 *              creation order; NULL = draw from the handle's shared counter in batch order,
 *              which reproduces one shared itertools.count(1) updated stream by stream
 *              (tracker.py:47, pipeline.py:452)
 * out          all surviving tracks per stream in insertion order (tracker.py:95), may be NULL
 * new_counts   DEVICE int32 [batch] number of tracks created by this call, may be NULL
 * The IoU is tracker.py's float64 arithmetic with Python's builtin min / max, track first: a NaN
 * coordinate of a detection is replaced by the track's in the intersection (so such a detection can
 * match, with an IoU above 1 even), a NaN coordinate of a track makes its IoU 0. */
B200VA_API int b200va_tracker_update(b200va_handle h, const int* stream_slots, int batch, const b200va_dets* dets,
                          int max_dets, const double* det_scale, const uint8_t* skip,
                          const b200va_tracker_cfg* cfg, const int64_t* id_base, const b200va_tracks* out,
                          int32_t* new_counts, void* stream);
/* Same, for float64 detections (no det_scale: the caller already holds final doubles). */
B200VA_API int b200va_tracker_update_f64(b200va_handle h, const int* stream_slots, int batch, const b200va_dets64* dets,
                              int max_dets, const uint8_t* skip, const b200va_tracker_cfg* cfg,
                              const int64_t* id_base, const b200va_tracks* out, int32_t* new_counts,
                              void* stream);
B200VA_API int b200va_tracker_reset(b200va_handle h, int stream_slot, void* stream);
/* Set the next id of the shared counter (default 1, like itertools.count(1)). */
B200VA_API int b200va_tracker_set_next_id(b200va_handle h, int64_t next_id, void* stream);

/* ---- a12 on the device: the per-stream gates and the adaptive-FPS state -----------------------
 * Replaces, for a batch of streams and without a host round trip, the gate logic of StreamWorker._process_packet:
 * `self._frame_index += 1` (pipeline.py:144), the motion decision `count / size >= threshold`
 * (frame_filter.py:38-40, pipeline.py:156-163; a stream's first frame always passes), the adaptive-FPS test
 * `(self._frame_index - 1) % self._process_every != 0` (pipeline.py:165-170) and _adjust_adaptive_state
 * (pipeline.py:242-262).  frame_index, idle_frames and process_every live in the handle per slot.
 *
 * b200va_gates_decide   after b200va_motion: writes skip_out[i] (DEVICE uint8 [batch]) = B200VA_GATE_PROCESS,
 *                       _SKIP_MOTION or _SKIP_ADAPTIVE.  `changed` = b200va_motion's changed_out (DEVICE; may be NULL
 *                       when no gate uses the motion filter); gates[i].changed_index picks the entry.
 * b200va_set_skip_mask  makes every later b200va_preprocess / b200va_preprocess_geom / b200va_postprocess* /
 *                       b200va_tracker_update* / b200va_tick call on this handle read `skip` (DEVICE uint8, one flag
 *                       per batch position, same order in all of them) ON THE DEVICE: a flagged frame is not
 *                       letterboxed (its rows of the output tensor are left as they are) and not decoded, its
 *                       detection count is 0, and its stream's tracker update is `update(stream, [])`
 *                       (_skip_frame, pipeline.py:214-222).  NULL switches the mask off.  The pointer is read by
 *                       the kernels, not by the call: it must stay valid while they run.
 * b200va_gates_commit   after the tracker update: _adjust_adaptive_state(len(filtered), len(tracks)) from the
 *                       device-side counts (det_count: b200va_dets.count, trk_count: b200va_tracks.count), and
 *                       state_out (DEVICE int32 [batch, 4], may be NULL) = {skip flag, process_every, idle_frames,
 *                       frame_index} after this frame -- what the caller copies back with its result tables. */
enum b200va_gate_decision { B200VA_GATE_PROCESS = 0, B200VA_GATE_SKIP_MOTION = 1, B200VA_GATE_SKIP_ADAPTIVE = 2 };
typedef struct b200va_gate {
  int32_t slot;              /* gate-state slot in [0, max_streams) (the stream's tracker slot)               */
  int32_t motion;            /* stream.motion_filter (config.py:67-73)                                        */
  int32_t changed_index;     /* index of this stream in `changed`; -1 = no motion result for it this tick      */
  int32_t adaptive;          /* stream.adaptive_fps                                                           */
  int32_t max_process_every; /* max(1, int(round(target_fps / max(min_target_fps, 1)))) (pipeline.py:107-111) */
  int32_t idle_tolerance;    /* max(int(idle_frame_tolerance), 1) (pipeline.py:112)                           */
  double motion_threshold;   /* MotionFilterConfig.threshold                                                  */
  int64_t pixels;            /* thresh.size: height * width of the frame the motion gate saw                  */
} b200va_gate;
B200VA_API int b200va_gates_decide(b200va_handle h, const b200va_gate* gates /* HOST [batch] */, int batch,
                                   const int32_t* changed, uint8_t* skip_out, void* stream);
B200VA_API int b200va_gates_commit(b200va_handle h, const b200va_gate* gates /* HOST [batch] */, int batch,
                                   const int32_t* det_count, const int32_t* trk_count, const uint8_t* skip,
                                   int32_t* state_out, void* stream);
B200VA_API int b200va_gates_reset(b200va_handle h, int slot, void* stream);
B200VA_API int b200va_set_skip_mask(b200va_handle h, const uint8_t* skip /* DEVICE or NULL */);

/* ---- Ultralytics semantics (SURVEY.md 8f row 2; additive) ---------------------------------
 * What `YOLO(...).predict(frame, conf, iou, classes, half)` -- the call UltralyticsDetector.predict makes
 * (detector.py:147-155) -- does around the model forward.  ultralytics==8.3.209 (pylock.toml:1432-1433) is not
 * part of /root/reference and not installed: these entry points restate its published algorithm (LetterBox,
 * ops.non_max_suppression, ops.scale_boxes); the NMS step is pinned against torchvision.ops.nms, the rest
 * against torch CPU arithmetic -- PARITY UNPINNED against ultralytics itself.
 *
 * Geometry: new size = round(size * r), r = min(dst_h/h, dst_w/w); padding split round(d/2 -+ 0.1);
 * auto_pad != 0 pads only the remainder modulo `stride` (the rect shape predict() uses for one image), so the
 * network input is out_h x out_w <= dst_h x dst_w.  out->scale = r. */
B200VA_API int b200va_letterbox_meta_ultralytics(int src_h, int src_w, int dst_h, int dst_w, int auto_pad, int stride,
                                                 b200va_letterbox* out, int* out_h, int* out_w);
/* b200va_preprocess with caller-supplied geometry (geom[i].new_h/new_w/pad_top/pad_left; e.g. from
 * b200va_letterbox_meta_ultralytics); every frame is written into a dst_h x dst_w canvas.  Same kernels, same
 * interpolation, pad value and output formats.  (torch CUDA computes `im /= 255` as im * float32(1/255), which
 * is exactly B200VA_OUT_F32_RGB_NCHW.) */
B200VA_API int b200va_preprocess_geom(b200va_handle h, const uint8_t* const* frames, const int* src_h, const int* src_w,
                                      const int64_t* src_pitch, int batch, const uint8_t* const* roi_masks,
                                      const b200va_letterbox* geom, void* out, int dst_h, int dst_w, int out_format,
                                      void* stream);
/* b200va_preprocess_geom for NV12 frames (b200va_nv12_frame, below): the letterbox of b200va_preprocess_nv12 with the
 * caller's geometry, byte-identical to b200va_preprocess_geom on cv2.cvtColor(frame, COLOR_YUV2BGR_NV12).  The checks of
 * both calls apply: the geometry matches each frame and fits the canvas; odd sizes and NULL planes are refused. */
B200VA_API int b200va_preprocess_geom_nv12(b200va_handle h, const b200va_nv12_frame* frames, const int* src_h,
                                           const int* src_w, int batch, const uint8_t* const* roi_masks,
                                           const b200va_letterbox* geom, void* out, int dst_h, int dst_w, int out_format,
                                           void* stream);
/* b200va_upload_frames / b200va_upload_frames_nv12 in rows mode 1 for frames that b200va_preprocess_geom* letterboxes
 * with the caller's geometry: geom HOST [batch] (geom[i].src_h / src_w must be the frame's size) instead of dst_h /
 * dst_w.  Only the rows the letterbox to geom[i].new_h rows reads cross the bus (NV12: those luma rows and the chroma
 * rows they use); the LetterBox geometry of b200va_letterbox_meta_ultralytics rounds new_h where the reference
 * geometry truncates it, so it can read rows the reference-geometry upload skips.  Rows that need more than eight
 * strided copies, or more than 80 % of a plane, go whole; bytes_copied receives the bytes put on the bus. */
B200VA_API int b200va_upload_frames_geom(b200va_handle h, const uint8_t* const* host_frames, uint8_t* const* dev_frames,
                                         const int* src_h, const int* src_w, const int64_t* host_pitch,
                                         const int64_t* dev_pitch, int batch, const b200va_letterbox* geom,
                                         int64_t* bytes_copied, void* stream);
B200VA_API int b200va_upload_frames_nv12_geom(b200va_handle h, const b200va_nv12_frame* host, const b200va_nv12_frame* dev,
                                              const int* src_h, const int* src_w, int batch, const b200va_letterbox* geom,
                                              int64_t* bytes_copied, void* stream);
/* ops.non_max_suppression + ops.scale_boxes for a decoded head [B, 4 + nc, A] / [B, A, 4 + nc]:
 * score_k = head[4 + k], candidate iff max_k > conf_thr (strict, float32); xywh -> xyxy in network-input pixels;
 * NMS on boxes shifted by class * 7680 in float32 (agnostic != 0: no shift) with torchvision's test
 * inter / (area_i + area_j - inter) > iou_thr (float32 IoU against the double threshold, CPU kernel), equal
 * scores keep the lower anchor first (stable descending sort); the first max_det survivors are un-letterboxed
 * with gain = min(in_h/h, in_w/w), pad = round((in - size * gain) / 2 - 0.1), true division by float32(gain),
 * clamp to [0, w] x [0, h].  max_nms (30000) is never reached: candidates are bounded by max_candidates.
 * in_h / in_w: shape of the network input the head was computed from.  filter_*, classes and signed zeros: as in
 * b200va_postprocess. */
B200VA_API int b200va_postprocess_ultralytics(b200va_handle h, const void* head, int layout, int batch, int channels,
                                              int anchors, const int* src_h, const int* src_w, int in_h, int in_w,
                                              double conf_thr, double iou_thr, const int32_t* classes, int n_classes,
                                              int agnostic, int max_det, double filter_conf_thr_f64, int use_filter,
                                              const b200va_dets* out, void* stream);

/* ---- one tick: pre ‖ post + track ------------------------------------------------------
 * The batched form of StreamWorker._process_packet's GPU work (pipeline.py:172-188) for callers that
 * pipeline around the detector: the letterbox of the frames that go to the detector NEXT and the
 * head post-process + tracker update of the head the detector produced LAST are independent, so
 * one call runs them as two branches -- the letterbox on `stream`, decode -> NMS -> tracker on an
 * internal high-priority stream forked from and joined back into `stream` (capturable in a CUDA
 * graph).  Every pointer has the meaning it has in b200va_preprocess / b200va_postprocess /
 * b200va_tracker_update; results are identical to calling those three in sequence.
 * schedule: 0 = serial on `stream`; 1 = the letterbox starts when the decode kernel has finished and
 *           overlaps NMS + tracker (the two HBM-bound kernels never share the bus); 2 = the letterbox
 *           overlaps the whole post-process branch; 3 = the decode kernel runs on `stream` and the letterbox
 *           follows it there as a programmatic dependent launch that never waits for it -- its CTAs fill the SMs
 *           beside the decode's as soon as all of those are running (HBM sees the decode's reads and the letterbox's
 *           writes together, no kernel-to-kernel gap) -- while NMS + tracker run on the internal stream behind
 *           an event recorded after the decode.
 *           5 = like 3, but the letterbox waits (griddepcontrol.wait) for the decode grid to drain before its first
 *           load: back to back on the bus instead of side by side, without a launch gap in between.
 *           4 = software-pipelined: this call only DECODES its head (into one of two candidate sets) and letterboxes
 *           its frames; NMS + tracker of the head the PREVIOUS call decoded run beside them on the internal stream.
 *           The latency-bound chain decode -> NMS -> tracker, which bounds schedules 1-3, leaves the critical path.
 *           The result tables of call k are complete after call k + 1 has run (or after a final call with neither
 *           frames nor head, which only drains the pipeline); `dets`, `tracks`, `new_counts` and the buffers they
 *           point to must stay valid and untouched until then.  A call with another schedule first runs what is owed.
 *           6 = automatic: 3 for batches of 24 frames or more while the scenes are sparse (the letterbox is the long
 *           pole), otherwise 1: small batches (the chain decode -> NMS -> tracker is, and 3 starts it later) and while
 *           the post-process reports dense frames (more than 256 candidates in a frame lately), where letterbox CTAs
 *           launched early would take SMs from the NMS chain.
 * Sparse scenes run NMS and the tracker update of the same rows as ONE kernel (a 256-thread CTA per stream);
 * otherwise the two kernels are chained by programmatic dependent launch.
 * ev_pre_begin / ev_pre_end: optional cudaEvent_t recorded on `stream` around the letterbox launch. */
typedef struct b200va_tick_args {
  /* b200va_preprocess */
  const uint8_t* const* frames;
  const int* src_h;
  const int* src_w;
  const int64_t* src_pitch;
  int batch;
  const uint8_t* const* roi_masks;
  void* net_out;
  int dst_h, dst_w, out_format;
  b200va_letterbox* meta_out;
  /* b200va_postprocess */
  const void* head; /* float32, or float16 with B200VA_HEAD_F16 in `layout` */
  int layout, head_batch, channels, anchors;
  const b200va_letterbox* meta;
  double conf_thr, iou_thr;
  const int32_t* classes;
  int n_classes, score_mode, nms_mode;
  double filter_conf_thr_f64;
  int use_filter;
  const b200va_dets* dets;
  /* b200va_tracker_update */
  const int* stream_slots;
  int trk_batch, max_dets;
  const double* det_scale;
  const uint8_t* skip;
  const b200va_tracker_cfg* trk_cfg;
  const int64_t* id_base;
  const b200va_tracks* tracks;
  int32_t* new_counts;
  /* scheduling */
  int schedule;
  void* ev_pre_begin;
  void* ev_pre_end;
} b200va_tick_args;
B200VA_API int b200va_tick(b200va_handle h, const b200va_tick_args* args, void* stream);
/* b200va_tick with the letterbox reading NV12 frames (b200va_preprocess_nv12): frames HOST [args->batch] plane
 * descriptors; args->frames and args->src_pitch are not read.  Every schedule, graph capture included; the results
 * are those of b200va_tick on the frames converted by cv2.cvtColor(frame, COLOR_YUV2BGR_NV12). */
B200VA_API int b200va_tick_nv12(b200va_handle h, const b200va_tick_args* args, const b200va_nv12_frame* frames, void* stream);
/* b200va_tick with Ultralytics semantics: the letterbox half is b200va_preprocess_geom (BGR, frames == NULL) or
 * b200va_preprocess_geom_nv12 (frames: HOST [args->batch] NV12 plane descriptors) with u->geom, the post half is
 * b200va_postprocess_ultralytics with u->src_h / src_w / in_h / in_w / agnostic / max_det, and the tracker half is
 * unchanged.  args->meta, args->score_mode and args->nms_mode are not read, and args->meta_out is not written.  Every
 * schedule, graph capture and the skip mask included; the results are those of the three separate calls. */
typedef struct b200va_tick_ultra {
  const b200va_letterbox* geom; /* HOST [args->batch] letterbox geometry of each frame (b200va_letterbox_meta_ultralytics) */
  const int* src_h;             /* HOST [args->head_batch] original frame sizes of the head's frames (scale_boxes)    */
  const int* src_w;
  int in_h, in_w;               /* network-input shape the head was computed from                                   */
  int agnostic, max_det;
} b200va_tick_ultra;
B200VA_API int b200va_tick_ultralytics(b200va_handle h, const b200va_tick_args* args, const b200va_tick_ultra* u,
                                       const b200va_nv12_frame* frames /* NULL = BGR */, void* stream);

/* ---- 8f-3: egress (the preview and the event the sink publishes) -------------------------------
 * Replaces, for a frame that is already in HBM, the pixel work of KafkaSink._render_frame
 * (sinks/kafka_sink.py:200-267) and the serialisation of KafkaSink.send_tracks (:105-134 with the producer's
 * value_serializer json.dumps, :88).  Glyph rasterisation (cv2.putText) and the JPEG / WebP encoder stay with the
 * caller: they are the reference's own OpenCV calls on the (much smaller) annotated preview.
 *
 * b200va_resize_area_u8: cv2.resize(frame, (dst_w, dst_h), interpolation=cv2.INTER_AREA) for BGR uint8 HWC frames,
 * shrinking only (kafka_sink.py:227-232 downscales frames above 1920x1080).  Bit-exact with OpenCV 4.x: whole 2x2
 * blocks round half up ((a+b+c+d+2)>>2, the vector kernel), other whole blocks multiply by float(1/area) and round
 * half to even, fractional ratios accumulate float32 products in computeResizeAreaTab order.
 * frames / dst: HOST arrays [batch] of DEVICE pointers; dst pitch = 3 * dst_w.  NV12 frames: b200va_resize_area_u8_nv12. */
B200VA_API int b200va_resize_area_u8(b200va_handle h, const uint8_t* const* frames, const int* src_h, const int* src_w,
                                     const int64_t* src_pitch, int batch, uint8_t* const* dst, const int* dst_h,
                                     const int* dst_w, void* stream);

/* b200va_draw_rects: the rectangles of kafka_sink.py:240 (cv2.rectangle(img, p1, p2, color, 2): kind 0) and
 * :249-255 (cv2.rectangle(.., color, -1): kind 1) drawn into BGR uint8 images IN LIST ORDER (a later rectangle
 * overwrites an earlier one, like successive cv2 calls).  Corner points may lie outside the image (clipped) and in
 * any order.  ops: HOST array; image b owns ops[op_offsets[b] .. op_offsets[b + 1]).  images: HOST array [batch] of
 * DEVICE pointers, pitch in bytes (NULL = 3 * w). */
typedef struct b200va_rect_op {
  int32_t kind;           /* 0 = outline, thickness 2; 1 = filled */
  int32_t x1, y1, x2, y2; /* the two corner points, inclusive */
  uint8_t b, g, r, pad_;
} b200va_rect_op;
B200VA_API int b200va_draw_rects(b200va_handle h, uint8_t* const* images, const int* img_h, const int* img_w,
                                 const int64_t* pitch, int batch, const b200va_rect_op* ops, const int* op_offsets,
                                 void* stream);

/* b200va_tracks_json: the bytes of json.dumps({"stream": .., "frame_id": .., "tracks": [{"track_id", "class_id",
 * "confidence", "bbox_xyxy"}, ..], "is_temporal": false[, "frame_jpeg": frame_data_url]}) exactly as CPython writes
 * them (", " / ": " separators, float.__repr__ shortest round-trip digits, ensure_ascii escapes, NaN / Infinity).
 * Host-only (no handle, no device work): all pointers are HOST arrays, e.g. rows of the pinned result tables
 * (track_id [n], cls [n], conf [n] float64, bbox_xyxy [n, 4] float64).  Writes at most `cap` bytes to `out` (not
 * NUL-terminated) and returns the number of bytes the document needs (call again with a larger buffer when the
 * return value exceeds cap); -1 on invalid arguments. */
B200VA_API int64_t b200va_tracks_json(const char* stream_name, int64_t frame_id, const int64_t* track_id, const int32_t* cls,
                                      const double* conf, const double* bbox_xyxy, int n, const char* frame_data_url,
                                      char* out, int64_t cap);

#ifdef __cplusplus
}
#endif
#endif /* B200VA_H_ */
