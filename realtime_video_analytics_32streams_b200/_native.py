"""ctypes binding of ``libb200va.so`` (C ABI declared in ``include/b200va.h``).

The shared library is the product: every compute entry point launches sm_100a kernels and
there is no Python/NumPy/torch fallback.  If the library is missing or fails to load this module
raises at import of the first symbol -- it never degrades silently.  PyTorch appears only as the
owner of device memory and CUDA streams; tensors are passed down as raw pointers.
"""

from __future__ import annotations

import ctypes as C
import os
from typing import List, Optional, Sequence

PKG_DIR = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.environ.get("B200VA_LIB") or os.path.join(PKG_DIR, "lib", "libb200va.so")

OK, ERR_INVALID, ERR_CUDA, ERR_CAPACITY, ERR_STATE = 0, -1, -2, -3, -4
OUT_F32_RGB_NCHW, OUT_F16_RGB_NCHW, OUT_U8_BGR_NCHW, OUT_U8_BGR_NHWC = 0, 1, 2, 3
OUT_FLAG_PADS_VALID = 0x100  # OR into the format: the pad rows of `out` are still valid from an earlier call
HEAD_CHANNEL_MAJOR, HEAD_ANCHOR_MAJOR = 0, 1
HEAD_F16 = 0x200  # OR into the layout: the head is float16 (read in place, exactly as its float32 widening)
SCORE_REF_COMPAT, SCORE_V8_NATIVE = 0, 1
NMS_AGNOSTIC, NMS_CLASS_AWARE = 0, 1


class B200VAError(RuntimeError):
    def __init__(self, status: int, message: str):
        super().__init__(f"libb200va: {message} (status {status})")
        self.status = status


class Config(C.Structure):
    _fields_ = [("device", C.c_int), ("max_batch", C.c_int), ("max_anchors", C.c_int), ("max_candidates", C.c_int),
                ("max_dets", C.c_int), ("max_streams", C.c_int), ("max_tracks", C.c_int)]


class Letterbox(C.Structure):
    _fields_ = [("src_h", C.c_int), ("src_w", C.c_int), ("new_h", C.c_int), ("new_w", C.c_int),
                ("pad_left", C.c_int), ("pad_top", C.c_int), ("scale", C.c_double)]

    def as_meta(self) -> dict:
        """The ``meta`` dict of detector.py:259-263."""
        return {"orig_shape": (self.src_h, self.src_w), "scale": self.scale, "pad": (self.pad_left, self.pad_top)}


class Dets(C.Structure):
    _fields_ = [("bbox_xyxy", C.c_void_p), ("conf", C.c_void_p), ("cls", C.c_void_p), ("count", C.c_void_p)]


class Dets64(C.Structure):
    _fields_ = [("bbox_xyxy", C.c_void_p), ("conf", C.c_void_p), ("cls", C.c_void_p), ("count", C.c_void_p)]


class TrackerCfg(C.Structure):
    _fields_ = [("max_age", C.c_int), ("min_hits", C.c_int), ("max_iou_distance", C.c_double)]


class Tracks(C.Structure):
    _fields_ = [("track_id", C.c_void_p), ("cls", C.c_void_p), ("conf", C.c_void_p), ("bbox_xyxy", C.c_void_p),
                ("age", C.c_void_p), ("hits", C.c_void_p), ("count", C.c_void_p), ("rows", C.c_int32)]


class Gate(C.Structure):
    """``b200va_gate`` (include/b200va.h): one stream's gates for the device-side decisions (pipeline.py:104-116, 156-170)."""

    _fields_ = [("slot", C.c_int32), ("motion", C.c_int32), ("changed_index", C.c_int32), ("adaptive", C.c_int32),
                ("max_process_every", C.c_int32), ("idle_tolerance", C.c_int32), ("motion_threshold", C.c_double),
                ("pixels", C.c_int64)]


GATE_PROCESS, GATE_SKIP_MOTION, GATE_SKIP_ADAPTIVE = 0, 1, 2


class RectOp(C.Structure):
    """``b200va_rect_op`` (include/b200va.h): kind 0 = thickness-2 outline, 1 = filled."""

    _fields_ = [("kind", C.c_int32), ("x1", C.c_int32), ("y1", C.c_int32), ("x2", C.c_int32), ("y2", C.c_int32),
                ("b", C.c_uint8), ("g", C.c_uint8), ("r", C.c_uint8), ("pad_", C.c_uint8)]


class Nv12Frame(C.Structure):
    """``b200va_nv12_frame`` (include/b200va.h): the two planes of an NV12 frame, each with its own pitch."""

    _fields_ = [("y", C.c_void_p), ("uv", C.c_void_p), ("y_pitch", C.c_int64), ("uv_pitch", C.c_int64)]


class TickArgs(C.Structure):
    """``b200va_tick_args`` (include/b200va.h)."""

    _fields_ = [
        ("frames", C.POINTER(C.c_void_p)), ("src_h", C.POINTER(C.c_int)), ("src_w", C.POINTER(C.c_int)),
        ("src_pitch", C.POINTER(C.c_int64)), ("batch", C.c_int), ("roi_masks", C.POINTER(C.c_void_p)),
        ("net_out", C.c_void_p), ("dst_h", C.c_int), ("dst_w", C.c_int), ("out_format", C.c_int),
        ("meta_out", C.POINTER(Letterbox)),
        ("head", C.c_void_p), ("layout", C.c_int), ("head_batch", C.c_int), ("channels", C.c_int), ("anchors", C.c_int),
        ("meta", C.POINTER(Letterbox)), ("conf_thr", C.c_double), ("iou_thr", C.c_double),
        ("classes", C.POINTER(C.c_int32)), ("n_classes", C.c_int), ("score_mode", C.c_int), ("nms_mode", C.c_int),
        ("filter_conf_thr_f64", C.c_double), ("use_filter", C.c_int), ("dets", C.POINTER(Dets)),
        ("stream_slots", C.POINTER(C.c_int)), ("trk_batch", C.c_int), ("max_dets", C.c_int),
        ("det_scale", C.POINTER(C.c_double)), ("skip", C.POINTER(C.c_uint8)), ("trk_cfg", C.POINTER(TrackerCfg)),
        ("id_base", C.POINTER(C.c_int64)), ("tracks", C.POINTER(Tracks)), ("new_counts", C.c_void_p),
        ("schedule", C.c_int), ("ev_pre_begin", C.c_void_p), ("ev_pre_end", C.c_void_p),
    ]


SCHEDULE_SERIAL, SCHEDULE_PRE_AFTER_DECODE, SCHEDULE_PRE_PARALLEL, SCHEDULE_PRE_BESIDE_DECODE = 0, 1, 2, 3
SCHEDULE_PRE_BEHIND_DECODE = 5  # like 3, the letterbox waits for the decode grid to drain (griddepcontrol.wait)
SCHEDULE_AUTO = 6  # 3 for large sparse batches, 1 for small batches and dense scenes (the default; include/b200va.h)
SCHEDULE_SOFTWARE_PIPELINED = 4  # decode + letterbox of this call beside NMS + tracker of the previous call's head


class TickPlan:
    """A fully prepared ``b200va_tick`` call: the argument block and everything it points to are
    built once, so a tick costs the host one foreign-function call."""

    def __init__(self, args: "TickArgs", keep: tuple):
        self.args = args
        self._keep = keep  # owners of every pointer inside `args`
        self.nv12 = None   # Nv12Frame array: the letterbox reads NV12 frames (b200va_tick_nv12)

    def set_events(self, begin=None, end=None) -> None:
        """Optional (already recorded once) ``torch.cuda.Event`` pair around the letterbox launch."""
        self.args.ev_pre_begin = C.c_void_p(begin.cuda_event) if begin is not None else None
        self.args.ev_pre_end = C.c_void_p(end.cuda_event) if end is not None else None


EXPORTS = (
    "b200va_version", "b200va_error_string", "b200va_create", "b200va_destroy", "b200va_last_error",
    "b200va_launch_count", "b200va_poll_status", "b200va_letterbox_meta", "b200va_preprocess",
    "b200va_resize_linear_u8", "b200va_roi_rasterize", "b200va_apply_mask", "b200va_motion",
    "b200va_postprocess", "b200va_tracker_update", "b200va_tracker_update_f64", "b200va_tracker_reset",
    "b200va_tracker_set_next_id", "b200va_upload_frames", "b200va_dfl_decode", "b200va_tick",
    "b200va_letterbox_meta_ultralytics", "b200va_preprocess_geom", "b200va_postprocess_ultralytics",
    "b200va_motion_preprocess", "b200va_set_profiling", "b200va_get_phase_times",
    "b200va_read_status_async", "b200va_resize_area_u8", "b200va_draw_rects", "b200va_tracks_json",
    "b200va_gates_decide", "b200va_gates_commit", "b200va_gates_reset", "b200va_set_skip_mask",
    "b200va_preprocess_nv12", "b200va_resize_linear_u8_nv12", "b200va_upload_frames_nv12", "b200va_tick_nv12",
    "b200va_resize_area_u8_nv12",
)
PHASES = ("upload", "roi", "resize", "motion", "preprocess", "decode", "nms", "tracker", "dfl", "tick", "egress")  # enum b200va_phase

_lib = None


def load_library() -> C.CDLL:
    """Load ``libb200va.so``; raises (never falls back) when it is absent."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise ImportError(
            f"{LIB_PATH} not found: build it with `python -m realtime_video_analytics_32streams_b200.build` "
            "(nvcc, sm_100a).  There is no CPU fallback.")
    lib = C.CDLL(LIB_PATH)
    vp, ip, i64p = C.c_void_p, C.POINTER(C.c_int), C.POINTER(C.c_int64)
    lib.b200va_version.restype = C.c_int
    lib.b200va_error_string.restype = C.c_char_p
    lib.b200va_error_string.argtypes = [C.c_int]
    lib.b200va_create.argtypes = [C.POINTER(Config), C.POINTER(vp)]
    lib.b200va_destroy.argtypes = [vp]
    lib.b200va_last_error.restype = C.c_char_p
    lib.b200va_last_error.argtypes = [vp]
    lib.b200va_launch_count.restype = C.c_int64
    lib.b200va_launch_count.argtypes = [vp]
    lib.b200va_poll_status.argtypes = [vp, vp]
    lib.b200va_letterbox_meta.argtypes = [C.c_int, C.c_int, C.c_int, C.c_int, C.POINTER(Letterbox)]
    lib.b200va_preprocess.argtypes = [vp, C.POINTER(vp), ip, ip, i64p, C.c_int, C.POINTER(vp), vp, C.c_int, C.c_int,
                                      C.c_int, C.POINTER(Letterbox), vp]
    lib.b200va_resize_linear_u8.argtypes = [vp, C.POINTER(vp), ip, ip, i64p, C.c_int, C.POINTER(vp), C.POINTER(vp),
                                            ip, ip, vp]
    lib.b200va_roi_rasterize.argtypes = [vp, C.POINTER(C.c_int32), ip, C.c_int, C.c_int, C.c_int, vp, vp]
    lib.b200va_apply_mask.argtypes = [vp, vp, C.c_int64, vp, C.c_int, C.c_int, vp, C.c_int64, vp]
    lib.b200va_motion.argtypes = [vp, C.POINTER(vp), ip, ip, i64p, C.c_int, C.POINTER(vp), C.POINTER(vp),
                                  C.POINTER(vp), ip, vp, vp]
    lib.b200va_postprocess.argtypes = [vp, vp, C.c_int, C.c_int, C.c_int, C.c_int, C.POINTER(Letterbox), C.c_double,
                                       C.c_double, C.POINTER(C.c_int32), C.c_int, C.c_int, C.c_int, C.c_double, C.c_int,
                                       C.POINTER(Dets), vp]
    lib.b200va_tracker_update.argtypes = [vp, ip, C.c_int, C.POINTER(Dets), C.c_int, C.POINTER(C.c_double),
                                          C.POINTER(C.c_uint8), C.POINTER(TrackerCfg), i64p, C.POINTER(Tracks), vp, vp]
    lib.b200va_tracker_update_f64.argtypes = [vp, ip, C.c_int, C.POINTER(Dets64), C.c_int, C.POINTER(C.c_uint8),
                                              C.POINTER(TrackerCfg), i64p, C.POINTER(Tracks), vp, vp]
    lib.b200va_upload_frames.argtypes = [vp, C.POINTER(vp), C.POINTER(vp), ip, ip, i64p, i64p, C.c_int, C.c_int,
                                         C.c_int, C.c_int, i64p, vp]
    lib.b200va_dfl_decode.argtypes = [vp, vp, C.c_int, C.c_int, C.c_int, ip, C.POINTER(C.c_float), C.c_int, vp, vp]
    lib.b200va_motion_preprocess.argtypes = [vp, C.POINTER(vp), ip, ip, i64p, C.c_int, C.POINTER(vp), C.POINTER(vp),
                                             C.POINTER(vp), ip, vp, vp, C.c_int, C.c_int, C.c_int, C.POINTER(Letterbox), vp]
    lib.b200va_tick.argtypes = [vp, C.POINTER(TickArgs), vp]
    lib.b200va_letterbox_meta_ultralytics.argtypes = [C.c_int, C.c_int, C.c_int, C.c_int, C.c_int, C.c_int,
                                                      C.POINTER(Letterbox), ip, ip]
    lib.b200va_preprocess_geom.argtypes = [vp, C.POINTER(vp), ip, ip, i64p, C.c_int, C.POINTER(vp), C.POINTER(Letterbox),
                                           vp, C.c_int, C.c_int, C.c_int, vp]
    lib.b200va_postprocess_ultralytics.argtypes = [vp, vp, C.c_int, C.c_int, C.c_int, C.c_int, ip, ip, C.c_int, C.c_int,
                                                   C.c_double, C.c_double, C.POINTER(C.c_int32), C.c_int, C.c_int, C.c_int,
                                                   C.c_double, C.c_int, C.POINTER(Dets), vp]
    lib.b200va_read_status_async.argtypes = [vp, vp, C.c_int, vp]
    lib.b200va_set_profiling.argtypes = [vp, C.c_int]
    lib.b200va_get_phase_times.argtypes = [vp, C.POINTER(C.c_float)]
    lib.b200va_tracker_reset.argtypes = [vp, C.c_int, vp]
    lib.b200va_tracker_set_next_id.argtypes = [vp, C.c_int64, vp]
    lib.b200va_resize_area_u8.argtypes = [vp, C.POINTER(vp), ip, ip, i64p, C.c_int, C.POINTER(vp), ip, ip, vp]
    lib.b200va_draw_rects.argtypes = [vp, C.POINTER(vp), ip, ip, i64p, C.c_int, C.POINTER(RectOp), ip, vp]
    lib.b200va_gates_decide.argtypes = [vp, C.POINTER(Gate), C.c_int, vp, vp, vp]
    lib.b200va_gates_commit.argtypes = [vp, C.POINTER(Gate), C.c_int, vp, vp, vp, vp, vp]
    lib.b200va_gates_reset.argtypes = [vp, C.c_int, vp]
    lib.b200va_set_skip_mask.argtypes = [vp, vp]
    nv = C.POINTER(Nv12Frame)
    lib.b200va_preprocess_nv12.argtypes = [vp, nv, ip, ip, C.c_int, C.POINTER(vp), vp, C.c_int, C.c_int, C.c_int,
                                           C.POINTER(Letterbox), vp]
    lib.b200va_resize_linear_u8_nv12.argtypes = [vp, nv, ip, ip, C.c_int, C.POINTER(vp), C.POINTER(vp), ip, ip, vp]
    lib.b200va_upload_frames_nv12.argtypes = [vp, nv, nv, ip, ip, C.c_int, C.c_int, C.c_int, C.c_int, i64p, vp]
    lib.b200va_tick_nv12.argtypes = [vp, C.POINTER(TickArgs), nv, vp]
    lib.b200va_resize_area_u8_nv12.argtypes = [vp, nv, ip, ip, C.c_int, C.POINTER(vp), ip, ip, vp]
    lib.b200va_tracks_json.restype = C.c_int64
    lib.b200va_tracks_json.argtypes = [C.c_char_p, C.c_int64, vp, vp, vp, vp, C.c_int, C.c_char_p, vp, C.c_int64]
    for name in EXPORTS:
        getattr(lib, name)  # AttributeError here = header / library mismatch
    _lib = lib
    return lib


def tracks_json(stream_name: str, frame_id: int, track_id, cls, conf, bbox_xyxy, frame_data_url: Optional[str] = None) -> bytes:
    """``json.dumps(payload).encode()`` of the reference's track event (kafka_sink.py:88, 105-134), written by
    ``b200va_tracks_json`` straight from result-table rows: ``track_id`` int64 [n], ``cls`` int32 [n], ``conf`` float64 [n],
    ``bbox_xyxy`` float64 [n, 4] (C-contiguous NumPy arrays, e.g. ``FrameResult.track_arrays``).  Host-only; needs no GPU."""
    import numpy as np

    lib = load_library()
    ids = np.ascontiguousarray(track_id, dtype=np.int64)
    cl = np.ascontiguousarray(cls, dtype=np.int32)
    cf = np.ascontiguousarray(conf, dtype=np.float64)
    bx = np.ascontiguousarray(bbox_xyxy, dtype=np.float64).reshape(-1, 4)
    n = int(ids.shape[0])
    if not (cl.shape[0] == n and cf.shape[0] == n and bx.shape[0] == n):
        raise ValueError("tracks_json: the four arrays must have one row per track")
    name = stream_name.encode("utf-8")
    url = frame_data_url.encode("ascii") if frame_data_url is not None else None
    cap = 96 + len(name) * 6 + n * 160 + (len(url) + 32 if url else 0)
    while True:
        buf = C.create_string_buffer(cap)
        need = lib.b200va_tracks_json(name, int(frame_id), ids.ctypes.data, cl.ctypes.data, cf.ctypes.data, bx.ctypes.data, n,
                                      url, C.cast(buf, C.c_void_p), cap)
        if need < 0:
            raise B200VAError(ERR_INVALID, "b200va_tracks_json: invalid arguments")
        if need <= cap:
            return buf.raw[:need]
        cap = int(need)


def letterbox_meta(src_h: int, src_w: int, dst_h: int, dst_w: int) -> Letterbox:
    """Host-only geometry helper (detector.py:209-230); needs no GPU."""
    m = Letterbox()
    rc = load_library().b200va_letterbox_meta(src_h, src_w, dst_h, dst_w, C.byref(m))
    if rc != OK:
        raise B200VAError(rc, f"bad letterbox geometry {src_w}x{src_h} -> {dst_w}x{dst_h}")
    return m


def letterbox_meta_ultralytics(src_h: int, src_w: int, dst_h: int, dst_w: int, auto: bool = False, stride: int = 32):
    """Host-only: ultralytics ``LetterBox`` geometry -> (Letterbox, out_h, out_w); needs no GPU."""
    m, oh, ow = Letterbox(), C.c_int(0), C.c_int(0)
    rc = load_library().b200va_letterbox_meta_ultralytics(src_h, src_w, dst_h, dst_w, 1 if auto else 0, int(stride),
                                                          C.byref(m), C.byref(oh), C.byref(ow))
    if rc != OK:
        raise B200VAError(rc, f"bad letterbox geometry {src_w}x{src_h} -> {dst_w}x{dst_h}")
    return m, oh.value, ow.value


def _ptr_array(ptrs: Sequence[Optional[int]]):
    return (C.c_void_p * len(ptrs))(*[C.c_void_p(p) if p else None for p in ptrs])


def _int_array(vals: Sequence[int]):
    return (C.c_int * len(vals))(*[int(v) for v in vals])


class FrameBatch:
    """A validated batch of CUDA frames (and optional ROI masks) with its ctypes argument arrays
    built once.  Re-use it across calls while the underlying tensors stay alive and in place --
    the per-call host cost drops to one foreign-function call."""

    def __init__(self, frames, roi_masks=None):
        import torch as t

        self.frames = list(frames)
        self.masks = list(roi_masks) if roi_masks is not None else None
        for f in self.frames:
            if not (f.is_cuda and f.dtype == t.uint8 and f.dim() == 3 and f.shape[2] == 3 and f.stride(2) == 1
                    and f.stride(1) == 3):
                raise ValueError("frames must be CUDA uint8 tensors [H, W, 3] with packed pixels")
        n = len(self.frames)
        self.n = n
        self.ptrs = _ptr_array([f.data_ptr() for f in self.frames])
        self.hs = _int_array([f.shape[0] for f in self.frames])
        self.ws = _int_array([f.shape[1] for f in self.frames])
        self.pitch = (C.c_int64 * n)(*[f.stride(0) for f in self.frames])
        self.mask_ptrs = None
        if self.masks is not None and any(m is not None for m in self.masks):
            for m, f in zip(self.masks, self.frames):
                if m is not None and not (m.is_cuda and m.dtype == t.uint8 and m.is_contiguous()
                                          and tuple(m.shape) == tuple(f.shape[:2])):
                    raise ValueError("roi masks must be contiguous CUDA uint8 tensors [H, W] matching their frame")
            self.mask_ptrs = _ptr_array([m.data_ptr() if m is not None else None for m in self.masks])
        self.metas = (Letterbox * max(n, 1))()

    def __len__(self):
        return self.n


def is_nv12(frame) -> bool:
    """True for an NV12 frame: a ``(y, uv)`` pair or a 2-D ``[3H/2, W]`` array / tensor (BGR frames are ``[H, W, 3]``)."""
    return isinstance(frame, (tuple, list)) or getattr(frame, "ndim", 3) == 2


def frame_hw(frame):
    """(height, width) of a BGR ``[H, W, 3]`` frame, or of an NV12 frame's luma: ``H`` of a ``[3H/2, W]`` array /
    tensor (host or CUDA) or the ``y`` plane's size of a ``(y, uv)`` pair."""
    if isinstance(frame, (tuple, list)):
        return int(frame[0].shape[0]), int(frame[0].shape[1])
    if is_nv12(frame):
        return int(frame.shape[0]) * 2 // 3, int(frame.shape[1])
    return int(frame.shape[0]), int(frame.shape[1])


def nv12_planes(frame):
    """``(y [H, W], uv [H/2, W])`` of an NV12 frame given as one ``[3H/2, W]`` tensor (OpenCV's layout; any row pitch)
    or as a ``(y, uv)`` pair (decoder surfaces: separate bases and pitches).  The planes are views, not copies."""
    if isinstance(frame, (tuple, list)):
        if len(frame) != 2:
            raise ValueError("an NV12 plane pair is (y, uv)")
        y, uv = frame
    else:
        if frame.dim() != 2 or frame.shape[0] % 3:
            raise ValueError("an NV12 frame is a [3H/2, W] uint8 tensor")
        h = frame.shape[0] * 2 // 3
        y, uv = frame[:h], frame[h:]
    return y, uv


class Nv12Batch:
    """``FrameBatch`` for NV12 frames: CUDA uint8 ``[3H/2, W]`` tensors (any ``stride(0)``, ``stride(1) == 1``) or
    ``(y [H, W], uv [H/2, W])`` pairs of CUDA uint8 tensors; H and W even.  ROI masks are ``[H, W]`` (luma size)."""

    def __init__(self, frames, roi_masks=None):
        import torch as t

        self.frames = list(frames)
        self.planes = [nv12_planes(f) for f in self.frames]
        for y, uv in self.planes:
            if not all(p.is_cuda and p.dtype == t.uint8 and p.dim() == 2 and p.stride(1) == 1 for p in (y, uv)):
                raise ValueError("NV12 planes must be CUDA uint8 tensors [H, W] / [H/2, W] with unit column stride")
            if y.shape[0] % 2 or y.shape[1] % 2 or tuple(uv.shape) != (y.shape[0] // 2, y.shape[1]):
                raise ValueError(f"NV12 needs an even size and a [H/2, W] chroma plane, got y {tuple(y.shape)}, "
                                 f"uv {tuple(uv.shape)}")
        n = len(self.frames)
        self.n = n
        self.nv = (Nv12Frame * max(n, 1))(*[Nv12Frame(y.data_ptr(), uv.data_ptr(), y.stride(0), uv.stride(0))
                                             for y, uv in self.planes])
        self.hs = _int_array([y.shape[0] for y, _ in self.planes])
        self.ws = _int_array([y.shape[1] for y, _ in self.planes])
        self.masks = list(roi_masks) if roi_masks is not None else None
        self.mask_ptrs = None
        if self.masks is not None and any(m is not None for m in self.masks):
            for m, (y, _) in zip(self.masks, self.planes):
                if m is not None and not (m.is_cuda and m.dtype == t.uint8 and m.is_contiguous()
                                          and tuple(m.shape) == tuple(y.shape)):
                    raise ValueError("roi masks must be contiguous CUDA uint8 tensors [H, W] matching their frame's luma")
            self.mask_ptrs = _ptr_array([m.data_ptr() if m is not None else None for m in self.masks])
        self.metas = (Letterbox * max(n, 1))()

    def __len__(self):
        return self.n


class Handle:
    """One ``b200va_handle``: scratch arenas + tracker state on one GPU."""

    def __init__(self, device: int = 0, max_batch: int = 32, max_anchors: int = 8400, max_candidates: int = 4096,
                 max_dets: int = 1024, max_streams: int = 64, max_tracks: int = 4096):
        import torch

        if not torch.cuda.is_available():
            raise RuntimeError("libb200va needs a CUDA device (sm_100a); there is no CPU fallback")
        self.lib = load_library()
        self.torch = torch
        self.device = torch.device("cuda", device)
        self.cfg = Config(device, max_batch, max_anchors, max_candidates, max_dets, max_streams, max_tracks)
        self._h = C.c_void_p()
        rc = self.lib.b200va_create(C.byref(self.cfg), C.byref(self._h))
        if rc != OK:
            raise B200VAError(rc, (self.lib.b200va_last_error(None) or b"create failed").decode())

    # -- plumbing ---------------------------------------------------------------------------
    def close(self) -> None:
        if getattr(self, "_h", None) is not None and self._h:
            self.lib.b200va_destroy(self._h)
            self._h = C.c_void_p()

    def __del__(self):  # pragma: no cover
        try:
            self.close()
        except Exception:
            pass

    def _check(self, rc: int) -> None:
        if rc != OK:
            raise B200VAError(rc, (self.lib.b200va_last_error(self._h) or b"").decode())

    def _stream(self) -> C.c_void_p:
        return C.c_void_p(self.torch.cuda.current_stream(self.device).cuda_stream)

    @property
    def launch_count(self) -> int:
        return int(self.lib.b200va_launch_count(self._h))

    def poll_status(self) -> None:
        """Synchronise and raise if any capacity limit was hit since the last poll."""
        self._check(self.lib.b200va_poll_status(self._h, self._stream()))

    STATUS_WORDS = 8
    _STATUS_NAMES = ("candidates > max_candidates", "detections > max_dets", "tracks > max_tracks",
                     "tracks > rows of the result table")

    def read_status_async(self, host_out, clear: bool = True) -> None:
        """Enqueue a copy of the capacity flags into ``host_out`` (pinned CPU int32 tensor of ``STATUS_WORDS``
        elements) on the current stream; valid once that stream has been synchronised.  See ``status_message``."""
        self._check(self.lib.b200va_read_status_async(self._h, C.c_void_p(host_out.data_ptr()), 1 if clear else 0,
                                                      self._stream()))

    @classmethod
    def status_message(cls, words) -> Optional[str]:
        """None when no capacity was exceeded, else what was truncated."""
        hit = [n for n, w in zip(cls._STATUS_NAMES, list(words)[:4]) if int(w)]
        return ("capacity exceeded (rows were dropped; the reference is unbounded -- raise the handle's limits): "
                + ", ".join(hit)) if hit else None

    # -- tracker stream slots ----------------------------------------------------------------
    # The track tables and the id counter live in the handle, so the handle owns the slot numbers: two trackers (or
    # engines) on one handle get disjoint slots, a slot is emptied when it is claimed, and the id counter restarts
    # at 1 (itertools.count(1), tracker.py:47) whenever the first tracker of an otherwise idle handle claims a slot.
    def claim_slot(self) -> int:
        free = self.__dict__.setdefault("_free_slots", list(range(self.cfg.max_streams - 1, -1, -1)))
        if not free:
            raise B200VAError(ERR_CAPACITY, f"all {self.cfg.max_streams} tracker stream slots are in use")
        if len(free) == self.cfg.max_streams:
            self.tracker_set_next_id(1)
        slot = free.pop()
        self.tracker_reset(slot)
        return slot

    def release_slot(self, slot: int) -> None:
        free = self.__dict__.setdefault("_free_slots", list(range(self.cfg.max_streams - 1, -1, -1)))
        if slot not in free:
            free.append(int(slot))

    def set_profiling(self, enable: bool = True) -> None:
        """Bracket every phase's kernels with CUDA events (``b200va_set_profiling``); read with ``phase_times``."""
        self._check(self.lib.b200va_set_profiling(self._h, 1 if enable else 0))

    def phase_times(self) -> dict:
        """Device milliseconds of the phases that ran since the last query, e.g. ``{"preprocess": 0.041, ...}``
        (waits for them to finish).  The per-packet ``dt`` of pipeline.py:145, 200-201, measured on the GPU."""
        ms = (C.c_float * len(PHASES))()
        self._check(self.lib.b200va_get_phase_times(self._h, ms))
        return {name: float(ms[i]) for i, name in enumerate(PHASES) if ms[i] >= 0.0}

    @staticmethod
    def _batch(frames, roi_masks=None, nv12_ok: bool = False):
        """A ``FrameBatch``, or with ``nv12_ok`` an ``Nv12Batch`` for an ``Nv12Batch`` / a list of NV12 frames."""
        if isinstance(frames, FrameBatch):
            return frames
        if not isinstance(frames, Nv12Batch):
            frames = list(frames)
            if not (frames and all(is_nv12(f) for f in frames)):
                return FrameBatch(frames, roi_masks)
            frames = Nv12Batch(frames, roi_masks) if nv12_ok else frames
        if not nv12_ok:
            raise ValueError("NV12 frames are taken by preprocess, resize, resize_area and plan_tick; convert them "
                             "with resize at their own size for the other calls")
        return frames

    # -- staging ----------------------------------------------------------------------------
    def upload_frames(self, host_ptrs, dev_frames, sparse_for=None) -> int:
        """Asynchronous host -> device copy of decoded frames.  ``host_ptrs[i]`` = (address, pitch) of
        frame i in host memory (pinned for a truly asynchronous copy); ``dev_frames`` the CUDA
        uint8 [H,W,3] destination buffers.  ``sparse_for=(dst_h, dst_w)`` copies only the rows the
        letterbox to that size reads.  Returns the bytes put on the bus."""
        n = len(dev_frames)
        if n == 0:
            return 0
        moved = C.c_int64(0)
        self._check(self.lib.b200va_upload_frames(
            self._h, _ptr_array([p for p, _ in host_ptrs]), _ptr_array([d.data_ptr() for d in dev_frames]),
            _int_array([d.shape[0] for d in dev_frames]), _int_array([d.shape[1] for d in dev_frames]),
            (C.c_int64 * n)(*[int(pt) for _, pt in host_ptrs]), (C.c_int64 * n)(*[d.stride(0) for d in dev_frames]),
            n, int(sparse_for[0]) if sparse_for else 0, int(sparse_for[1]) if sparse_for else 0,
            1 if sparse_for else 0, C.byref(moved), self._stream()))
        return int(moved.value)

    def upload_frames_nv12(self, host_frames, dev_frames, sparse_for=None) -> int:
        """``upload_frames`` for NV12: ``host_frames[i]`` = ``Nv12Frame`` (host plane addresses and pitches; pinned for
        a truly asynchronous copy), ``dev_frames`` the CUDA NV12 destinations (``[3H/2, W]`` tensors or ``(y, uv)``
        pairs).  ``sparse_for=(dst_h, dst_w)`` copies only the luma rows the letterbox to that size reads and the
        chroma rows they use.  Returns the bytes put on the bus."""
        n = len(dev_frames)
        if n == 0:
            return 0
        db = Nv12Batch(dev_frames)
        hb = (Nv12Frame * n)(*host_frames)
        moved = C.c_int64(0)
        self._check(self.lib.b200va_upload_frames_nv12(
            self._h, hb, db.nv, db.hs, db.ws, n, int(sparse_for[0]) if sparse_for else 0,
            int(sparse_for[1]) if sparse_for else 0, 1 if sparse_for else 0, C.byref(moved), self._stream()))
        return int(moved.value)

    # -- a1 ---------------------------------------------------------------------------------
    def preprocess(self, frames, dst_hw=(640, 640), fmt: int = OUT_F32_RGB_NCHW, roi_masks=None, out=None):
        """Batched letterbox.  ``frames``: list of CUDA tensors or a ``FrameBatch``; NV12 frames (``[3H/2, W]`` tensors
        or ``(y, uv)`` pairs) or an ``Nv12Batch`` give the result of the BGR call on their ``cv2.cvtColor`` conversion.
        Returns (tensor [B,3,H,W] or [B,H,W,3], list of Letterbox)."""
        t = self.torch
        fb = self._batch(frames, roi_masks, nv12_ok=True)
        b = fb.n
        dh, dw = int(dst_hw[0]), int(dst_hw[1])
        dtype = {OUT_F32_RGB_NCHW: t.float32, OUT_F16_RGB_NCHW: t.float16}.get(fmt & 0xff, t.uint8)
        shape = (b, dh, dw, 3) if (fmt & 0xff) == OUT_U8_BGR_NHWC else (b, 3, dh, dw)
        if out is None:
            out = t.empty(shape, dtype=dtype, device=self.device)
        elif tuple(out.shape) != shape or out.dtype != dtype or not out.is_contiguous():
            raise ValueError("preprocess: `out` has the wrong shape / dtype / layout")
        if b and isinstance(fb, Nv12Batch):
            self._check(self.lib.b200va_preprocess_nv12(self._h, fb.nv, fb.hs, fb.ws, b, fb.mask_ptrs,
                                                        C.c_void_p(out.data_ptr()), dh, dw, fmt, fb.metas, self._stream()))
        elif b:
            self._check(self.lib.b200va_preprocess(self._h, fb.ptrs, fb.hs, fb.ws, fb.pitch, b, fb.mask_ptrs,
                                                   C.c_void_p(out.data_ptr()), dh, dw, fmt, fb.metas, self._stream()))
        return out, [fb.metas[i] for i in range(b)]

    # -- a10 --------------------------------------------------------------------------------
    def resize(self, frames, dst_hw_list, roi_masks=None, outs=None):
        """``cv2.resize(frame, (w, h), INTER_LINEAR)`` per frame; returns uint8 HWC tensors (``outs`` when given:
        contiguous CUDA uint8 [h, w, 3] tensors the caller keeps, else freshly allocated ones)."""
        t = self.torch
        if outs is None:
            outs = [t.empty((int(h), int(w), 3), dtype=t.uint8, device=self.device) for h, w in dst_hw_list]
        elif any(tuple(o.shape) != (int(h), int(w), 3) or o.dtype != t.uint8 or not o.is_contiguous() or not o.is_cuda
                 for o, (h, w) in zip(outs, dst_hw_list)) or len(outs) != len(dst_hw_list):
            raise ValueError("resize: `outs` must be contiguous CUDA uint8 tensors [h, w, 3] matching dst_hw_list")
        fb = self._batch(frames, roi_masks, nv12_ok=True)
        if fb.n and isinstance(fb, Nv12Batch):  # BGR out: at the frame's own size this is cv2.cvtColor itself
            self._check(self.lib.b200va_resize_linear_u8_nv12(
                self._h, fb.nv, fb.hs, fb.ws, fb.n, fb.mask_ptrs, _ptr_array([o.data_ptr() for o in outs]),
                _int_array([h for h, _ in dst_hw_list]), _int_array([w for _, w in dst_hw_list]), self._stream()))
        elif fb.n:
            self._check(self.lib.b200va_resize_linear_u8(
                self._h, fb.ptrs, fb.hs, fb.ws, fb.pitch, fb.n, fb.mask_ptrs,
                _ptr_array([o.data_ptr() for o in outs]), _int_array([h for h, _ in dst_hw_list]),
                _int_array([w for _, w in dst_hw_list]), self._stream()))
        return outs

    # -- 8f-3 -------------------------------------------------------------------------------
    def resize_area(self, frames, dst_hw_list, outs=None):
        """``cv2.resize(frame, (w, h), interpolation=cv2.INTER_AREA)`` per frame, shrinking only (kafka_sink.py:227-232).
        NV12 frames (``[3H/2, W]`` tensors, ``(y, uv)`` pairs or an ``Nv12Batch``) give the result of the BGR call on
        their ``cv2.cvtColor`` conversion; at their own size that is the conversion itself."""
        t = self.torch
        if outs is None:
            outs = [t.empty((int(h), int(w), 3), dtype=t.uint8, device=self.device) for h, w in dst_hw_list]
        elif any(tuple(o.shape) != (int(h), int(w), 3) or o.dtype != t.uint8 or not o.is_contiguous() or not o.is_cuda
                 for o, (h, w) in zip(outs, dst_hw_list)) or len(outs) != len(dst_hw_list):
            raise ValueError("resize_area: `outs` must be contiguous CUDA uint8 tensors [h, w, 3] matching dst_hw_list")
        fb = self._batch(frames, nv12_ok=True)
        hs, ws = _int_array([h for h, _ in dst_hw_list]), _int_array([w for _, w in dst_hw_list])
        if fb.n and isinstance(fb, Nv12Batch):
            self._check(self.lib.b200va_resize_area_u8_nv12(
                self._h, fb.nv, fb.hs, fb.ws, fb.n, _ptr_array([o.data_ptr() for o in outs]), hs, ws, self._stream()))
        elif fb.n:
            self._check(self.lib.b200va_resize_area_u8(
                self._h, fb.ptrs, fb.hs, fb.ws, fb.pitch, fb.n, _ptr_array([o.data_ptr() for o in outs]), hs, ws,
                self._stream()))
        return outs

    @staticmethod
    def pack_rects(ops_per_image):
        """``[(kind, x1, y1, x2, y2, (b, g, r)), ...]`` per image -> the ``b200va_rect_op`` array and offsets
        ``draw_rects`` passes down (pack once when the same overlay is drawn repeatedly)."""
        offs, flat = [0], []
        for ops in ops_per_image:
            flat.extend(ops)
            offs.append(len(flat))
        arr = (RectOp * max(len(flat), 1))()
        for i, (kind, x1, y1, x2, y2, col) in enumerate(flat):
            arr[i] = RectOp(int(kind), int(x1), int(y1), int(x2), int(y2), int(col[0]), int(col[1]), int(col[2]), 0)
        return arr, _int_array(offs), len(ops_per_image)

    def draw_rects(self, images, ops_per_image) -> None:
        """Draw, in place and in list order, ``(kind, x1, y1, x2, y2, (b, g, r))`` rectangles into CUDA uint8 [H, W, 3]
        images: kind 0 = ``cv2.rectangle(.., color, 2)``, kind 1 = ``cv2.rectangle(.., color, -1)`` (kafka_sink.py:240,
        249-255).  ``ops_per_image``: one list per image, or the result of ``pack_rects``."""
        fb = self._batch(images)
        if not fb.n:
            return
        arr, offs, n = ops_per_image if isinstance(ops_per_image, tuple) else self.pack_rects(ops_per_image)
        if n != fb.n:
            raise ValueError("draw_rects: one operation list per image")
        self._check(self.lib.b200va_draw_rects(self._h, fb.ptrs, fb.hs, fb.ws, fb.pitch, fb.n, arr, offs, self._stream()))

    # -- a9 ---------------------------------------------------------------------------------
    def roi_rasterize(self, polygons, height: int, width: int):
        """Union of ``cv2.fillPoly`` masks (frame_filter.py:46-49) -> CUDA uint8 [H, W]."""
        t = self.torch
        flat: List[int] = []
        sizes: List[int] = []
        for poly in polygons:
            sizes.append(len(poly))
            for x, y in poly:
                # np.array(polygon, dtype=np.int32) truncates toward zero
                flat.extend((int(x), int(y)))
        mask = t.empty((height, width), dtype=t.uint8, device=self.device)
        pts = (C.c_int32 * max(len(flat), 1))(*flat)
        self._check(self.lib.b200va_roi_rasterize(self._h, pts, _int_array(sizes) if sizes else None, len(sizes),
                                                  height, width, C.c_void_p(mask.data_ptr()), self._stream()))
        return mask

    def apply_mask(self, frame, mask, out=None):
        t = self.torch
        if out is None:
            out = t.empty((frame.shape[0], frame.shape[1], 3), dtype=t.uint8, device=self.device)
        self._check(self.lib.b200va_apply_mask(self._h, C.c_void_p(frame.data_ptr()), frame.stride(0),
                                               C.c_void_p(mask.data_ptr()), frame.shape[0], frame.shape[1],
                                               C.c_void_p(out.data_ptr()), out.stride(0), self._stream()))
        return out

    # -- a11 --------------------------------------------------------------------------------
    def motion(self, frames, prev_gray, next_gray, roi_masks=None, changed_out=None):
        """Blurred-gray update + changed-pixel counts.  ``prev_gray[i]`` may be None (first frame:
        count -1).  Returns the int32 device tensor of counts."""
        t = self.torch
        fb = self._batch(frames, roi_masks)
        b = fb.n
        if changed_out is None:
            changed_out = t.empty((b,), dtype=t.int32, device=self.device)
        if b:
            has_prev = _int_array([0 if p is None else 1 for p in prev_gray])
            self._check(self.lib.b200va_motion(
                self._h, fb.ptrs, fb.hs, fb.ws, fb.pitch, b, fb.mask_ptrs,
                _ptr_array([p.data_ptr() if p is not None else None for p in prev_gray]),
                _ptr_array([n.data_ptr() for n in next_gray]), has_prev, C.c_void_p(changed_out.data_ptr()),
                self._stream()))
        return changed_out

    # -- a11 + a1 fused -----------------------------------------------------------------------
    def motion_preprocess(self, frames, prev_gray, next_gray, dst_hw=(640, 640), fmt: int = OUT_F32_RGB_NCHW,
                          roi_masks=None, changed_out=None, out=None):
        """``motion`` and ``preprocess`` of the same frames in one pass over each frame.
        Returns (changed counts int32 [B], network input [B,3,H,W], list of Letterbox)."""
        t = self.torch
        fb = self._batch(frames, roi_masks)
        b = fb.n
        dh, dw = int(dst_hw[0]), int(dst_hw[1])
        dtype = {OUT_F32_RGB_NCHW: t.float32, OUT_F16_RGB_NCHW: t.float16}[fmt & 0xff]
        if out is None:
            out = t.empty((b, 3, dh, dw), dtype=dtype, device=self.device)
        elif tuple(out.shape) != (b, 3, dh, dw) or out.dtype != dtype or not out.is_contiguous():
            raise ValueError("motion_preprocess: `out` has the wrong shape / dtype / layout")
        if changed_out is None:
            changed_out = t.empty((b,), dtype=t.int32, device=self.device)
        if b:
            has_prev = _int_array([0 if p is None else 1 for p in prev_gray])
            self._check(self.lib.b200va_motion_preprocess(
                self._h, fb.ptrs, fb.hs, fb.ws, fb.pitch, b, fb.mask_ptrs,
                _ptr_array([p.data_ptr() if p is not None else None for p in prev_gray]),
                _ptr_array([n.data_ptr() for n in next_gray]), has_prev, C.c_void_p(changed_out.data_ptr()),
                C.c_void_p(out.data_ptr()), dh, dw, fmt, fb.metas, self._stream()))
        return changed_out, out, [fb.metas[i] for i in range(b)]

    # -- a3-a7 ------------------------------------------------------------------------------
    _DET_FIELDS = (("bbox_xyxy", "float32", 4), ("conf", "float32", 1), ("cls", "int32", 1))
    _TRK_FIELDS = (("bbox_xyxy", "float64", 4), ("track_id", "int64", 1), ("conf", "float64", 1), ("cls", "int32", 1),
                   ("age", "int32", 1), ("hits", "int32", 1))

    def _alloc_soa(self, fields, batch: int, rows: int, extra_counts, pinned_host: bool = False):
        """Structure-of-arrays carved from ONE flat byte buffer (field-major), so a whole result set
        moves device -> host in a single copy.  Returns {name: typed view, "_flat": bytes}."""
        t = self.torch
        sizes, off = [], 0
        for name, dtype, width in fields:
            nbytes = batch * rows * width * getattr(t, dtype).itemsize
            sizes.append((name, dtype, width, off, nbytes))
            off += (nbytes + 255) & ~255
        for name in extra_counts:
            sizes.append((name, "int32", 0, off, batch * 4))
            off += (batch * 4 + 255) & ~255
        flat = (t.zeros(off, dtype=t.uint8).pin_memory() if pinned_host
                else t.zeros(off, dtype=t.uint8, device=self.device))
        out = {"_flat": flat}
        for name, dtype, width, o, nbytes in sizes:
            v = flat[o:o + nbytes].view(getattr(t, dtype))
            out[name] = v.view(batch) if width == 0 else (v.view(batch, rows) if width == 1 else v.view(batch, rows, width))
        return out

    def alloc_dets(self, batch: int, pinned_host: bool = False):
        return self._alloc_soa(self._DET_FIELDS, batch, self.cfg.max_dets, ("count",), pinned_host)

    @staticmethod
    def _dets_struct(d) -> Dets:
        return Dets(d["bbox_xyxy"].data_ptr(), d["conf"].data_ptr(), d["cls"].data_ptr(), d["count"].data_ptr())

    def _head_args(self, head, layout):
        """(batch, layout | HEAD_F16 for a float16 head, channels, anchors) of a contiguous CUDA float32 / float16 head
        [B, C, A] (channel major) or [B, A, C] (anchor major).  layout=None: detector.py:282-283 -- transpose when
        shape[0] < shape[1]."""
        t = self.torch
        if not (head.is_cuda and head.dtype in (t.float32, t.float16) and head.dim() == 3 and head.is_contiguous()):
            raise ValueError("head must be a contiguous CUDA float32 / float16 tensor [B, C, A] or [B, A, C]")
        b, d1, d2 = head.shape
        if layout is None:
            layout = HEAD_CHANNEL_MAJOR if (d1 != 0 and d1 < d2) else HEAD_ANCHOR_MAJOR
        layout &= ~HEAD_F16
        channels, anchors = (d1, d2) if layout == HEAD_CHANNEL_MAJOR else (d2, d1)
        return b, layout | (HEAD_F16 if head.dtype == t.float16 else 0), channels, anchors

    def postprocess(self, head, metas, conf_thr: float, iou_thr: float, classes=None, layout=None,
                    filter_conf: Optional[float] = None, out=None, score_mode: int = SCORE_REF_COMPAT,
                    nms_mode: int = NMS_AGNOSTIC):
        """Decode + filter + NMS for ``head`` [B,C,A] (channel major) or [B,A,C] (anchor major), float32 or float16
        (read in place: the same results as ``head.float()``)."""
        b, layout, channels, anchors = self._head_args(head, layout)
        if out is None:
            out = self.alloc_dets(b)
        marr = metas if isinstance(metas, C.Array) else (Letterbox * max(b, 1))(*metas)
        cls_arr = (C.c_int32 * len(classes))(*[int(c) for c in classes]) if classes else None
        ds = self._dets_struct(out)
        self._check(self.lib.b200va_postprocess(
            self._h, C.c_void_p(head.data_ptr()), layout, b, channels, anchors, marr, float(conf_thr), float(iou_thr),
            cls_arr, len(classes) if classes else 0, int(score_mode), int(nms_mode),
            float(filter_conf) if filter_conf is not None else 0.0, 1 if filter_conf is not None else 0,
            C.byref(ds), self._stream()))
        return out

    # -- Ultralytics semantics (SURVEY 8f row 2) ---------------------------------------------
    def preprocess_geom(self, frames, geoms, dst_hw, fmt: int = OUT_F32_RGB_NCHW, roi_masks=None, out=None):
        """Letterbox with caller-supplied geometry (``geoms``: one ``Letterbox`` per frame, e.g. from
        ``letterbox_meta_ultralytics``) into a ``dst_hw`` canvas."""
        t = self.torch
        fb = self._batch(frames, roi_masks)
        b = fb.n
        dh, dw = int(dst_hw[0]), int(dst_hw[1])
        dtype = {OUT_F32_RGB_NCHW: t.float32, OUT_F16_RGB_NCHW: t.float16}.get(fmt & 0xff, t.uint8)
        shape = (b, dh, dw, 3) if (fmt & 0xff) == OUT_U8_BGR_NHWC else (b, 3, dh, dw)
        if out is None:
            out = t.empty(shape, dtype=dtype, device=self.device)
        elif tuple(out.shape) != shape or out.dtype != dtype or not out.is_contiguous():
            raise ValueError("preprocess_geom: `out` has the wrong shape / dtype / layout")
        garr = geoms if isinstance(geoms, C.Array) else (Letterbox * max(b, 1))(*geoms)
        if b:
            self._check(self.lib.b200va_preprocess_geom(self._h, fb.ptrs, fb.hs, fb.ws, fb.pitch, b, fb.mask_ptrs, garr,
                                                        C.c_void_p(out.data_ptr()), dh, dw, fmt, self._stream()))
        return out

    def postprocess_ultralytics(self, head, frame_hw, in_hw, conf_thr: float = 0.25, iou_thr: float = 0.45, classes=None,
                                agnostic: bool = False, max_det: int = 300, layout=None,
                                filter_conf: Optional[float] = None, out=None):
        """``ops.non_max_suppression`` + ``ops.scale_boxes`` for ``head`` [B, 4 + nc, A] (or [B, A, 4 + nc]).
        ``frame_hw``: (h, w) of every original frame; ``in_hw``: the network-input shape the head came from."""
        b, layout, channels, anchors = self._head_args(head, layout)
        if out is None:
            out = self.alloc_dets(b)
        cls_arr = (C.c_int32 * len(classes))(*[int(c) for c in classes]) if classes else None
        ds = self._dets_struct(out)
        self._check(self.lib.b200va_postprocess_ultralytics(
            self._h, C.c_void_p(head.data_ptr()), layout, b, channels, anchors, _int_array([hw[0] for hw in frame_hw]),
            _int_array([hw[1] for hw in frame_hw]), int(in_hw[0]), int(in_hw[1]), float(conf_thr), float(iou_thr), cls_arr,
            len(classes) if classes else 0, 1 if agnostic else 0, int(max_det),
            float(filter_conf) if filter_conf is not None else 0.0, 1 if filter_conf is not None else 0, C.byref(ds),
            self._stream()))
        return out

    # -- a14 --------------------------------------------------------------------------------
    def dfl_decode(self, raw, num_classes: int, reg_max: int = 16, levels=((80, 80), (40, 40), (20, 20)),
                   strides=(8.0, 16.0, 32.0), out=None):
        """Raw Detect head [B, 4*reg_max + nc, A] -> decoded [B, 4 + nc, A] (within a derived float32 error bound of
        the float64 decode, tests/dfl_bound.py)."""
        t = self.torch
        b = raw.shape[0]
        a = sum(h * w for h, w in levels)
        if len(strides) != len(levels):
            raise ValueError("dfl_decode: one stride per level")
        if not (raw.is_cuda and raw.dtype == t.float32 and raw.is_contiguous()
                and tuple(raw.shape) == (b, 4 * reg_max + num_classes, a)):
            raise ValueError("raw must be a contiguous CUDA float32 tensor [B, 4*reg_max + nc, sum(h*w)]")
        if out is None:
            out = t.empty((b, 4 + num_classes, a), dtype=t.float32, device=self.device)
        elif not (out.is_cuda and out.device == self.device and out.dtype == t.float32 and out.is_contiguous()
                  and tuple(out.shape) == (b, 4 + num_classes, a)):
            raise ValueError("dfl_decode: `out` must be a contiguous float32 tensor [B, 4 + nc, sum(h*w)] on the "
                             "handle's device")
        hw = _int_array([v for lv in levels for v in lv])
        st = (C.c_float * len(strides))(*[float(s) for s in strides])
        self._check(self.lib.b200va_dfl_decode(self._h, C.c_void_p(raw.data_ptr()), b, int(num_classes), int(reg_max),
                                               hw, st, len(levels), C.c_void_p(out.data_ptr()), self._stream()))
        return out

    # -- a8 ---------------------------------------------------------------------------------
    def alloc_tracks(self, batch: int, pinned_host: bool = False, rows: Optional[int] = None):
        """Track result tables.  ``rows`` (default ``max_tracks``) is how many rows per stream the caller wants back:
        the state always holds up to ``max_tracks``; ``count`` reports the true number and a capacity flag is raised
        when it exceeds ``rows``."""
        rows = self.cfg.max_tracks if rows is None else max(1, min(int(rows), self.cfg.max_tracks))
        return self._alloc_soa(self._TRK_FIELDS, batch, rows, ("count", "new_count"), pinned_host)

    @staticmethod
    def _tracks_struct(out) -> Tracks:
        return Tracks(out["track_id"].data_ptr(), out["cls"].data_ptr(), out["conf"].data_ptr(), out["bbox_xyxy"].data_ptr(),
                      out["age"].data_ptr(), out["hits"].data_ptr(), out["count"].data_ptr(), int(out["track_id"].shape[1]))

    def tracker_update(self, slots, dets, max_age: int, min_hits: int, max_iou_distance: float, det_scale=None,
                       skip=None, id_base=None, out=None, f64: bool = False):
        b = len(slots)
        if out is None:
            out = self.alloc_tracks(b)
        cfg = TrackerCfg(int(max_age), int(min_hits), float(max_iou_distance))
        slot_arr = slots if isinstance(slots, C.Array) else _int_array(slots)
        ts = self._tracks_struct(out)
        skip_arr = (C.c_uint8 * b)(*[1 if s else 0 for s in skip]) if skip is not None else None
        idb = (C.c_int64 * b)(*[int(v) for v in id_base]) if id_base is not None else None
        max_dets = int(dets["conf"].shape[1])
        if f64:
            ds = Dets64(dets["bbox_xyxy"].data_ptr(), dets["conf"].data_ptr(), dets["cls"].data_ptr(),
                        dets["count"].data_ptr())
            self._check(self.lib.b200va_tracker_update_f64(self._h, slot_arr, b, C.byref(ds), max_dets,
                                                           skip_arr, C.byref(cfg), idb, C.byref(ts),
                                                           C.c_void_p(out["new_count"].data_ptr()), self._stream()))
        else:
            ds = self._dets_struct(dets)
            sc = (C.c_double * b)(*[float(v) for v in det_scale]) if det_scale is not None else None
            self._check(self.lib.b200va_tracker_update(self._h, slot_arr, b, C.byref(ds), max_dets, sc,
                                                       skip_arr, C.byref(cfg), idb, C.byref(ts),
                                                       C.c_void_p(out["new_count"].data_ptr()), self._stream()))
        return out

    # -- one tick: letterbox || decode + NMS + tracker -----------------------------------------
    def plan_tick(self, frames=None, net_out=None, dst_hw=(640, 640), fmt: int = OUT_F32_RGB_NCHW, roi_masks=None,
                  head=None, metas=None, conf_thr: float = 0.25, iou_thr: float = 0.45, classes=None, layout=None,
                  filter_conf: Optional[float] = None, dets=None, score_mode: int = SCORE_REF_COMPAT,
                  nms_mode: int = NMS_AGNOSTIC, slots=None, tracker_cfg=None, det_scale=None, skip=None,
                  tracks=None, schedule: int = SCHEDULE_AUTO) -> TickPlan:
        """Prepare a ``b200va_tick``: the letterbox of ``frames`` into ``net_out`` and the post-process
        of ``head`` into ``dets`` followed by the tracker update of ``slots`` into ``tracks``.  Either
        half may be omitted.  ``tracker_cfg`` = (max_age, min_hits, max_iou_distance)."""
        t = self.torch
        a = TickArgs()
        keep = []
        if frames is not None:
            fb = self._batch(frames, roi_masks, nv12_ok=True)
            dh, dw = int(dst_hw[0]), int(dst_hw[1])
            dtype = {OUT_F32_RGB_NCHW: t.float32, OUT_F16_RGB_NCHW: t.float16}.get(fmt & 0xff, t.uint8)
            shape = (fb.n, dh, dw, 3) if (fmt & 0xff) == OUT_U8_BGR_NHWC else (fb.n, 3, dh, dw)
            if net_out is None or tuple(net_out.shape) != shape or net_out.dtype != dtype or not net_out.is_contiguous():
                raise ValueError("plan_tick: `net_out` must be a contiguous tensor of the letterbox output shape / dtype")
            if isinstance(fb, Nv12Batch):
                a.src_h, a.src_w, a.batch = fb.hs, fb.ws, fb.n
            else:
                a.frames, a.src_h, a.src_w, a.src_pitch, a.batch = fb.ptrs, fb.hs, fb.ws, fb.pitch, fb.n
            a.roi_masks = fb.mask_ptrs
            a.net_out, a.dst_h, a.dst_w, a.out_format, a.meta_out = net_out.data_ptr(), dh, dw, fmt, fb.metas
            keep += [fb, net_out]
        if head is not None:
            b, layout, channels, anchors = self._head_args(head, layout)
            marr = metas if isinstance(metas, C.Array) else (Letterbox * max(b, 1))(*metas)
            cls_arr = (C.c_int32 * len(classes))(*[int(c) for c in classes]) if classes else None
            if dets is None:
                dets = self.alloc_dets(b)
            ds = self._dets_struct(dets)
            a.head, a.layout, a.head_batch, a.channels, a.anchors = head.data_ptr(), layout, b, channels, anchors
            a.meta, a.conf_thr, a.iou_thr = marr, float(conf_thr), float(iou_thr)
            a.classes, a.n_classes = cls_arr, len(classes) if classes else 0
            a.score_mode, a.nms_mode = int(score_mode), int(nms_mode)
            a.filter_conf_thr_f64 = float(filter_conf) if filter_conf is not None else 0.0
            a.use_filter = 1 if filter_conf is not None else 0
            a.dets = C.pointer(ds)
            keep += [head, marr, cls_arr, dets, ds]
        if slots is not None:
            if dets is None or tracker_cfg is None:
                raise ValueError("plan_tick: the tracker half needs `dets` and `tracker_cfg`")
            b = len(slots)
            if tracks is None:
                tracks = self.alloc_tracks(b)
            if not a.dets:
                ds = self._dets_struct(dets)
                a.dets = C.pointer(ds)
                keep.append(ds)
            cfg = TrackerCfg(int(tracker_cfg[0]), int(tracker_cfg[1]), float(tracker_cfg[2]))
            slot_arr = slots if isinstance(slots, C.Array) else _int_array(slots)
            ts = self._tracks_struct(tracks)
            sc = (C.c_double * b)(*[float(v) for v in det_scale]) if det_scale is not None else None
            skip_arr = (C.c_uint8 * b)(*[1 if s else 0 for s in skip]) if skip is not None else None
            a.stream_slots, a.trk_batch, a.max_dets = slot_arr, b, int(dets["conf"].shape[1])
            a.det_scale, a.skip, a.trk_cfg, a.id_base = sc, skip_arr, C.pointer(cfg), None
            a.tracks, a.new_counts = C.pointer(ts), tracks["new_count"].data_ptr()
            keep += [slot_arr, ts, sc, skip_arr, cfg, tracks, dets]
        a.schedule = int(schedule)
        plan = TickPlan(a, tuple(keep))
        plan.dets, plan.tracks = dets, tracks
        if frames is not None and isinstance(fb, Nv12Batch):
            plan.nv12 = fb.nv
        return plan

    def tick(self, plan: TickPlan) -> None:
        """Run a prepared tick on the current stream (results land in the plan's buffers)."""
        if plan.nv12 is not None:
            self._check(self.lib.b200va_tick_nv12(self._h, C.byref(plan.args), plan.nv12, self._stream()))
        else:
            self._check(self.lib.b200va_tick(self._h, C.byref(plan.args), self._stream()))

    # -- a12 on the device: gates --------------------------------------------------------------
    def gates_decide(self, gates, changed, skip_out) -> None:
        """``gates``: a ctypes array of ``Gate``; ``changed``: the int32 device tensor ``motion`` returned (or None);
        ``skip_out``: uint8 device tensor [len(gates)] receiving GATE_PROCESS / GATE_SKIP_MOTION / GATE_SKIP_ADAPTIVE."""
        self._check(self.lib.b200va_gates_decide(self._h, gates, len(gates),
                                                 C.c_void_p(changed.data_ptr()) if changed is not None else None,
                                                 C.c_void_p(skip_out.data_ptr()), self._stream()))

    def gates_commit(self, gates, det_count, trk_count, skip, state_out) -> None:
        """``_adjust_adaptive_state`` on the device; ``state_out``: int32 device tensor [len(gates), 4] =
        (skip flag, process_every, idle_frames, frame_index)."""
        self._check(self.lib.b200va_gates_commit(self._h, gates, len(gates), C.c_void_p(det_count.data_ptr()),
                                                 C.c_void_p(trk_count.data_ptr()),
                                                 C.c_void_p(skip.data_ptr()) if skip is not None else None,
                                                 C.c_void_p(state_out.data_ptr()) if state_out is not None else None,
                                                 self._stream()))

    def gates_reset(self, slot: int) -> None:
        self._check(self.lib.b200va_gates_reset(self._h, int(slot), self._stream()))

    def set_skip_mask(self, skip) -> None:
        """Device uint8 tensor (one flag per batch position) read by the kernels of every later preprocess /
        postprocess / tracker_update / tick call, or None to switch the mask off.  The caller keeps the tensor alive."""
        self._skip_mask = skip
        self._check(self.lib.b200va_set_skip_mask(self._h, C.c_void_p(skip.data_ptr()) if skip is not None else None))

    def tracker_reset(self, slot: int) -> None:
        self._check(self.lib.b200va_tracker_reset(self._h, int(slot), self._stream()))

    def tracker_set_next_id(self, next_id: int) -> None:
        self._check(self.lib.b200va_tracker_set_next_id(self._h, int(next_id), self._stream()))
