"""CPU restatement of the reference's per-frame hot path (pre -> post -> track, ROI, motion).

TEST INFRASTRUCTURE ONLY -- see ``oracle/__init__.py``.  The product package never
imports this module; it exists so that ``tests/`` can check the CUDA path bit-for-bit,
``__graft_entry__.smoke()`` can self-check, and ``bench.py`` can report a CPU baseline.

Every function cites the reference lines (relative to ``/root/reference``) it restates.
The restatement is pinned by ``tests/golden/*.npz``: vectors produced by importing and
running the reference's own functions in the build container
(``tests/golden/make_golden.py``); ``tests/test_oracle_golden.py`` replays them.

Two arithmetic back ends are available for the OpenCV calls:

* ``backend="numpy"``  -- the bit-exact NumPy restatements in ``oracle/cv_restate.py``.
* ``backend="cv2"``    -- the same call sequence the reference issues, through the
  installed OpenCV.  Used for the reported CPU baseline (it is what the reference's CPU
  path actually costs) and cross-checked against the NumPy back end.
"""

from __future__ import annotations

import itertools
from dataclasses import dataclass, field
from typing import Dict, Iterable, List, Optional, Sequence, Tuple

import numpy as np

from . import cv_restate as cvr

F32 = np.float32


# --------------------------------------------------------------------------------------
# plain result records (the reference's Detection / Track dataclasses, detector.py:32-40,
# tracker.py:18-33, reduced to the fields the hot path produces)
# --------------------------------------------------------------------------------------
@dataclass
class Det:
    class_id: int
    confidence: float
    bbox_xyxy: Tuple[float, float, float, float]


@dataclass
class Trk:
    track_id: int
    class_id: int
    confidence: float
    bbox_xyxy: Tuple[float, float, float, float]
    age: int = 0
    hits: int = 0


# --------------------------------------------------------------------------------------
# a1: letterbox preprocess -- detector.py:198-264
# --------------------------------------------------------------------------------------
def letterbox_meta(h: int, w: int, in_h: int, in_w: int) -> dict:
    """Geometry of the letterbox: detector.py:209-230, 259-263."""
    scale = min(in_w / w, in_h / h)  # Python float64, :211
    new_w = int(w * scale)  # truncation, :214
    new_h = int(h * scale)  # :215
    pad_w = in_w - new_w
    pad_h = in_h - new_h
    top = pad_h // 2
    left = pad_w // 2
    return {
        "orig_shape": (h, w),
        "scale": scale,
        "pad": (left, top),
        "new_wh": (new_w, new_h),
    }


def preprocess(frame: np.ndarray, input_hw=(640, 640), half: bool = False, backend: str = "numpy"):
    """``_TensorRTBaseDetector._preprocess`` (detector.py:198-264).

    resize INTER_LINEAR -> constant pad 114 -> BGR2RGB -> astype * (1/255) -> CHW + batch.
    """
    h, w = frame.shape[:2]
    in_h, in_w = input_hw
    meta = letterbox_meta(h, w, in_h, in_w)
    new_w, new_h = meta["new_wh"]
    left, top = meta["pad"]
    if backend == "cv2":
        import cv2

        resized = cv2.resize(frame, (new_w, new_h), interpolation=cv2.INTER_LINEAR)
    else:
        resized = cvr.resize_linear_u8(frame, new_w, new_h)
    canvas = np.full((in_h, in_w, 3), 114, dtype=np.uint8)  # copyMakeBorder, :233-241
    canvas[top:top + new_h, left:left + new_w] = resized
    rgb = canvas[:, :, ::-1]  # cvtColor BGR2RGB, :245
    dtype = np.float16 if half else np.float32
    # NumPy weak-scalar promotion: the Python float 1/255 is rounded to ``dtype`` first (:248-251)
    image = rgb.astype(dtype) * dtype(1.0 / 255.0)
    tensor = np.ascontiguousarray(np.transpose(image, (2, 0, 1)))[None]
    meta_out = {k: meta[k] for k in ("orig_shape", "scale", "pad")}
    return tensor, meta_out


def preprocess_u8(frame: np.ndarray, input_hw=(640, 640), nhwc: bool = True, backend: str = "numpy"):
    """``RKNNDetector._preprocess`` (detector.py:777-839): same letterbox, stays BGR uint8."""
    h, w = frame.shape[:2]
    in_h, in_w = input_hw
    meta = letterbox_meta(h, w, in_h, in_w)
    new_w, new_h = meta["new_wh"]
    left, top = meta["pad"]
    if backend == "cv2":
        import cv2

        resized = cv2.resize(frame, (new_w, new_h), interpolation=cv2.INTER_LINEAR)
    else:
        resized = cvr.resize_linear_u8(frame, new_w, new_h)
    canvas = np.full((in_h, in_w, 3), 114, dtype=np.uint8)
    canvas[top:top + new_h, left:left + new_w] = resized
    out = canvas if nhwc else np.ascontiguousarray(np.transpose(canvas, (2, 0, 1)))
    return out[None], {k: meta[k] for k in ("orig_shape", "scale", "pad")}


# --------------------------------------------------------------------------------------
# a3-a6: head post-process -- detector.py:266-375, 469-481
# --------------------------------------------------------------------------------------
def pairwise_iou_f32(boxes: np.ndarray) -> np.ndarray:
    """IoU of every pair with the op order of ``_iou`` (detector.py:469-481), float32."""
    b = boxes.astype(F32, copy=False)
    x1 = np.maximum(b[:, None, 0], b[None, :, 0])
    y1 = np.maximum(b[:, None, 1], b[None, :, 1])
    x2 = np.minimum(b[:, None, 2], b[None, :, 2])
    y2 = np.minimum(b[:, None, 3], b[None, :, 3])
    inter = np.maximum(F32(0), x2 - x1) * np.maximum(F32(0), y2 - y1)
    area = (b[:, 2] - b[:, 0]) * (b[:, 3] - b[:, 1])
    union = (area[:, None] + area[None, :]) - inter
    return inter / np.maximum(union, F32(1e-6))


def nms_order(scores: np.ndarray) -> np.ndarray:
    """``scores.argsort()[::-1]`` (detector.py:365) with the tie rule fixed to what a stable
    ascending sort gives after reversal (equal scores: higher index first).  NumPy's
    default sort is unspecified on ties; tie-free inputs are order-identical."""
    return np.argsort(scores, kind="stable")[::-1]


def nms(boxes: np.ndarray, scores: np.ndarray, iou_threshold: float, cls: Optional[np.ndarray] = None) -> List[int]:
    """Greedy class-agnostic NMS, detector.py:361-375: keep the best, drop every remaining
    box whose IoU with it is ``> float32(iou_threshold)``.

    ``cls`` (not a reference feature; the additive CLASS_AWARE mode of the C ABI): a kept box only
    suppresses boxes of its own class."""
    n = len(boxes)
    if n == 0:
        return []
    order = nms_order(scores)
    sb = boxes[order]
    iou = pairwise_iou_f32(sb)
    thr = F32(iou_threshold)
    hit = ~(iou <= thr)
    if cls is not None:
        sc = np.asarray(cls)[order]
        hit &= sc[:, None] == sc[None, :]
    suppressed = np.zeros(n, dtype=bool)
    keep: List[int] = []
    for i in range(n):
        if suppressed[i]:
            continue
        keep.append(int(order[i]))
        suppressed[i + 1:] |= hit[i, i + 1:]
    return keep


def decode_candidates(pred: np.ndarray, conf_thr: float, classes: Optional[Sequence[int]], v8_native: bool = False,
                      layout: Optional[str] = None):
    """detector.py:278-317: layout fix-up, objectness x class score, argmax, filters.

    ``layout`` (not a reference feature; the explicit ``layout`` argument of the C ABI): ``"cm"`` for a
    [C, A] head, ``"am"`` for [A, C]; None applies the reference's rule (transpose when rows < columns),
    which calls a head with A <= C anchor-major.

    Returns (xywh[N,4] f32, conf[N] f32, cls[N] int64, anchor_index[N]) or None for the
    "unexpected shape" early-out (:285-287).
    """
    if isinstance(pred, list):
        pred = pred[0]
    if pred.ndim == 3:
        if pred.shape[0] != 1:
            raise ValueError("cannot select an axis to squeeze out which has size not equal to one")
        pred = pred[0]
    if layout is None:
        if pred.shape[0] != 0 and pred.shape[0] < pred.shape[1]:
            pred = pred.T
    elif layout == "cm":
        pred = pred.T
    elif layout != "am":
        raise ValueError(f"unknown layout {layout!r}")
    if pred.ndim != 2 or pred.shape[1] < 5:
        return None
    pred = pred.astype(F32, copy=False)
    boxes = pred[:, :4]
    if v8_native:  # additive V8_NATIVE mode of the C ABI (not the reference's rule)
        scores = pred[:, 4:]
    elif pred.shape[1] > 5:
        scores = pred[:, 5:] * pred[:, 4:5]  # both model types, :294-305
    else:
        scores = pred[:, 4:]
    cls = np.argmax(scores, axis=1)
    conf = scores[np.arange(scores.shape[0]), cls]
    mask = conf >= F32(conf_thr)
    if classes:
        mask &= np.isin(cls, np.array(classes))
    idx = np.nonzero(mask)[0]
    return boxes[idx], conf[idx], cls[idx], idx


def xywh2xyxy(b: np.ndarray) -> np.ndarray:
    """detector.py:352-359."""
    half_w = b[:, 2] / F32(2.0)
    half_h = b[:, 3] / F32(2.0)
    return np.stack([b[:, 0] - half_w, b[:, 1] - half_h, b[:, 0] + half_w, b[:, 1] + half_h], axis=1).astype(F32)


def scale_boxes(b: np.ndarray, meta: dict) -> np.ndarray:
    """detector.py:340-350: un-pad, true division by float32(scale), clip to the frame."""
    left, top = meta["pad"]
    oh, ow = meta["orig_shape"]
    s = F32(meta["scale"])
    out = b.astype(F32).copy()
    out[:, 0] = np.clip((out[:, 0] - F32(left)) / s, F32(0), F32(ow - 1))
    out[:, 2] = np.clip((out[:, 2] - F32(left)) / s, F32(0), F32(ow - 1))
    out[:, 1] = np.clip((out[:, 1] - F32(top)) / s, F32(0), F32(oh - 1))
    out[:, 3] = np.clip((out[:, 3] - F32(top)) / s, F32(0), F32(oh - 1))
    return out


def postprocess(pred: np.ndarray, meta: dict, conf_thr: float, iou_thr: float,
                classes: Optional[Sequence[int]] = None, v8_native: bool = False, class_aware: bool = False,
                layout: Optional[str] = None) -> List[Det]:
    """``_TensorRTBaseDetector._postprocess`` (detector.py:266-338); output in keep order.
    ``v8_native`` / ``class_aware`` / ``layout`` select the additive modes (all default = the reference)."""
    cand = decode_candidates(pred, conf_thr, classes, v8_native, layout)
    if cand is None:
        return []
    xywh, conf, cls, _ = cand
    if xywh.size == 0:
        return []
    boxes = scale_boxes(xywh2xyxy(xywh), meta)
    keep = nms(boxes, conf, iou_thr, cls if class_aware else None)
    return [
        Det(int(cls[i]), float(conf[i]), (float(boxes[i, 0]), float(boxes[i, 1]), float(boxes[i, 2]), float(boxes[i, 3])))
        for i in keep
    ]


def filter_detections(dets: Iterable[Det], min_confidence: float) -> List[Det]:
    """detector.py:99-103 -- a float64 comparison against the un-rounded threshold."""
    return [d for d in dets if d.confidence >= min_confidence]


def rescale_detections(dets: List[Det], ratio: float) -> List[Det]:
    """``StreamWorker._rescale_detections`` pipeline.py:224-240 (float64 multiply)."""
    if ratio >= 0.999:
        return dets
    s = 1.0 / max(ratio, 1e-6)
    return [Det(d.class_id, d.confidence, tuple(v * s for v in d.bbox_xyxy)) for d in dets]


# --------------------------------------------------------------------------------------
# a8: IoU tracker -- tracker.py:36-147
# --------------------------------------------------------------------------------------
def iou_f64(a, b) -> float:
    """tracker.py:129-147 (Python floats = IEEE double)."""
    iw = max(0.0, min(a[2], b[2]) - max(a[0], b[0]))
    ih = max(0.0, min(a[3], b[3]) - max(a[1], b[1]))
    inter = iw * ih
    area_a = max(0.0, a[2] - a[0]) * max(0.0, a[3] - a[1])
    area_b = max(0.0, b[2] - b[0]) * max(0.0, b[3] - b[1])
    union = area_a + area_b - inter
    if union <= 0:
        return 0.0
    return inter / union


class IouTracker:
    """Sequential greedy tracker of tracker.py:36-126 (one shared id counter, :47)."""

    def __init__(self, max_age: int = 30, max_iou_distance: float = 0.7, min_hits: int = 3):
        self.max_age = max_age
        self.max_iou_distance = max_iou_distance
        self.min_hits = min_hits
        self._ids = itertools.count(1)
        self._tracks: Dict[str, List[Trk]] = {}  # insertion-ordered, like the reference dict

    def update(self, stream_name: str, detections: Iterable[Det]) -> List[Trk]:
        tracks = self._tracks.setdefault(stream_name, [])
        touched = set()
        for det in detections:
            best, best_iou = None, 0.0
            for t in tracks:  # dict order == insertion order, tracker.py:102
                if t.class_id != det.class_id:
                    continue
                v = iou_f64(t.bbox_xyxy, det.bbox_xyxy)
                if v >= self.max_iou_distance and v > best_iou:
                    best, best_iou = t, v
            if best is None:  # tracker.py:69-80: new track, matchable at once
                best = Trk(next(self._ids), det.class_id, det.confidence, tuple(det.bbox_xyxy), age=0, hits=1)
                tracks.append(best)
            else:  # tracker.py:82-92: overwrite immediately
                best.bbox_xyxy = tuple(det.bbox_xyxy)
                best.confidence = det.confidence
                best.hits += 1
                best.age = 0
            touched.add(best.track_id)
        survivors = []
        for t in tracks:  # tracker.py:111-126
            if t.track_id not in touched:
                t.age += 1
                if t.age > self.max_age or t.hits < self.min_hits:
                    continue
            survivors.append(t)
        self._tracks[stream_name] = survivors
        return list(survivors)


# --------------------------------------------------------------------------------------
# a9-a11: frame filters -- utils/frame_filter.py
# --------------------------------------------------------------------------------------
def roi_mask(shape_hw, polygons, backend: str = "numpy") -> np.ndarray:
    """frame_filter.py:46-49: union of one ``fillPoly`` per polygon."""
    h, w = shape_hw
    if backend == "cv2":
        import cv2

        m = np.zeros((h, w), dtype=np.uint8)
        for poly in polygons:
            cv2.fillPoly(m, [np.array(poly, dtype=np.int32)], 255)
        return m
    return cvr.fill_poly_mask(h, w, polygons)


def apply_roi(frame: np.ndarray, polygons, backend: str = "numpy") -> np.ndarray:
    """frame_filter.py:43-50."""
    if not polygons:
        return frame
    mask = roi_mask(frame.shape[:2], polygons, backend)
    if backend == "cv2":
        import cv2

        return cv2.bitwise_and(frame, frame, mask=mask)
    return cvr.apply_mask(frame, mask)


def downsample(frame: np.ndarray, scale: float, backend: str = "numpy") -> np.ndarray:
    """frame_filter.py:53-57."""
    if scale >= 0.999:
        return frame
    h, w = frame.shape[:2]
    dw, dh = int(w * scale), int(h * scale)
    if backend == "cv2":
        import cv2

        return cv2.resize(frame, (dw, dh), interpolation=cv2.INTER_LINEAR)
    return cvr.resize_linear_u8(frame, dw, dh)


class MotionFilter:
    """frame_filter.py:19-40.  ``last_count`` exposes the changed-pixel count for tests."""

    def __init__(self, threshold: float = 0.02, backend: str = "numpy"):
        self.threshold = threshold
        self.backend = backend
        self.previous_gray: Optional[np.ndarray] = None
        self.last_count: Optional[int] = None

    def _blurred_gray(self, frame):
        if self.backend == "cv2":
            import cv2

            return cv2.GaussianBlur(cv2.cvtColor(frame, cv2.COLOR_BGR2GRAY), (5, 5), 0)
        return cvr.gaussian_blur5(cvr.bgr2gray(frame))

    def should_process(self, frame: np.ndarray) -> bool:
        gray = self._blurred_gray(frame)
        if self.previous_gray is None:
            self.previous_gray = gray
            self.last_count = None
            return True
        if self.backend == "cv2":
            import cv2

            _, th = cv2.threshold(cv2.absdiff(gray, self.previous_gray), 25, 255, cv2.THRESH_BINARY)
            count = int(np.count_nonzero(th))
        else:
            count = cvr.motion_changed_count(gray, self.previous_gray)
        self.last_count = count
        ratio = float(count) / float(gray.size)
        self.previous_gray = gray
        return ratio >= self.threshold


# --------------------------------------------------------------------------------------
# a12: per-stream driver state machine -- pipeline.py:88-262
# --------------------------------------------------------------------------------------
@dataclass
class StreamSpec:
    """The StreamConfig knobs the hot path reads (config.py:61-73)."""

    name: str
    roi_polygons: Optional[list] = None
    motion_filter: bool = False
    motion_threshold: float = 0.02
    downsample_ratio: float = 1.0
    adaptive_fps: bool = False
    target_fps: Optional[float] = None
    min_target_fps: float = 5.0
    idle_frame_tolerance: int = 60


@dataclass
class FrameResult:
    processed: bool
    detections: List[Det] = field(default_factory=list)
    tracks: List[Trk] = field(default_factory=list)
    skip_reason: Optional[str] = None


class StreamWorker:
    """``StreamWorker._process_packet`` and helpers (pipeline.py:88-262) without the I/O:
    ROI -> downsample -> motion gate -> adaptive-FPS gate -> predict -> rescale ->
    float64 re-threshold -> tracker -> adaptive state update."""

    def __init__(self, spec: StreamSpec, infer, tracker: IouTracker, conf_thr: float, iou_thr: float,
                 classes=None, input_hw=(640, 640), half=False, backend: str = "numpy"):
        self.spec = spec
        self.infer = infer  # callable(tensor[1,3,H,W], frame_index) -> head ndarray
        self.tracker = tracker
        self.conf_thr, self.iou_thr, self.classes = conf_thr, iou_thr, classes
        self.input_hw, self.half, self.backend = input_hw, half, backend
        self.motion: Optional[MotionFilter] = None
        self.frame_index = 0
        self.idle_frames = 0
        self.process_every = 1
        if spec.adaptive_fps:  # pipeline.py:107-113
            target = spec.target_fps or 30.0
            min_fps = max(spec.min_target_fps, 1.0)
            self.max_process_every = max(1, int(round(target / min_fps)))
            self.idle_tolerance = max(int(spec.idle_frame_tolerance), 1)
        else:
            self.max_process_every = 1
            self.idle_tolerance = 0

    def _adjust(self, n_det: int, n_trk: int) -> None:  # pipeline.py:242-262
        if not self.spec.adaptive_fps:
            return
        if n_det > 0 or n_trk > 0:
            self.idle_frames = 0
            self.process_every = 1
        else:
            self.idle_frames += 1
            if self.idle_frames >= self.idle_tolerance:
                self.process_every = max(self.max_process_every, 1)

    def _skip(self, reason: str) -> FrameResult:  # pipeline.py:214-222
        tracks = self.tracker.update(self.spec.name, [])
        self._adjust(0, len(tracks))
        return FrameResult(False, [], tracks, reason)

    def process(self, frame: np.ndarray) -> FrameResult:  # pipeline.py:143-201
        self.frame_index += 1
        f = frame
        if self.spec.roi_polygons:
            f = apply_roi(f, self.spec.roi_polygons, self.backend)
        ratio = self.spec.downsample_ratio
        if ratio < 0.999:
            f = downsample(f, ratio, self.backend)
        if self.spec.motion_filter:
            if self.motion is None:
                self.motion = MotionFilter(self.spec.motion_threshold, self.backend)
            if not self.motion.should_process(f):
                return self._skip("motion")
        if self.spec.adaptive_fps and self.process_every > 1:
            if (self.frame_index - 1) % self.process_every != 0:
                return self._skip("adaptive")
        tensor, meta = preprocess(f, self.input_hw, self.half, self.backend)
        head = self.infer(tensor, self.frame_index)
        dets = postprocess(head, meta, self.conf_thr, self.iou_thr, self.classes)
        if ratio < 0.999:
            dets = rescale_detections(dets, ratio)
        dets = filter_detections(dets, self.conf_thr)
        tracks = self.tracker.update(self.spec.name, dets)
        self._adjust(len(dets), len(tracks))
        return FrameResult(True, dets, tracks, None)
