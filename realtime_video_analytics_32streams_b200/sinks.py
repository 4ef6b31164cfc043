"""Egress plug-in: the reference's ``KafkaSink`` contract (sinks/kafka_sink.py:30-310) with the per-pixel work and the
serialisation done by ``libb200va`` (SURVEY.md §8f-3).

``B200KafkaSink`` keeps the reference's constructor, ``connect`` / ``send_tracks`` / ``close``, the frame rate limit
(kafka_sink.py:151-163), the adaptive quality (:165-192), the colour rule (:303-310) and the payload layout; what moves:

* the event document is written by ``b200va_tracks_json`` from the tick's result-table rows -- the bytes
  ``json.dumps(payload).encode("utf-8")`` would produce, without building a dict, a list of dicts and a Python float
  per coordinate first (the producer is created without a value serialiser and gets those bytes);
* the preview (``_render_frame``, :200-301): INTER_AREA downscale of frames above 1920x1080, the thickness-2 boxes and
  the filled label backgrounds are drawn on the GPU into a copy of the frame; only the annotated preview (at most
  1920x1080) comes back to the host, where the label glyphs (``cv2.putText``) and the encoder (``cv2.imencode``,
  progressive JPEG / WebP) run -- the same OpenCV calls the reference makes, on the same pixels.

The image handed to the encoder is bit-identical to the reference's.  One ordering subtlety: the reference draws box,
background and text track by track, so a LATER track's rectangle can paint over an EARLIER track's text.  When no such
overlap exists (checked on the host from the rectangles' bounding boxes) the texts are simply drawn last; when one does,
the overlay of that frame is replayed in the reference's order with OpenCV on the downscaled, un-annotated image.
"""

from __future__ import annotations

import asyncio
import base64
import logging
import threading
import time
from typing import Dict, Iterable, List, Optional, Sequence, Tuple

import numpy as np

from . import _native
from .runtime import FrameStager, get_handle

LOGGER = logging.getLogger(__name__)

_FONT_SCALE, _FONT_THICKNESS = 0.5, 2


def color_for(class_id: int) -> Tuple[int, int, int]:
    """kafka_sink.py:303-310."""
    seed = (hash(class_id) & 0xFFFFFF) or 0xFFAA33
    return int(seed & 0xFF), int((seed >> 8) & 0xFF), int((seed >> 16) & 0xFF)


def preview_geometry(h: int, w: int) -> Tuple[float, int, int]:
    """(scale_factor, new_w, new_h) of kafka_sink.py:224-232."""
    if w > 1920 or h > 1080:
        sf = min(1920 / w, 1080 / h)
        return sf, int(w * sf), int(h * sf)
    return 1.0, w, h


def _text_box(x: int, y: int, lw: int, lh: int, base: int) -> Tuple[int, int, int, int]:
    # generous bounds of putText(label, (x, y)): glyph cell plus the stroke radius and the anti-aliasing fringe
    return x - 4, y - lh - 6, x + lw + 4, y + base + 6


def overlay_plan(track_list: Sequence[dict], sf: float, label_size):
    """The drawing operations of kafka_sink.py:235-267 for one frame: ``ops`` (rectangles, in order: outline then label
    background per track), ``texts`` ((label, x, y, w, h, baseline) per track) and whether a later rectangle reaches into
    an earlier label (then the overlay must be replayed strictly in order).  Pure host code."""
    ops, texts = [], []
    for trk in track_list:
        x1, y1, x2, y2 = [int(v * sf) for v in trk["bbox_xyxy"]]
        color = color_for(trk["class_id"])
        label = f'ID {trk["track_id"]}'
        lw, lh, base = label_size(label)
        ops.append((0, x1, y1, x2, y2, color))
        ops.append((1, x1, max(0, y1 - lh - base - 4), x1 + lw, max(0, y1), color))
        texts.append((label, x1, max(0, y1 - 4), lw, lh, base))
    # does a later rectangle reach into an earlier label?  Per track five boxes: the four 3-pixel bands of the outline
    # and the label background
    conflict = False
    if len(texts) > 1:
        tb = np.array([_text_box(x, y, lw, lh, b) for _, x, y, lw, lh, b in texts], dtype=np.int64)
        cover = np.empty((len(texts), 5, 4), dtype=np.int64)
        for i in range(len(texts)):
            _, ax, ay, bx, by, _c = ops[2 * i]
            x1, x2, y1, y2 = min(ax, bx), max(ax, bx), min(ay, by), max(ay, by)
            cover[i, 0] = (x1 - 1, y1 - 1, x2 + 1, y1 + 1)
            cover[i, 1] = (x1 - 1, y2 - 1, x2 + 1, y2 + 1)
            cover[i, 2] = (x1 - 1, y1 - 1, x1 + 1, y2 + 1)
            cover[i, 3] = (x2 - 1, y1 - 1, x2 + 1, y2 + 1)
            _, ax, ay, bx, by, _c = ops[2 * i + 1]
            cover[i, 4] = (min(ax, bx), min(ay, by), max(ax, bx), max(ay, by))
        for i in range(len(texts) - 1):
            later = cover[i + 1:].reshape(-1, 4)
            hit = (later[:, 0] <= tb[i, 2]) & (later[:, 2] >= tb[i, 0]) & (later[:, 1] <= tb[i, 3]) & (later[:, 3] >= tb[i, 1])
            if hit.any():
                conflict = True
                break
    return ops, texts, conflict


class PreviewRenderer:
    """``KafkaSink._render_frame`` up to (not including) the encoder: frame + tracks -> annotated BGR preview (host)."""

    def __init__(self, handle: Optional[_native.Handle] = None):
        import cv2

        self.cv2 = cv2
        self.h = handle if handle is not None else get_handle()
        self._stager = FrameStager(self.h)
        self._bufs: Dict[tuple, tuple] = {}   # (h, w) -> (device preview, pinned host mirror)
        self._label_sizes: Dict[str, Tuple[int, int, int]] = {}
        self.replayed = 0                    # frames whose overlay had to be replayed in order on the host
        self._lock = threading.Lock()

    def _label_size(self, label: str) -> Tuple[int, int, int]:
        s = self._label_sizes.get(label)
        if s is None:
            (lw, lh), base = self.cv2.getTextSize(label, self.cv2.FONT_HERSHEY_SIMPLEX, _FONT_SCALE, _FONT_THICKNESS)
            if len(self._label_sizes) > 65536:
                self._label_sizes.clear()
            s = self._label_sizes[label] = (int(lw), int(lh), int(base))
        return s

    def _buffers(self, h: int, w: int):
        b = self._bufs.get((h, w))
        if b is None:
            t = self.h.torch
            b = self._bufs[(h, w)] = (t.empty((h, w, 3), dtype=t.uint8, device=self.h.device),
                                      t.empty((h, w, 3), dtype=t.uint8).pin_memory())
        return b

    def render(self, frame, track_list: Sequence[dict]) -> np.ndarray:
        """``frame``: host ndarray [H, W, 3] uint8 (uploaded whole) or CUDA uint8 tensor, or an NV12 frame as
        ``HotPathEngine`` takes it -- a host ``[3H/2, W]`` array / CPU tensor (uploaded whole, 1.5 bytes per pixel), a
        CUDA ``[3H/2, W]`` tensor or a ``(y, uv)`` pair of CUDA planes; ``track_list``: the dicts of kafka_sink.py:105-123
        (``track_id``, ``class_id``, ``bbox_xyxy``).  Returns the annotated preview the reference would hand to
        ``cv2.imencode`` (for NV12: the one it would for ``cv2.cvtColor(frame, COLOR_YUV2BGR_NV12)``)."""
        cv2, t = self.cv2, self.h.torch
        # B200KafkaSink renders in worker threads (send_tracks -> asyncio.to_thread), and frames of one size share the
        # staging and preview buffers: one render at a time uses them, and the host image leaves as a private copy
        with self._lock:
            on_device = isinstance(frame, (tuple, list)) or (hasattr(frame, "is_cuda") and frame.is_cuda)
            dev = frame if on_device else self._stager.upload([frame])[0]
            fh, fw = _native.frame_hw(dev)
            sf, nw, nh = preview_geometry(fh, fw)
            img_dev, img_host = self._buffers(nh, nw)
            # NV12 is converted in the INTER_AREA taps, at the frame's own size too (there the call is cv2.cvtColor)
            if (nh, nw) != (fh, fw) or _native.is_nv12(dev):
                self.h.resize_area([dev], [(nh, nw)], outs=[img_dev])
            else:
                img_dev.copy_(dev)  # image = frame.copy() (kafka_sink.py:220)
            ops, texts, conflict = overlay_plan(track_list, sf, self._label_size)
            if not conflict and ops:
                self.h.draw_rects([img_dev], [ops])
            img_host.copy_(img_dev, non_blocking=True)
            t.cuda.current_stream().synchronize()
            image = img_host.numpy().copy()
            if conflict:
                self.replayed += 1
        if conflict:
            for (kind, x1, y1, x2, y2, color), k in zip(ops, range(len(ops))):
                cv2.rectangle(image, (x1, y1), (x2, y2), color, -1 if kind else 2)
                if kind:  # the label follows its background (kafka_sink.py:258-267)
                    label, x, y = texts[k // 2][:3]
                    cv2.putText(image, label, (x, y), cv2.FONT_HERSHEY_SIMPLEX, _FONT_SCALE, (255, 255, 255), _FONT_THICKNESS, cv2.LINE_AA)
        else:
            for label, x, y, *_ in texts:
                cv2.putText(image, label, (x, y), cv2.FONT_HERSHEY_SIMPLEX, _FONT_SCALE, (255, 255, 255), _FONT_THICKNESS, cv2.LINE_AA)
        return image


class B200KafkaSink:
    """Drop-in for ``realtime_analytics.sinks.kafka_sink.KafkaSink``."""

    accepts_results = True  # send_tracks(tracks=FrameResult) serialises straight from the result-table rows

    def __init__(self, config, handle: Optional[_native.Handle] = None, producer=None):
        self.config = config
        self._producer = producer  # tests / embedders may inject anything with `async send_and_wait(topic, bytes)`
        self._lock = asyncio.Lock()
        self._last_frame_time: Dict[str, float] = {}
        self._frame_send_interval = 0.1
        self._use_adaptive_quality = True
        self._base_quality = self.config.frame_quality
        self._handle = handle
        self._renderer: Optional[PreviewRenderer] = None
        self._webp_available = self._check_webp_support()

    def _check_webp_support(self) -> bool:  # kafka_sink.py:55-63
        try:
            import cv2

            ok, _ = cv2.imencode(".webp", np.zeros((10, 10, 3), dtype=np.uint8), [cv2.IMWRITE_WEBP_QUALITY, 75])
            return bool(ok)
        except Exception:
            return False

    async def connect(self) -> None:  # kafka_sink.py:65-91
        if not self.config.enabled:
            LOGGER.info("Kafka sink disabled; skipping connection")
            return
        if self._producer:
            return
        try:
            from aiokafka import AIOKafkaProducer
        except ImportError as exc:  # pragma: no cover - the reference raises the same way
            raise RuntimeError("aiokafka is required when Kafka sink is enabled") from exc
        producer = AIOKafkaProducer(bootstrap_servers=self.config.bootstrap_servers, linger_ms=self.config.linger_ms,
                                    max_batch_size=self.config.max_batch_size)  # no value_serializer: bytes go out as they are
        await producer.start()
        self._producer = producer

    # ---- the event ------------------------------------------------------------------------------
    @staticmethod
    def _arrays(tracks) -> Tuple[np.ndarray, np.ndarray, np.ndarray, np.ndarray]:
        """``tracks``: a ``FrameResult`` (its table rows are used as they are), a dict of arrays, or Track objects."""
        a = getattr(tracks, "track_arrays", None)
        if a is None and isinstance(tracks, dict):
            a = tracks
        if a is not None:
            return (np.asarray(a["track_id"], dtype=np.int64), np.asarray(a["cls"], dtype=np.int32),
                    np.asarray(a["conf"], dtype=np.float64), np.asarray(a["bbox_xyxy"], dtype=np.float64).reshape(-1, 4))
        tl = list(tracks)
        for trk in tl:
            if getattr(trk, "action_label", None) is not None or getattr(trk, "temporal_score", None) is not None:
                raise NotImplementedError("temporal track fields (kafka_sink.py:113-121) are outside the GPU hot path; "
                                          "publish those streams through the reference's own KafkaSink")
        return (np.array([trk.track_id for trk in tl], dtype=np.int64), np.array([trk.class_id for trk in tl], dtype=np.int32),
                np.array([trk.confidence for trk in tl], dtype=np.float64),
                np.array([trk.bbox_xyxy for trk in tl], dtype=np.float64).reshape(-1, 4))

    def encode_event(self, stream_name: str, frame_id: int, tracks, frame=None, send_frame: Optional[bool] = None) -> bytes:
        """The message body of ``send_tracks`` (kafka_sink.py:105-149) as bytes."""
        ids, cls, conf, box = self._arrays(tracks)
        url = None
        if send_frame is None:
            send_frame = self.config.include_frames and frame is not None and self._should_send_frame(stream_name)
        if send_frame and frame is not None:
            try:
                quality = self._calculate_adaptive_quality(int(ids.shape[0]))
                track_list = [{"track_id": int(i), "class_id": int(c), "bbox_xyxy": tuple(b)}
                              for i, c, b in zip(ids.tolist(), cls.tolist(), box.tolist())]
                url = self._render_frame(frame, track_list, quality)
            except Exception:  # noqa: BLE001 -- kafka_sink.py:142-143: a failed preview never loses the event
                LOGGER.exception("Failed to encode frame preview for stream '%s'", stream_name)
        return _native.tracks_json(stream_name, int(frame_id), ids, cls, conf, box, url)

    async def send_tracks(self, stream_name: str, frame_id: int, tracks: Iterable, frame=None) -> None:
        if not self.config.enabled or not self._producer:
            return
        send_frame = self.config.include_frames and frame is not None and self._should_send_frame(stream_name)
        if send_frame:
            body = await asyncio.to_thread(self.encode_event, stream_name, frame_id, tracks, frame, True)
        else:
            body = self.encode_event(stream_name, frame_id, tracks, None, False)
        async with self._lock:
            await self._producer.send_and_wait(self.config.topic, body)

    def _should_send_frame(self, stream_name: str) -> bool:  # kafka_sink.py:151-163
        now = time.time()
        if now - self._last_frame_time.get(stream_name, 0.0) >= self._frame_send_interval:
            self._last_frame_time[stream_name] = now
            return True
        return False

    def _calculate_adaptive_quality(self, detection_count: int) -> int:  # kafka_sink.py:165-192
        if not self._use_adaptive_quality:
            return self._base_quality
        boost = -10 if detection_count == 0 else (0 if detection_count <= 3 else (5 if detection_count <= 10 else 10))
        return max(50, min(95, self._base_quality + boost))

    async def close(self) -> None:
        if self._producer is None:
            return
        stop = getattr(self._producer, "stop", None)
        if stop is not None:
            await stop()
        LOGGER.info("Kafka producer closed")

    # ---- the preview ----------------------------------------------------------------------------
    def render_image(self, frame, track_list: Sequence[dict]) -> np.ndarray:
        if self._renderer is None:
            self._renderer = PreviewRenderer(self._handle)
        return self._renderer.render(frame, track_list)

    def _render_frame(self, frame, track_list: Sequence[dict], quality: Optional[int] = None) -> str:  # kafka_sink.py:200-301
        import cv2

        if quality is None:
            quality = self._base_quality
        image = self.render_image(frame, track_list)
        if self._webp_available and quality >= 80:
            ok, buffer = cv2.imencode(".webp", image, [cv2.IMWRITE_WEBP_QUALITY, quality])
            mime = "image/webp"
        else:
            ok, buffer = cv2.imencode(".jpg", image, [cv2.IMWRITE_JPEG_QUALITY, quality, cv2.IMWRITE_JPEG_PROGRESSIVE, 1,
                                                      cv2.IMWRITE_JPEG_OPTIMIZE, 1])
            mime = "image/jpeg"
        if not ok:
            raise RuntimeError("cv2.imencode failed")
        return f"data:{mime};base64,{base64.b64encode(buffer).decode('ascii')}"

    _color_for = staticmethod(color_for)
