"""Detector plug-in: the reference's ``BaseDetector`` contract on top of the sm_100a kernels.

Mirrors ``_TensorRTBaseDetector`` (detector.py:182-379 of the reference): ``predict`` is
``_preprocess -> _infer -> _postprocess`` with the same argument meaning, the same ``meta`` dict
and the same error behaviour, but the three steps run on the GPU through ``libb200va`` and every
intermediate stays in HBM.  ``_infer`` is the detector forward -- outside the kernel scope -- and
is supplied by the caller as any callable from the network input ``[B,3,H,W]`` (CUDA) to the
decoded head ``[B,C,A]`` / ``[B,A,C]`` (CUDA), e.g. a ``torch.nn.Module``.

``predict_batch`` is additive API (the reference is strictly batch-1, detector.py:280-281).
"""

from __future__ import annotations

import logging
from typing import Callable, List, Optional, Sequence

import numpy as np

from . import _native
from .runtime import FrameStager, get_handle
from .types import Detection, FramePacket

LOGGER = logging.getLogger(__name__)


def filter_detections(detections, min_confidence: float) -> List[Detection]:
    """detector.py:99-103 -- kept for callers that hold Python detections; the batched path folds
    this float64 comparison into the NMS emit step instead."""
    return [det for det in detections if det.confidence >= min_confidence]


class B200Detector:
    """Drop-in for the reference's numpy-path detectors (``backend: b200``)."""

    def __init__(self, config, input_hw: Optional[Sequence[int]] = None, infer: Optional[Callable] = None,
                 handle: Optional[_native.Handle] = None, fold_filter: bool = False):
        self.config = config
        if input_hw is None:
            size = getattr(config, "input_size", None)
            input_hw = (int(size[0]), int(size[1])) if size else (640, 640)
        self.input_hw = (int(input_hw[0]), int(input_hw[1]))
        self.h = handle if handle is not None else get_handle()
        self._infer_fn = infer
        self._stager = FrameStager(self.h)
        # fold_filter=True applies filter_detections (pipeline.py:182) inside the kernel
        self.fold_filter = fold_filter
        self._bufs = {}  # batch size -> (device detection SoA, pinned host mirror, numpy views, pinned status words)

    def _result_buffers(self, batch: int):
        """Persistent result tables per batch size: the post-process writes the device SoA, ONE copy of its flat
        buffer (plus the capacity flags) brings a call's detections back."""
        b = self._bufs.get(batch)
        if b is None:
            t = self.h.torch
            dev, host = self.h.alloc_dets(batch), self.h.alloc_dets(batch, pinned_host=True)
            b = self._bufs[batch] = (dev, host, {k: v.numpy() for k, v in host.items() if not k.startswith("_")},
                                     t.zeros(self.h.STATUS_WORDS, dtype=t.int32).pin_memory())
        return b

    # ---- the three reference steps ---------------------------------------------------------
    @property
    def _fmt(self) -> int:
        return _native.OUT_F16_RGB_NCHW if getattr(self.config, "half", False) else _native.OUT_F32_RGB_NCHW

    def _preprocess(self, frame, roi_mask=None):
        """detector.py:198-264.  Returns (CUDA tensor [1,3,H,W], meta dict).  A host frame is staged into a
        device buffer only this detector reads, so just the rows the letterbox taps cross PCIe (one in three
        for 1080p -> 640x360)."""
        dev = self._stager.upload([frame], sparse_for=self.input_hw)
        tensor, metas = self.h.preprocess(dev, self.input_hw, self._fmt, [roi_mask] if roi_mask is not None else None)
        return tensor, metas[0].as_meta()

    def _preprocess_batch(self, frames, roi_masks=None):
        dev = self._stager.upload(frames, sparse_for=self.input_hw)
        return self.h.preprocess(dev, self.input_hw, self._fmt, roi_masks)

    def _infer(self, tensor):
        if self._infer_fn is None:
            raise RuntimeError("B200Detector has no model: pass infer=<callable [B,3,H,W] -> head>")
        return self._infer_fn(tensor)

    def _as_head(self, predictions):
        """Normalise whatever ``_infer`` returned to a contiguous CUDA [B, d1, d2]: float16 stays float16 (the decode
        reads it in place, with the results of its float32 widening), every other dtype becomes float32."""
        t = self.h.torch
        if isinstance(predictions, (list, tuple)):
            predictions = predictions[0]  # detector.py:278-279
        if isinstance(predictions, np.ndarray):
            dtype = np.float16 if predictions.dtype == np.float16 else np.float32  # fp16 crosses PCIe at half the bytes
            predictions = t.from_numpy(np.ascontiguousarray(predictions, dtype=dtype))
        if not predictions.is_cuda:
            predictions = predictions.to(self.h.device, non_blocking=True)
        if predictions.dtype not in (t.float32, t.float16):
            predictions = predictions.float()
        return predictions.contiguous()

    def _postprocess(self, predictions, packet: FramePacket, meta: dict) -> List[Detection]:
        """detector.py:266-338 for one frame (batch-1 like the reference)."""
        head = self._as_head(predictions)
        if head.dim() == 3:
            if head.shape[0] != 1:  # np.squeeze(axis=0) on a batch > 1
                raise ValueError("cannot select an axis to squeeze out which has size not equal to one")
        elif head.dim() == 2:
            head = head[None]
        else:
            LOGGER.warning("Unexpected prediction shape: %s", tuple(head.shape))
            return []
        _, d1, d2 = head.shape
        channels = d2 if not (d1 != 0 and d1 < d2) else d1
        if channels < 5:
            LOGGER.warning("Unexpected prediction shape: %s", (d1, d2))
            return []
        oh, ow = meta["orig_shape"]
        lb = _native.letterbox_meta(int(oh), int(ow), self.input_hw[0], self.input_hw[1])
        # honour a caller-edited meta (scale / pad) exactly like _scale_boxes would
        lb.scale = float(meta["scale"])
        lb.pad_left, lb.pad_top = int(meta["pad"][0]), int(meta["pad"][1])
        dets = self._run_post(head, [lb], self._result_buffers(1)[0])
        return self._to_detections(dets, [packet])[0]

    # ---- public API ------------------------------------------------------------------------
    def predict(self, packet: FramePacket) -> List[Detection]:
        tensor, meta = self._preprocess(packet.frame)
        raw = self._infer(tensor)
        return self._postprocess(raw, packet, meta)

    def predict_batch(self, packets: Sequence[FramePacket], roi_masks=None) -> List[List[Detection]]:
        if not packets:
            return []
        dets, _ = self.predict_batch_device([p.frame for p in packets], roi_masks, self._result_buffers(len(packets))[0])
        return self._to_detections(dets, packets)

    def predict_batch_device(self, frames, roi_masks=None, dets_out=None):
        """Frames (host arrays or CUDA tensors) -> detections as device SoA tensors + metas."""
        tensor, metas = self._preprocess_batch(frames, roi_masks)
        head = self._as_head(self._infer(tensor))
        if head.dim() != 3 or head.shape[0] != len(frames):
            raise ValueError(f"infer returned {tuple(head.shape)} for a batch of {len(frames)}")
        return self._run_post(head, metas, dets_out), metas

    def _run_post(self, head, metas, dets_out=None):
        cfg = self.config
        thr = float(cfg.confidence_threshold)
        return self.h.postprocess(head, metas, thr, float(cfg.iou_threshold), getattr(cfg, "classes", None) or None,
                                  filter_conf=thr if self.fold_filter else None, out=dets_out)

    def _to_detections(self, dets, packets) -> List[List[Detection]]:
        """Device SoA -> ``Detection`` objects: one pinned device->host copy of the flat table (and the capacity
        flags), one synchronisation."""
        h, t = self.h, self.h.torch
        nb = len(packets)
        dev, host, views, status = self._result_buffers(nb)
        if dets is not dev:  # a caller-owned SoA: bring it into the persistent table first (device-side copy)
            dev["_flat"].copy_(dets["_flat"]) if "_flat" in dets and dets["_flat"].numel() == dev["_flat"].numel() else [
                dev[k][:nb].copy_(dets[k][:nb]) for k in ("bbox_xyxy", "conf", "cls", "count")]
        host["_flat"].copy_(dev["_flat"], non_blocking=True)
        h.read_status_async(status)
        t.cuda.current_stream(h.device).synchronize()
        msg = h.status_message(status.tolist())
        if msg:
            raise _native.B200VAError(_native.ERR_CAPACITY, msg)
        counts = views["count"].tolist()
        out = []
        for b, packet in enumerate(packets):
            n = int(counts[b])
            if n == 0:
                out.append([])
                continue
            name = getattr(packet.stream, "name", str(packet.stream))
            fid = packet.frame_id
            # float32 -> Python float exactly as `float(np.float32)` in detector.py:330-336
            out.append([Detection(name, fid, c, f, tuple(bx)) for c, f, bx in
                        zip(views["cls"][b, :n].tolist(), views["conf"][b, :n].astype(np.float64).tolist(),
                            views["bbox_xyxy"][b, :n].astype(np.float64).tolist())])
        return out


class B200UltralyticsDetector(B200Detector):
    """Drop-in for ``UltralyticsDetector`` (detector.py:106-179): what ``YOLO(...).predict(frame, conf, iou,
    classes, half)`` does around the model forward -- ``LetterBox`` (rounded sizes; ``auto=True`` rect padding
    for a single image, like ``predict`` on an ndarray with a PyTorch model), ``ops.non_max_suppression``
    (strict ``>``, class-shifted boxes, ``max_det``) and ``ops.scale_boxes`` -- on the sm_100a kernels.
    ``infer`` maps the network input ``[B, 3, h, w]`` to the decoded Detect head ``[B, 4 + nc, A]``
    (what ``model.model(im)[0]`` returns).  Parity against ultralytics itself is unpinned (package absent);
    see ``oracle/ultralytics_restate.py`` for what the tests pin."""

    def __init__(self, config, input_hw=None, infer=None, handle=None, auto: bool = True, stride: int = 32,
                 max_det: int = 300, agnostic: bool = False, fold_filter: bool = False):
        super().__init__(config, input_hw=input_hw, infer=infer, handle=handle, fold_filter=fold_filter)
        self.auto, self.stride, self.max_det, self.agnostic = bool(auto), int(stride), int(max_det), bool(agnostic)

    def _geometry(self, shapes):
        geoms, outs = [], set()
        for h, w in shapes:
            m, oh, ow = _native.letterbox_meta_ultralytics(int(h), int(w), self.input_hw[0], self.input_hw[1], self.auto,
                                                           self.stride)
            geoms.append(m)
            outs.add((oh, ow))
        if len(outs) != 1:
            # LetterBox(auto=...) is only rect when every image of the batch has the same shape (same_shapes)
            geoms = [_native.letterbox_meta_ultralytics(int(h), int(w), self.input_hw[0], self.input_hw[1], False,
                                                        self.stride)[0] for h, w in shapes]
            outs = {self.input_hw}
        return geoms, next(iter(outs))

    def _preprocess(self, frame, roi_mask=None):
        dev = self._stager.upload([frame])  # every row: the sparse upload pattern is the reference letterbox's
        geoms, in_hw = self._geometry([dev[0].shape[:2]])
        tensor = self.h.preprocess_geom(dev, geoms, in_hw, self._fmt, [roi_mask] if roi_mask is not None else None)
        return tensor, {"orig_shape": tuple(int(v) for v in dev[0].shape[:2]), "in_shape": in_hw}

    def _postprocess(self, predictions, packet: FramePacket, meta: dict) -> List[Detection]:
        head = self._as_head(predictions)
        if head.dim() == 2:
            head = head[None]
        dets = self._run_post_ultra(head, [meta["orig_shape"]], meta["in_shape"], self._result_buffers(1)[0])
        return self._to_detections(dets, [packet])[0]

    def predict_batch_device(self, frames, roi_masks=None, dets_out=None):
        dev = self._stager.upload(frames)
        shapes = [tuple(int(v) for v in d.shape[:2]) for d in dev]
        geoms, in_hw = self._geometry(shapes)
        tensor = self.h.preprocess_geom(dev, geoms, in_hw, self._fmt, roi_masks)
        head = self._as_head(self._infer(tensor))
        if head.dim() != 3 or head.shape[0] != len(frames):
            raise ValueError(f"infer returned {tuple(head.shape)} for a batch of {len(frames)}")
        return self._run_post_ultra(head, shapes, in_hw, dets_out), geoms

    def _run_post_ultra(self, head, shapes, in_hw, dets_out=None):
        cfg = self.config
        thr = float(cfg.confidence_threshold)
        return self.h.postprocess_ultralytics(head, shapes, in_hw, thr, float(cfg.iou_threshold),
                                              getattr(cfg, "classes", None) or None, self.agnostic, self.max_det,
                                              filter_conf=thr if self.fold_filter else None, out=dets_out)
