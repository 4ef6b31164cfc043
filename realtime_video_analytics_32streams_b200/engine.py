"""Batched per-tick driver: ``StreamWorker._process_packet`` (pipeline.py:143-262 of the
reference) for many streams at once.

One tick takes the latest decoded frame of every stream and runs, in the reference's order,
ROI -> downsample -> motion gate -> adaptive-FPS gate -> predict -> rescale -> float64 re-threshold
-> tracker -> adaptive state update.  The per-stream gates are O(streams) integers and stay on the
host exactly as the reference computes them; everything that touches pixels, head tensors or
track tables is one batched kernel launch per step.  Skipped streams still age their tracks
(``_skip_frame``: ``tracker.update(stream, [])``).

``tick`` = ``submit`` + ``collect``.  ``submit`` only enqueues work (uploads, kernels, one
device->host copy of the result tables into pinned memory); ``collect`` waits for it and hands out
``FrameResult`` objects whose ``Detection`` / ``Track`` lists are materialised lazily from the host
arrays.  When no stream uses the motion gate or adaptive FPS (whose decisions depend on the
previous tick's results) a caller may submit tick k+1 before collecting tick k, which overlaps the
PCIe upload of the next frames with the host-side handling of the current results.
"""

from __future__ import annotations

import logging
from dataclasses import dataclass
from typing import Callable, Dict, List, Optional, Sequence

import numpy as np

from . import _native
from .detector import B200Detector
from .frame_filter import MotionFilter, roi_mask
from .runtime import FrameStager, get_handle
from .tracker import B200IouTracker
from .types import Detection, MotionFilterConfig, Track

LOGGER = logging.getLogger(__name__)


@dataclass
class _StreamState:
    """Host-side gate state of one stream (pipeline.py:88-116)."""

    cfg: object
    motion: Optional[MotionFilter] = None
    frame_index: int = 0
    idle_frames: int = 0
    process_every: int = 1
    max_process_every: int = 1
    idle_tolerance: int = 0
    adaptive: bool = False

    def __post_init__(self):
        s = self.cfg
        self.adaptive = bool(getattr(s, "adaptive_fps", False))
        if self.adaptive:
            target = getattr(s, "target_fps", None) or 30.0
            min_fps = max(getattr(s, "min_target_fps", 5.0), 1.0)
            self.max_process_every = max(1, int(round(target / min_fps)))
            self.idle_tolerance = max(int(getattr(s, "idle_frame_tolerance", 60)), 1)

    def adjust(self, n_det: int, n_trk: int) -> None:
        """``_adjust_adaptive_state`` (pipeline.py:242-262)."""
        if not self.adaptive:
            return
        if n_det > 0 or n_trk > 0:
            self.idle_frames = 0
            self.process_every = 1
        else:
            self.idle_frames += 1
            if self.idle_frames >= self.idle_tolerance:
                self.process_every = max(self.max_process_every, 1)


class FrameResult:
    """What one stream produced in one tick.  ``n_detections`` / ``n_tracks`` and the ``*_arrays``
    are plain host data; ``detections`` / ``tracks`` build the reference's ``Detection`` / ``Track``
    objects on first access (the sinks that want objects pay for them, nobody else does).

    Lifetime: the arrays are views into the pinned result buffers of the tick that produced them, and those
    buffers are reused ``depth`` submits later.  Read (or ``.copy()``) them before then; an access after the
    buffers were handed to a newer tick raises instead of returning the newer tick's rows.  ``device_ms`` is the
    GPU time of the tick's phases (``Handle.phase_times``) when the engine was built with ``profile=True`` -- the
    ``dt`` the reference feeds to ``health.update_success`` (pipeline.py:145, 200-201)."""

    __slots__ = ("stream_name", "frame_id", "processed", "skip_reason", "n_detections", "n_tracks", "_ctx", "_pos",
                 "_dets", "_tracks", "_gen", "device_ms", "adaptive_state")

    def __init__(self, stream_name, frame_id, processed, skip_reason, n_det, n_trk, ctx, pos, device_ms=None):
        self.stream_name, self.frame_id, self.processed, self.skip_reason = stream_name, frame_id, processed, skip_reason
        self.n_detections, self.n_tracks = n_det, n_trk
        self._ctx, self._pos, self._gen = ctx, pos, ctx.gen
        self._dets = self._tracks = None
        self.device_ms = device_ms
        self.adaptive_state = None  # (process_every, idle_frames) after this frame (pipeline.py:242-262), set by collect()

    def _live_ctx(self):
        if self._ctx.gen != self._gen:
            raise RuntimeError("FrameResult read after its result buffers were reused by a later tick: read or copy the "
                               "arrays before submitting `depth` more ticks")
        return self._ctx

    @property
    def track_arrays(self) -> Dict[str, np.ndarray]:
        """Host views: track_id, cls, conf, bbox_xyxy, age, hits -- rows [0, n_tracks)."""
        h, n, p = self._live_ctx().host_tracks, self.n_tracks, self._pos
        return {k: h[k][p, :n] for k in ("track_id", "cls", "conf", "bbox_xyxy", "age", "hits")}

    @property
    def detection_arrays(self) -> Dict[str, np.ndarray]:
        """Host views: cls, conf (float64), bbox_xyxy (float64, rescaled like pipeline.py:224-240)."""
        h, n, p = self._live_ctx().host_dets, self.n_detections, self._pos
        box = h["bbox_xyxy"][p, :n].astype(np.float64)
        sc = self._ctx.scale[p]
        if sc != 1.0:
            box = box * sc
        return {"cls": h["cls"][p, :n], "conf": h["conf"][p, :n].astype(np.float64), "bbox_xyxy": box}

    @property
    def tracks(self) -> List[Track]:
        if self._tracks is None:
            a = self.track_arrays
            self._tracks = [Track(i, c, f, tuple(b), g, k) for i, c, f, b, g, k in
                            zip(a["track_id"].tolist(), a["cls"].tolist(), a["conf"].tolist(), a["bbox_xyxy"].tolist(),
                                a["age"].tolist(), a["hits"].tolist())]
        return self._tracks

    @property
    def detections(self) -> List[Detection]:
        if self._dets is None:
            if not self.processed or self.n_detections == 0:
                self._dets = []
            else:
                a = self.detection_arrays
                nm, fid = self.stream_name, self.frame_id
                self._dets = [Detection(nm, fid, c, f, tuple(b)) for c, f, b in
                              zip(a["cls"].tolist(), a["conf"].tolist(), a["bbox_xyxy"].tolist())]
        return self._dets


class _TickCtx:
    """Buffers of one in-flight tick."""

    def __init__(self, h: _native.Handle, n: int):
        t = h.torch
        self.dets = h.alloc_dets(n)
        self.tracks = h.alloc_tracks(n)
        self.host_dets_t = h.alloc_dets(n, pinned_host=True)
        self.host_tracks_t = h.alloc_tracks(n, pinned_host=True)
        self.host_dets = {k: v.numpy() for k, v in self.host_dets_t.items() if not k.startswith("_")}
        self.host_tracks = {k: v.numpy() for k, v in self.host_tracks_t.items() if not k.startswith("_")}
        self.status = t.zeros(h.STATUS_WORDS, dtype=t.int32).pin_memory()  # capacity flags, copied back with the tables
        # device-side gates: skip flags decided on the device and (skip, process_every, idle_frames, frame_index) per row
        self.skip = t.zeros((n,), dtype=t.uint8, device=h.device)
        self.gate_state = t.zeros((n, 4), dtype=t.int32, device=h.device)
        self.host_gate_state = t.zeros((n, 4), dtype=t.int32).pin_memory()
        self.device_gates = False
        self.done = t.cuda.Event()
        self.busy = False
        self.gen = 0       # bumped by every submit that takes these buffers (FrameResult lifetime check)
        self.keep = None   # upload sources of this tick: alive until it is collected (raw async copies read them)
        self.phase_ms = None
        # filled by submit()
        self.order: List[int] = []
        self.n_act = 0
        self.names: List[str] = []
        self.ids: List[int] = []
        self.states: List[_StreamState] = []
        self.skip_reason: List[Optional[str]] = []
        self.scale: List[float] = []
        self.live: List[int] = []


class HotPathEngine:
    """pre + post + track for a set of streams, one tick at a time."""

    def __init__(self, streams: Sequence, detector_config, tracker_config, infer: Callable,
                 handle: Optional[_native.Handle] = None, input_hw=None, depth: int = 2, static_pads: bool = True,
                 on_overflow: str = "raise", profile: bool = False, device_gates: bool = False):
        """``device_gates``: take the motion and adaptive-FPS decisions on the device (``b200va_gates_decide`` /
        ``b200va_gates_commit``): no host round trip inside a tick, every live frame keeps its batch position (``infer``
        sees all of them; rows of gated-off frames hold stale pixels and their heads are ignored), and ticks may be
        pipelined (``submit`` before ``collect``) even for streams with motion_filter / adaptive_fps.  Results are
        identical to the host-side gates.
        ``on_overflow``: what ``collect`` does when a frame exceeded ``max_candidates`` / ``max_dets`` /
        ``max_tracks`` (rows were dropped; the reference has no such limits): "raise" (default) or "warn".
        ``profile``: record per-phase device times (``FrameResult.device_ms``); costs one event pair per phase."""
        if on_overflow not in ("raise", "warn"):
            raise ValueError("on_overflow must be 'raise' or 'warn'")
        self.on_overflow, self.profile = on_overflow, bool(profile)
        self.h = handle if handle is not None else get_handle()
        if self.profile:
            self.h.set_profiling(True)
        self.streams = list(streams)
        self.detector = B200Detector(detector_config, input_hw=input_hw, infer=infer, handle=self.h, fold_filter=True)
        self.tracker = B200IouTracker(tracker_config, handle=self.h)
        self.state: Dict[str, _StreamState] = {s.name: _StreamState(s) for s in self.streams}
        self.stager = FrameStager(self.h)
        n = max(len(self.streams), 1)
        self._ctxs = [_TickCtx(self.h, n) for _ in range(max(depth, 1))]
        self._turn = 0
        self.active_streams: List[int] = []
        self._changed = self.h.torch.empty((n,), dtype=self.h.torch.int32, device=self.h.device)
        self._batches: Dict[tuple, _native.FrameBatch] = {}
        self._persistent = set()  # ids of the engine's own persistent device tensors (downsample outputs)
        self._small: Dict[tuple, object] = {}
        self._net = None
        self._net_shapes = []
        # the network-input buffer is persistent: pad rows are written once per geometry (B200VA_OUT_FLAG_PADS_VALID).
        # Needs an `infer` that does not write into its input; pass static_pads=False otherwise.
        self.static_pads = bool(static_pads)
        # a tick's gates depend on the previous tick's results for these features
        self.device_gates = bool(device_gates)
        self.sequential = (not self.device_gates) and any(getattr(s, "motion_filter", False) or getattr(s, "adaptive_fps", False)
                                                          for s in self.streams)
        if self.device_gates:
            for s in self.streams:
                self.h.gates_reset(self.tracker.slot_of(s.name))

    def reset_tracks(self) -> None:
        """Drop every stream's tracks (the id counter keeps running, like a reference tracker that lost its streams)."""
        for st in self.streams:
            self.tracker.reset(st.name)

    # --------------------------------------------------------------------------------------
    def _frame_batch(self, frames, masks):
        """Argument arrays are cached per set of device pointers (staging buffers are persistent).  ``frames`` are
        all BGR or all NV12."""
        make = _native.Nv12Batch if _native.is_nv12(frames[0]) else _native.FrameBatch
        if not all(self.stager.owns(f) or id(f) in self._persistent for f in frames):
            # caller-supplied CUDA frames: their addresses change from tick to tick, and a cached batch would
            # keep the tensors (and their HBM) alive -- build the argument arrays for this tick only
            return make(frames, masks)
        key = tuple((f.data_ptr(), f.shape[0], f.shape[1], f.stride(0), m.data_ptr() if m is not None else 0)
                    for f, m in zip(frames, masks))
        fb = self._batches.get(key)
        if fb is None:
            if len(self._batches) > 64:
                self._batches.clear()
            fb = self._batches[key] = make(frames, masks)
        return fb

    def _letterbox(self, frames, masks, fmt, out, skip=None):
        """``preprocess`` of a batch whose frames may mix BGR and NV12: one call per run of consecutive frames of one
        kind, into the rows of ``out`` (and, with device-side gates, the entries of ``skip``) at their positions."""
        kinds = [_native.is_nv12(f) for f in frames]
        metas = []
        b = 0
        while b < len(frames):
            e = b + 1
            while e < len(frames) and kinds[e] == kinds[b]:
                e += 1
            if skip is not None and (b, e) != (0, len(frames)):
                self.h.set_skip_mask(skip[b:e])
            _, m = self.h.preprocess(self._frame_batch(frames[b:e], masks[b:e]), self.detector.input_hw, fmt, out=out[b:e])
            metas += m
            b = e
        return out, metas

    def _net_in(self, n: int):
        t = self.h.torch
        dtype = t.float16 if self.detector._fmt == _native.OUT_F16_RGB_NCHW else t.float32
        if self._net is None or self._net.shape[0] < n or self._net.dtype != dtype:
            self._net = t.empty((max(n, len(self.streams)), 3, *self.detector.input_hw), dtype=dtype, device=self.h.device)
            self._net_shapes = [None] * self._net.shape[0]  # source (h, w) whose pad rows each position holds
        return self._net[:n]

    def _bgr_buffer(self, pos: int, hw, full: bool = False):
        """One persistent BGR buffer per (stream position, size, purpose): stable addresses, no per-tick allocation."""
        key = (pos, tuple(hw), full)
        buf = self._small.get(key)
        if buf is None:
            buf = self._small[key] = self.h.torch.empty((hw[0], hw[1], 3), dtype=self.h.torch.uint8, device=self.h.device)
            self._persistent.add(id(buf))
        return buf

    def _pads_flag(self, frames) -> int:
        """B200VA_OUT_FLAG_PADS_VALID when every batch position was last written from a frame of the same size
        (same letterbox geometry, same format): its pad rows are already in the persistent buffer."""
        shapes = [_native.frame_hw(f) for f in frames]
        valid = all(self._net_shapes[k] == sh for k, sh in enumerate(shapes))
        for k, sh in enumerate(shapes):
            self._net_shapes[k] = sh
        return _native.OUT_FLAG_PADS_VALID if (valid and self.static_pads) else 0

    # --------------------------------------------------------------------------------------
    def tick(self, frames: Sequence, frame_ids: Optional[Sequence[int]] = None, infer_ctx=None) -> List[FrameResult]:
        """``frames[i]`` is the new frame of ``streams[i]`` (host array, pinned CPU tensor or CUDA
        tensor) or None when that stream delivered nothing this tick.  A frame may be BGR ``[H, W, 3]`` or NV12: a
        2-D ``[3H/2, W]`` uint8 host array / CPU tensor / CUDA tensor, or a ``(y, uv)`` pair of CUDA planes.  NV12
        results equal those of the same engine fed ``cv2.cvtColor(frame, cv2.COLOR_YUV2BGR_NV12)``."""
        ctx = self.submit(frames, frame_ids, infer_ctx)
        return self.collect(ctx) if ctx is not None else []

    def submit(self, frames: Sequence, frame_ids: Optional[Sequence[int]] = None, infer_ctx=None) -> Optional[_TickCtx]:
        live = [i for i, f in enumerate(frames) if f is not None]
        if not live:
            return None
        ctx = self._ctxs[self._turn]
        self._turn = (self._turn + 1) % len(self._ctxs)
        if ctx.busy:
            raise RuntimeError("HotPathEngine: collect() the oldest tick before submitting another one")
        if self.sequential and any(c.busy for c in self._ctxs):
            raise RuntimeError("HotPathEngine: streams with motion_filter / adaptive_fps need collect() before the next submit()")
        names = [self.streams[i].name for i in live]
        states = [self.state[n] for n in names]
        # frames that only feed the letterbox need just its tapped rows on the device
        sparse_ok = [False] * len(frames)
        for i, st in zip(live, states):
            sparse_ok[i] = (not getattr(st.cfg, "motion_filter", False)
                            and float(getattr(st.cfg, "downsample_ratio", 1.0)) >= 0.999)
        staged = self.stager.upload(list(frames), sparse_for=self.detector.input_hw, sparse_ok=sparse_ok)
        ctx.keep = self.stager.take_sources()
        ctx.gen += 1
        dev_frames = [staged[i] for i in live]
        for st in states:
            st.frame_index += 1
        ids = [frame_ids[i] if frame_ids is not None else st.frame_index for i, st in zip(live, states)]

        # 1-2. ROI (fused into the consumers) and downsample
        masks, ratios = [], []
        for st, f in zip(states, dev_frames):
            polys = getattr(st.cfg, "roi_polygons", None) or []
            masks.append(roi_mask(polys, *_native.frame_hw(f), self.h) if polys else None)
            ratios.append(float(getattr(st.cfg, "downsample_ratio", 1.0)))
        down = [k for k, r in enumerate(ratios) if r < 0.999]
        work = list(dev_frames)
        work_masks = list(masks)
        if down:
            sizes = {k: tuple(int(v * ratios[k]) for v in _native.frame_hw(dev_frames[k])) for k in down}
            # NV12 frames are converted in the same taps (resize_linear_u8_nv12); one call per source format
            for group in ([k for k in down if not _native.is_nv12(dev_frames[k])], [k for k in down if _native.is_nv12(dev_frames[k])]):
                if not group:
                    continue
                outs = [self._bgr_buffer(live[k], sizes[k]) for k in group]
                small = self.h.resize([dev_frames[k] for k in group], [sizes[k] for k in group], [masks[k] for k in group],
                                      outs=outs)
                for k, s in zip(group, small):
                    work[k] = s
                    work_masks[k] = None  # the ROI is already baked into the downsampled frame

        mot = [k for k, st in enumerate(states) if getattr(st.cfg, "motion_filter", False)]
        # the motion gate reads BGR: an NV12 frame it sees is converted at its own size (cv2.cvtColor) into a
        # persistent per-stream buffer, which the letterbox then reads too
        cvt = [k for k in mot if _native.is_nv12(work[k])]
        if cvt:
            outs = [self._bgr_buffer(live[k], _native.frame_hw(work[k]), full=True) for k in cvt]
            full = self.h.resize([work[k] for k in cvt], [_native.frame_hw(work[k]) for k in cvt], outs=outs)
            for k, f in zip(cvt, full):
                work[k] = f
        if self.device_gates:
            return self._submit_device_gates(ctx, live, names, states, ids, work, work_masks, ratios, mot, infer_ctx)

        # 3. motion gate (one launch for every stream that has it enabled, one count read-back)
        skip_reason: List[Optional[str]] = [None] * len(live)
        if mot:
            prevs, nexts = [], []
            for k in mot:
                st = states[k]
                if st.motion is None:
                    st.motion = MotionFilter(MotionFilterConfig(enable=True, threshold=st.cfg.motion_threshold),
                                             tuple(work[k].shape), handle=self.h)
                p, n = st.motion.buffers(work[k].shape[0], work[k].shape[1])
                prevs.append(p)
                nexts.append(n)
            counts = self.h.motion([work[k] for k in mot], prevs, nexts, [work_masks[k] for k in mot],
                                   self._changed[:len(mot)]).cpu().numpy()
            for j, k in enumerate(mot):
                if not states[k].motion.commit(int(counts[j])):
                    skip_reason[k] = "motion"

        # 4. adaptive-FPS gate (pipeline.py:165-170)
        for k, st in enumerate(states):
            if skip_reason[k] is None and st.adaptive and st.process_every > 1:
                if (st.frame_index - 1) % st.process_every != 0:
                    skip_reason[k] = "adaptive"

        # 5-8. predict on the active subset, then the tracker over every live stream
        active = [k for k in range(len(live)) if skip_reason[k] is None]
        skipped = [k for k in range(len(live)) if skip_reason[k] is not None]
        order = active + skipped  # skipped streams create no tracks, so id order is unaffected
        n_act = len(active)
        nb = len(order)
        dets = {k_: v[:nb] for k_, v in ctx.dets.items() if not k_.startswith("_")}
        if n_act:
            net = self._net_in(n_act)
            act_frames = [work[k] for k in active]
            tensor, metas = self._letterbox(act_frames, [work_masks[k] for k in active],
                                            self.detector._fmt | self._pads_flag(act_frames), net)
            # which stream each row of `tensor` belongs to (index into self.streams), for callers whose forward
            # is per-stream (model selection, synthetic heads in tests)
            self.active_streams = [live[k] for k in active]
            head = self.detector._infer(tensor) if infer_ctx is None else self.detector._infer_fn(tensor, infer_ctx)
            head = self.detector._as_head(head)
            if head.dim() != 3 or head.shape[0] != n_act:
                raise ValueError(f"infer returned {tuple(head.shape)} for a batch of {n_act}")
            self.detector._run_post(head, metas, {k_: v[:n_act] for k_, v in dets.items()})
        scale = [1.0 / max(ratios[k], 1e-6) if ratios[k] < 0.999 else 1.0 for k in order]
        out = {k_: v[:nb] for k_, v in ctx.tracks.items() if not k_.startswith("_")}
        self.tracker.update_batch([names[k] for k in order], dets,
                                  det_scale=scale if any(s != 1.0 for s in scale) else None,
                                  skip=[0] * n_act + [1] * len(skipped), out=out)
        # 9. one device -> host copy per result table, into pinned memory
        ctx.host_dets_t["_flat"].copy_(ctx.dets["_flat"], non_blocking=True)
        ctx.host_tracks_t["_flat"].copy_(ctx.tracks["_flat"], non_blocking=True)
        self.h.read_status_async(ctx.status)
        ctx.done.record()
        ctx.busy = True
        ctx.device_gates = False
        ctx.order, ctx.n_act, ctx.names, ctx.ids, ctx.states = order, n_act, names, ids, states
        ctx.skip_reason, ctx.scale, ctx.live = skip_reason, scale, live
        return ctx

    def _submit_device_gates(self, ctx, live, names, states, ids, work, work_masks, ratios, mot, infer_ctx):
        """Steps 3-9 of ``submit`` with the gates on the device: nothing here waits for the GPU."""
        h = self.h
        nb = len(live)
        changed = None
        if mot:
            prevs, nexts = [], []
            for k in mot:
                st = states[k]
                if st.motion is None:
                    st.motion = MotionFilter(MotionFilterConfig(enable=True, threshold=st.cfg.motion_threshold),
                                             tuple(work[k].shape), handle=h)
                p, n = st.motion.buffers(work[k].shape[0], work[k].shape[1])
                prevs.append(p)
                nexts.append(n)
            changed = h.motion([work[k] for k in mot], prevs, nexts, [work_masks[k] for k in mot], self._changed[:len(mot)])
            for k in mot:
                states[k].motion.advance()
        gates = (_native.Gate * nb)()
        where = {k: j for j, k in enumerate(mot)}
        for k, st in enumerate(states):
            g = gates[k]
            g.slot = self.tracker.slot_of(names[k])
            g.motion = 1 if k in where else 0
            g.changed_index = where.get(k, -1)
            g.adaptive = 1 if st.adaptive else 0
            g.max_process_every = max(st.max_process_every, 1)
            g.idle_tolerance = max(st.idle_tolerance, 1)
            g.motion_threshold = float(st.cfg.motion_threshold) if k in where else 0.0
            fh, fw = _native.frame_hw(work[k])
            g.pixels = fh * fw
        skip = ctx.skip[:nb]
        h.gates_decide(gates, changed, skip)
        dets = {k_: v[:nb] for k_, v in ctx.dets.items() if not k_.startswith("_")}
        out = {k_: v[:nb] for k_, v in ctx.tracks.items() if not k_.startswith("_")}
        try:
            net = self._net_in(nb)
            pads = self._pads_flag(work)
            # a batch position whose pad rows were never written must be letterboxed whatever its gate says
            h.set_skip_mask(skip if pads else None)
            tensor, metas = self._letterbox(work, work_masks, self.detector._fmt | pads, net, skip if pads else None)
            h.set_skip_mask(skip)
            self.active_streams = list(live)
            head = self.detector._infer(tensor) if infer_ctx is None else self.detector._infer_fn(tensor, infer_ctx)
            head = self.detector._as_head(head)
            if head.dim() != 3 or head.shape[0] != nb:
                raise ValueError(f"infer returned {tuple(head.shape)} for a batch of {nb}")
            self.detector._run_post(head, metas, dets)
            scale = [1.0 / max(r, 1e-6) if r < 0.999 else 1.0 for r in ratios]
            self.tracker.update_batch(names, dets, det_scale=scale if any(s != 1.0 for s in scale) else None, out=out)
            h.gates_commit(gates, dets["count"], out["count"], skip, ctx.gate_state[:nb])
        finally:
            h.set_skip_mask(None)
        ctx.host_dets_t["_flat"].copy_(ctx.dets["_flat"], non_blocking=True)
        ctx.host_tracks_t["_flat"].copy_(ctx.tracks["_flat"], non_blocking=True)
        ctx.host_gate_state.copy_(ctx.gate_state, non_blocking=True)
        h.read_status_async(ctx.status)
        ctx.done.record()
        ctx.busy = True
        ctx.device_gates = True
        ctx.order, ctx.n_act, ctx.names, ctx.ids, ctx.states = list(range(nb)), nb, names, ids, states
        ctx.skip_reason, ctx.scale, ctx.live = [None] * nb, scale, live
        return ctx

    def collect(self, ctx: _TickCtx) -> List[FrameResult]:
        """Wait for a submitted tick; update the adaptive-FPS state (pipeline.py:197) and return
        one FrameResult per live stream, in stream order."""
        ctx.done.synchronize()
        ctx.busy = False
        ctx.keep = None
        msg = self.h.status_message(ctx.status.tolist())
        if msg:
            if self.on_overflow == "raise":
                raise _native.B200VAError(_native.ERR_CAPACITY, msg)
            LOGGER.warning("HotPathEngine: %s", msg)
        phase_ms = self.h.phase_times() if self.profile else None
        det_counts = ctx.host_dets["count"]
        trk_counts = ctx.host_tracks["count"]
        results: List[Optional[FrameResult]] = [None] * len(ctx.order)
        gate = ctx.host_gate_state.tolist() if ctx.device_gates else None
        for pos, k in enumerate(ctx.order):
            if gate is not None:  # decided and committed on the device: mirror the state, do not recompute it
                flag, pe, idle, _ = gate[pos]
                processed = flag == _native.GATE_PROCESS
                ctx.skip_reason[k] = None if processed else ("motion" if flag == _native.GATE_SKIP_MOTION else "adaptive")
                n_det = int(det_counts[pos]) if processed else 0
                n_trk = int(trk_counts[pos])
                if ctx.states[k].adaptive:
                    ctx.states[k].process_every, ctx.states[k].idle_frames = pe, idle
                results[k] = FrameResult(ctx.names[k], ctx.ids[k], processed, ctx.skip_reason[k], n_det, n_trk, ctx, pos, phase_ms)
                results[k].adaptive_state = (ctx.states[k].process_every, ctx.states[k].idle_frames)
                continue
            processed = pos < ctx.n_act
            n_det = int(det_counts[pos]) if processed else 0
            n_trk = int(trk_counts[pos])
            ctx.states[k].adjust(n_det, n_trk)
            results[k] = FrameResult(ctx.names[k], ctx.ids[k], processed, ctx.skip_reason[k], n_det, n_trk, ctx, pos, phase_ms)
            results[k].adaptive_state = (ctx.states[k].process_every, ctx.states[k].idle_frames)
        return results  # type: ignore[return-value]
