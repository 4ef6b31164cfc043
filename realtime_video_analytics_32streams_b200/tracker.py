"""Tracker plug-in: ``IouTracker``'s contract (tracker.py:36-126 of the reference) with the track
table resident in HBM and the matching done by ``b200va_tracker_update``.

``update(stream_name, detections)`` keeps the reference signature: Python ``Detection`` objects in
(their float64 fields go down unchanged), all surviving ``Track`` objects out, one id counter
shared by every stream.  It costs one pinned host->device copy and one device->host copy per call.
``update_batch`` is the additive batched entry: device SoA detections straight from
``B200Detector.predict_batch_device`` for many streams in one launch.

Stream slots belong to the handle (``Handle.claim_slot``): trackers that share a handle never share a
slot, a slot is empty when a tracker first maps a stream to it, and ``close()`` gives the slots back.
The id counter is handle-wide -- the reference's ``itertools.count(1)`` lives in the tracker instance
(tracker.py:47), so give every tracker that must number its tracks from 1 its own handle, or create it
while no other tracker on the handle is alive (the counter restarts at 1 then).
"""

from __future__ import annotations

import logging
from typing import Dict, Iterable, List, Optional, Sequence

import numpy as np

from . import _native
from .runtime import get_handle
from .types import Track

LOGGER = logging.getLogger(__name__)


class _HostDets:
    """Pinned staging for the float64 detections of one ``update`` call and the device mirror: box, conf, cls and
    count are carved from ONE flat buffer on each side, so the call uploads them in one copy."""

    def __init__(self, h: "_native.Handle", cap: int):
        t = h.torch
        self.cap = cap
        o_conf = cap * 32
        o_cls = o_conf + cap * 8
        o_cnt = o_cls + ((cap * 4 + 7) & ~7)
        self.nbytes = o_cnt + 8
        self.host = t.zeros(self.nbytes, dtype=t.uint8).pin_memory()
        self.dev = t.zeros(self.nbytes, dtype=t.uint8, device=h.device)
        hn = self.host.numpy()
        self.box = hn[:o_conf].view(np.float64).reshape(cap, 4)
        self.conf = hn[o_conf:o_cls].view(np.float64)
        self.cls = hn[o_cls:o_cls + cap * 4].view(np.int32)
        self.count = hn[o_cnt:o_cnt + 4].view(np.int32)
        d = self.dev
        self.soa = {"bbox_xyxy": d[:o_conf].view(t.float64).view(1, cap, 4), "conf": d[o_conf:o_cls].view(t.float64).view(1, cap),
                    "cls": d[o_cls:o_cls + cap * 4].view(t.int32).view(1, cap), "count": d[o_cnt:o_cnt + 4].view(t.int32)}
        self.o_cnt = o_cnt


class B200IouTracker:
    def __init__(self, config, handle: Optional[_native.Handle] = None):
        self.config = config
        self.h = handle if handle is not None else get_handle()
        self._slots: Dict[str, int] = {}
        self._out = None       # device result SoA of update()
        self._host_out = None  # pinned mirror
        self._in: Optional[_HostDets] = None
        self._status = None

    # ---- helpers ---------------------------------------------------------------------------
    def slot_of(self, stream_name: str) -> int:
        s = self._slots.get(stream_name)
        if s is None:
            s = self._slots[stream_name] = self.h.claim_slot()  # emptied by the handle when it is claimed
        return s

    def _cfg(self):
        c = self.config
        return int(c.max_age), int(c.min_hits), float(c.max_iou_distance)

    def reset(self, stream_name: str) -> None:
        if stream_name in self._slots:
            self.h.tracker_reset(self._slots[stream_name])

    def close(self) -> None:
        """Give the stream slots back to the handle (their tracks are dropped when the slots are claimed again)."""
        for s in self._slots.values():
            self.h.release_slot(s)
        self._slots.clear()

    def __del__(self):  # pragma: no cover
        try:
            self.close()
        except Exception:
            pass

    @staticmethod
    def tracks_from_soa(out, index: int) -> List[Track]:
        n = int(out["count"][index])
        return [Track(int(out["track_id"][index, i]), int(out["cls"][index, i]), float(out["conf"][index, i]),
                      tuple(float(v) for v in out["bbox_xyxy"][index, i]), int(out["age"][index, i]),
                      int(out["hits"][index, i])) for i in range(n)]

    @staticmethod
    def tracks_from_soa_all(host) -> List[List[Track]]:
        """All rows of a host SoA -> lists of Track objects (vectorised conversions)."""
        counts = host["count"].tolist()
        ids, cls, conf = host["track_id"].tolist(), host["cls"].tolist(), host["conf"].tolist()
        box, age, hits = host["bbox_xyxy"].tolist(), host["age"].tolist(), host["hits"].tolist()
        return [[Track(ids[b][i], cls[b][i], conf[b][i], tuple(box[b][i]), age[b][i], hits[b][i]) for i in range(n)]
                for b, n in enumerate(counts)]

    @staticmethod
    def soa_to_host(out, kmax: Optional[int] = None):
        """Device SoA -> dict of numpy arrays (one synchronising copy per field; a debugging / test helper --
        ``update`` and ``HotPathEngine`` move the whole table in one copy of its flat buffer instead)."""
        counts = out["count"].cpu().numpy()
        k = int(counts.max()) if len(counts) else 0
        if kmax is not None:
            k = min(k, kmax)
        host = {"count": counts, "new_count": out["new_count"].cpu().numpy()}
        for key in ("track_id", "cls", "conf", "bbox_xyxy", "age", "hits"):
            host[key] = out[key][:, :max(k, 1)].cpu().numpy()
        return host

    # ---- reference API ---------------------------------------------------------------------
    def update(self, stream_name: str, detections: Iterable) -> List[Track]:
        """tracker.py:50-95.  One pinned flat upload (boxes, confidences, classes, count), one launch, one flat
        read-back (track table + capacity flags).  Takes at most ``TRACKER_MAX_DETS`` (32768) detections per call and
        raises ``B200VAError`` with ``ERR_INVALID`` for more, leaving the tracker as it was (the reference takes any
        number)."""
        h, t = self.h, self.h.torch
        dets = detections if isinstance(detections, (list, tuple)) else list(detections)
        n = len(dets)
        if n > _native.TRACKER_MAX_DETS:  # checked before the staging grows: its row count is the call's max_dets
            raise _native.B200VAError(_native.ERR_INVALID, f"{n} detections in one update (at most "
                                                           f"{_native.TRACKER_MAX_DETS})")
        if self._in is None or self._in.cap < n:
            self._in = _HostDets(h, max(64, 1 << max(n - 1, 0).bit_length()))
        if self._out is None:
            self._out = h.alloc_tracks(1)
            self._host_out = h.alloc_tracks(1, pinned_host=True)
            self._host_np = {k: v.numpy() for k, v in self._host_out.items() if not k.startswith("_")}
            self._status = t.zeros(h.STATUS_WORDS, dtype=t.int32).pin_memory()
        buf = self._in
        if n:
            buf.box[:n] = [d.bbox_xyxy for d in dets]
            buf.conf[:n] = [d.confidence for d in dets]
            buf.cls[:n] = [d.class_id for d in dets]
        buf.count[0] = n
        # the used prefix of every field and the count word travel in one copy of the flat staging buffer
        buf.dev.copy_(buf.host, non_blocking=True)
        max_age, min_hits, thr = self._cfg()
        h.tracker_update([self.slot_of(stream_name)], buf.soa, max_age, min_hits, thr, f64=True, out=self._out)
        self._host_out["_flat"].copy_(self._out["_flat"], non_blocking=True)
        h.read_status_async(self._status)
        t.cuda.current_stream(h.device).synchronize()
        msg = h.status_message(self._status.tolist())
        if msg:
            raise _native.B200VAError(_native.ERR_CAPACITY, msg)
        return self.tracks_from_soa_all({k: (v[:1, :max(int(self._host_np["count"][0]), 1)] if v.ndim > 1 else v[:1])
                                         for k, v in self._host_np.items()})[0]

    # ---- batched API -----------------------------------------------------------------------
    def update_batch(self, stream_names: Sequence[str], dets, det_scale=None, skip=None, id_base=None, out=None):
        """One launch for many streams.  ``dets`` is the device SoA of ``postprocess`` (row i belongs to
        ``stream_names[i]``); ``skip[i]`` reproduces ``tracker.update(stream, [])``.  Ids are drawn
        from the shared counter in the order of ``stream_names``.  Returns the device SoA."""
        slots = [self.slot_of(s) for s in stream_names]
        max_age, min_hits, thr = self._cfg()
        return self.h.tracker_update(slots, dets, max_age, min_hits, thr, det_scale=det_scale, skip=skip,
                                     id_base=id_base, out=out)
