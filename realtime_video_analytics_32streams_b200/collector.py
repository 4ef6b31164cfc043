"""In-pipeline tick collector (SURVEY.md §8f-1): one batched tick for all of the reference's stream workers.

The reference runs one asyncio task per stream (pipeline.py:460-515); each task awaits
``StreamWorker._process_packet`` (pipeline.py:143-212) for every packet, and that method calls
``detector.predict`` / ``tracker.update`` synchronously for ONE frame.  Behind ``backend: b200`` that reaches the
kernels at batch 1, 32 times per frame period.

``TickCollector`` turns those 32 independent calls into one ``HotPathEngine.tick``:

* every worker hands its packet to ``collector.process(stream_name, packet)`` and awaits the result; a worker has at
  most one packet outstanding (the reference's own back-pressure: the ``async for`` loop does not pull the next
  packet before ``_process_packet`` returns);
* a tick fires when every registered stream has a packet waiting, or ``max_wait_s`` after the first packet of the
  tick arrived (a slow or stalled camera never holds the others back: it simply contributes ``None`` to that tick);
* the tick itself (upload, ROI / downsample / motion / adaptive gates, letterbox, forward, decode + NMS, tracker,
  result read-back) runs on the collector's own thread, so the event loop keeps receiving frames meanwhile;
* each worker then does, for its own stream and on the event loop, exactly what the reference does after
  ``predict`` / ``update``: ``metrics.update_counters`` (pipeline.py:184-189 / 216-221), ``kafka.send_tracks``
  (pipeline.py:190-195), ``_maybe_save_snapshot``, the mirrored adaptive-FPS fields, ``health.update_success(dt)``
  (pipeline.py:200-201) or ``health.update_error()`` (pipeline.py:205).

``install(pipeline_module, engine_factory)`` patches the reference's ``AnalyticsPipeline`` / ``StreamWorker`` in
place (``register_with_reference(..., batched=True)`` calls it); nothing else of the reference changes.
"""

from __future__ import annotations

import asyncio
import logging
import threading
import time
from concurrent.futures import ThreadPoolExecutor
from typing import Callable, Dict, List, Optional, Sequence

LOGGER = logging.getLogger(__name__)


class TickCollector:
    """Gathers the newest packet of every stream and runs them through ``engine.tick`` as one batch.

    ``engine`` needs ``streams`` (objects with ``.name``, fixed order) and
    ``tick(frames, frame_ids) -> list of per-stream results`` (``None`` frame = stream absent this tick; the result list
    holds one entry per PRESENT stream, in stream order) -- ``HotPathEngine`` has exactly this shape."""

    def __init__(self, engine, max_wait_s: float = 0.010):
        self.engine = engine
        self.names: List[str] = [s.name for s in engine.streams]
        self._index: Dict[str, int] = {n: i for i, n in enumerate(self.names)}
        self.max_wait_s = float(max_wait_s)
        self._pending: Dict[str, tuple] = {}      # stream -> (packet, future)
        self._expected = set(self.names)          # streams that are still delivering (see retire())
        self._wake: Optional[asyncio.Event] = None
        self._task: Optional[asyncio.Task] = None
        self._pool = ThreadPoolExecutor(max_workers=1, thread_name_prefix="b200va-tick")
        self._closed = False
        self.ticks = 0
        self.frames = 0
        self.last_tick_s = 0.0                    # wall time of the last engine.tick (for dashboards / tests)
        self._lock = threading.Lock()

    # ---- worker side ---------------------------------------------------------------------
    async def process(self, stream_name: str, packet):
        """Queue ``packet`` for the next tick and wait for this stream's result."""
        if self._closed:
            raise RuntimeError("TickCollector is closed")
        if stream_name not in self._index:
            raise KeyError(f"stream '{stream_name}' is not part of this collector's engine")
        if stream_name in self._pending:
            raise RuntimeError(f"stream '{stream_name}' already has a packet waiting (one outstanding packet per worker)")
        loop = asyncio.get_running_loop()
        if self._task is None or self._task.done():
            self._wake = asyncio.Event()
            self._task = loop.create_task(self._run(), name="b200va-tick-collector")
        fut = loop.create_future()
        self._pending[stream_name] = (packet, fut)
        self._expected.add(stream_name)
        self._wake.set()
        return await fut

    def retire(self, stream_name: str) -> None:
        """The stream ended (or its worker is reconnecting): stop waiting for it when deciding that a tick is full."""
        self._expected.discard(stream_name)
        if self._wake is not None:
            self._wake.set()

    # ---- collector task ------------------------------------------------------------------
    def _full(self) -> bool:
        return bool(self._pending) and all(n in self._pending for n in self._expected)

    async def _run(self) -> None:
        loop = asyncio.get_running_loop()
        while not self._closed:
            if not self._pending:
                self._wake.clear()
                await self._wake.wait()
                continue
            deadline = loop.time() + self.max_wait_s
            while not self._full():
                left = deadline - loop.time()
                if left <= 0:
                    break
                self._wake.clear()
                try:
                    await asyncio.wait_for(self._wake.wait(), timeout=left)
                except asyncio.TimeoutError:
                    break
            batch, self._pending = self._pending, {}
            frames: List[Optional[object]] = [None] * len(self.names)
            ids: List[int] = [0] * len(self.names)
            for name, (packet, _) in batch.items():
                frames[self._index[name]] = packet.frame
                ids[self._index[name]] = int(getattr(packet, "frame_id", 0))
            t0 = time.perf_counter()
            try:
                results = await loop.run_in_executor(self._pool, self.engine.tick, frames, ids)
            except BaseException as exc:  # every waiting worker sees the failure (pipeline.py:203-212 logs and re-raises)
                for _, fut in batch.values():
                    if not fut.done():
                        fut.set_exception(exc if isinstance(exc, Exception) else RuntimeError(repr(exc)))
                if isinstance(exc, asyncio.CancelledError):
                    raise
                continue
            self.last_tick_s = time.perf_counter() - t0
            self.ticks += 1
            self.frames += len(batch)
            by_name = {r.stream_name: r for r in results}
            for name, (_, fut) in batch.items():
                if fut.done():
                    continue
                r = by_name.get(name)
                if r is None:
                    fut.set_exception(RuntimeError(f"engine returned no result for stream '{name}'"))
                else:
                    fut.set_result(r)

    async def close(self) -> None:
        self._closed = True
        if self._task is not None:
            self._task.cancel()
            try:
                await self._task
            except (asyncio.CancelledError, Exception):
                pass
        for _, fut in self._pending.values():
            if not fut.done():
                fut.cancel()
        self._pending.clear()
        self._pool.shutdown(wait=True)


# ------------------------------------------------------------------------------------------------
# the reference-side patch
# ------------------------------------------------------------------------------------------------
def make_process_packet(collector_of: Callable):
    """Builds the replacement for ``StreamWorker._process_packet`` (pipeline.py:143-212).  ``collector_of(worker)``
    returns the TickCollector serving that worker."""

    async def _process_packet(self, packet) -> None:
        self._frame_index += 1
        start_time = time.time()
        name = packet.stream.name
        try:
            r = await collector_of(self).process(name, packet)
            if r.processed:
                tracks = r.tracks
                self.ctx.metrics.update_counters(stream=name, frames_processed=1, detections_emitted=r.n_detections,
                                                 active_tracks=len(tracks))
                # a sink that reads result tables (B200KafkaSink) gets the FrameResult, anything else the Track objects
                payload = r if getattr(self.ctx.kafka, "accepts_results", False) else tracks
                await self.ctx.kafka.send_tracks(stream_name=name, frame_id=packet.frame_id, tracks=payload,
                                                 frame=packet.frame)
                self._maybe_save_snapshot(packet, tracks)
            else:  # pipeline.py:214-222 (_skip_frame): counters only, nothing is published
                self.ctx.metrics.update_counters(stream=name, frames_processed=1, detections_emitted=0,
                                                 active_tracks=r.n_tracks)
            # the adaptive-FPS state lives in the engine (it gates on the device side of the tick); mirror it so that
            # anything that inspects the worker sees the reference's fields (pipeline.py:104-113, 242-262)
            st = getattr(r, "adaptive_state", None)
            if st is not None:
                self._process_every, self._idle_frames = st
            self.ctx.health.update_success(time.time() - start_time)
        except Exception as exc:
            self.ctx.health.update_error()
            LOGGER.error("Error processing frame %d for stream '%s': %s", getattr(packet, "frame_id", -1), name, exc)
            raise

    return _process_packet


def install(rpipe, engine_factory: Callable, max_wait_s: float = 0.010) -> None:
    """Patch the reference's pipeline module so that its stream workers share one tick.

    ``engine_factory(streams, detector, pipeline_config) -> engine`` builds the batched engine for the streams that use
    one detector instance (the reference allows a ``detector_id`` per stream, pipeline.py:468-482: there is one
    collector per detector object, all of them on the pipeline's single tracker handle)."""
    if getattr(rpipe.StreamWorker, "_b200va_batched", False):
        return
    orig_init = rpipe.AnalyticsPipeline.__init__
    orig_worker_init = rpipe.StreamWorker.__init__
    orig_wait_closed = rpipe.AnalyticsPipeline.wait_closed
    orig_run = rpipe.StreamWorker.run

    def pipeline_init(self, config):
        orig_init(self, config)
        self._b200va = {"config": config, "collectors": {}, "factory": engine_factory, "max_wait_s": max_wait_s}
        self.tracker._b200va_pipeline = self  # the worker context carries the tracker, not the pipeline (pipeline.py:64-72)

    def collector_of(worker) -> TickCollector:
        pipe = getattr(worker.ctx.tracker, "_b200va_pipeline", None)
        if pipe is None:
            raise RuntimeError("batched mode: the worker's tracker does not belong to a patched AnalyticsPipeline")
        reg = pipe._b200va
        key = id(worker.ctx.detector)
        col = reg["collectors"].get(key)
        if col is None:
            cfg = reg["config"]
            default = cfg.detector
            streams = []
            for s in cfg.streams:
                if not s.enabled:
                    continue
                # the same selection rule as pipeline.py:472-482: a stream follows `detector_id`, else the default
                det_cfg = cfg.detectors.get(s.detector_id, default) if s.detector_id else default
                if det_cfg is worker.ctx.detector.config:
                    streams.append(s)
            if worker.ctx.stream not in streams:
                streams.append(worker.ctx.stream)
            col = reg["collectors"][key] = TickCollector(reg["factory"](streams, worker.ctx.detector, cfg), reg["max_wait_s"])
        return col

    def worker_init(self, context):
        orig_worker_init(self, context)

    async def worker_run(self):
        try:
            await orig_run(self)
        finally:  # the stream ended or was cancelled: do not let the others wait for it
            pipe = getattr(self.ctx.tracker, "_b200va_pipeline", None)
            if pipe is not None:
                col = pipe._b200va["collectors"].get(id(self.ctx.detector))
                if col is not None:
                    col.retire(self.ctx.stream.name)

    async def wait_closed(self):
        await orig_wait_closed(self)
        for col in list(getattr(self, "_b200va", {}).get("collectors", {}).values()):
            await col.close()

    rpipe.AnalyticsPipeline.__init__ = pipeline_init
    rpipe.AnalyticsPipeline.wait_closed = wait_closed
    rpipe.StreamWorker.__init__ = worker_init
    rpipe.StreamWorker.run = worker_run
    rpipe.StreamWorker._process_packet = make_process_packet(collector_of)
    rpipe.StreamWorker._b200va_batched = True


def default_engine_factory(streams: Sequence, detector, pipeline_config):
    """``HotPathEngine`` over ``streams`` with the pipeline's detector: its forward, thresholds, handle and semantics (a
    ``B200UltralyticsDetector`` gives an engine that runs LetterBox / non_max_suppression / scale_boxes)."""
    from .engine import HotPathEngine

    return HotPathEngine(streams, detector.config, pipeline_config.tracker, infer=detector._infer_fn, on_overflow="warn",
                         detector=detector)
