"""The in-pipeline tick collector (SURVEY.md §8f-1, collector.py).

CPU part: workers patched with the collector's ``_process_packet`` share one tick per frame period and reproduce, per
stream, what the reference's own ``StreamWorker`` objects (pipeline.py:88-262) did one frame at a time, as stored in
tests/golden/pipeline.npz -- processed or skipped, the published track table (ids, boxes, hits), the counters, the
health calls and the adaptive-FPS fields.  The engine behind the collector is an oracle-backed stand-in there (no
GPU); the GPU part runs the same collector over the real ``HotPathEngine``.
"""
import asyncio
import types

import numpy as np
import pytest

import golden_util as G
from oracle import hotpath as O
from realtime_video_analytics_32streams_b200 import synth
from realtime_video_analytics_32streams_b200.collector import TickCollector, make_process_packet
from realtime_video_analytics_32streams_b200.types import StreamConfig

H, W, IN_HW = 108, 192, (64, 64)
CONF, IOU = 0.35, 0.5
N_STREAMS, N_FRAMES = 4, 20
POLYS = [[(10, 8), (180, 12), (170, 100), (20, 95)]]


def _stream_kwargs(i):
    return dict(name=f"cam{i}", roi_polygons=POLYS if i % 2 == 0 else None, motion_filter=(i != 3),
                motion_threshold=0.02, downsample_ratio=1.0 if i != 1 else 0.75, adaptive_fps=True, target_fps=25,
                min_target_fps=5, idle_frame_tolerance=3)


def _scene(i):
    return synth.MotionScene(61 + i, H, W, rect=30, speed=11, static=(i == 2))


def _head(i, t):
    n_obj = 5 if (i != 2 and (t < 6 or t > 13)) else 0
    return synth.synth_head(7000 + 10 * t + i, 20, 256, n_obj, dup=2, input_hw=IN_HW)[None]


class Recorder:
    """Stub sinks: record every call a worker makes, per stream."""

    def __init__(self):
        self.calls = []

    def update_counters(self, **kw):
        self.calls.append(("metrics", kw["stream"], kw["frames_processed"], kw["detections_emitted"], kw["active_tracks"]))

    async def send_tracks(self, stream_name, frame_id, tracks, frame=None):
        arr = G.tracks_arrays(list(tracks))
        self.calls.append(("kafka", stream_name, frame_id, {k: v.copy() for k, v in arr.items()}, frame is not None))


class Health:
    def __init__(self, log, name):
        self.log, self.name = log, name

    def update_success(self, dt):
        assert dt >= 0.0
        self.log.append(("health_ok", self.name))

    def update_error(self):
        self.log.append(("health_err", self.name))


class OracleEngine:
    """Stand-in for HotPathEngine on a box without a GPU: same ``streams`` / ``tick`` contract, CPU oracle inside."""

    def __init__(self, streams, conf, iou, trk_cfg, head_fn):
        self.streams = list(streams)
        self.t = {s.name: 0 for s in self.streams}
        tracker = O.IouTracker(*trk_cfg)
        self.workers = {}
        for i, s in enumerate(self.streams):
            spec = O.StreamSpec(name=s.name, roi_polygons=s.roi_polygons, motion_filter=s.motion_filter,
                                motion_threshold=s.motion_threshold, downsample_ratio=s.downsample_ratio,
                                adaptive_fps=s.adaptive_fps, target_fps=s.target_fps, min_target_fps=s.min_target_fps,
                                idle_frame_tolerance=s.idle_frame_tolerance)
            self.workers[s.name] = O.StreamWorker(spec, (lambda tensor, idx, i=i, n=s.name: head_fn(i, self.t[n])), tracker,
                                                  conf, iou, None, IN_HW, False, backend="cv2")
        self.batches = []

    def tick(self, frames, frame_ids=None):
        out = []
        self.batches.append([f is not None for f in frames])
        for i, (s, f) in enumerate(zip(self.streams, frames)):
            if f is None:
                continue
            self.t[s.name] = frame_ids[i]
            w = self.workers[s.name]
            r = w.process(f)
            out.append(types.SimpleNamespace(stream_name=s.name, frame_id=frame_ids[i], processed=r.processed,
                                             skip_reason=r.skip_reason, n_detections=len(r.detections),
                                             n_tracks=len(r.tracks), tracks=r.tracks, detections=r.detections,
                                             adaptive_state=(w.process_every, w.idle_frames)))
        return out


class _Packet:
    def __init__(self, stream, frame, frame_id):
        self.stream, self.frame, self.frame_id = stream, frame, frame_id


def test_collector_workers_reproduce_the_reference_workers_per_frame_trace():
    """Workers patched with the collector's ``_process_packet``, both streams sharing one tick per frame period, against
    what the reference's own ``StreamWorker._process_packet`` did one frame at a time on the same inputs
    (tests/golden/pipeline.npz, tests/golden/make_golden.py): per frame whether it was processed, the adaptive-FPS
    fields and the stream's track table, which is what the worker publishes."""
    z = G.load("pipeline")
    h, w, ih, iw = z["pipe_cfg"].tolist()
    polys = [[tuple(p) for p in z["pipe_polys"].tolist()]]
    scenes = [synth.MotionScene(61, h, w, rect=30, speed=11), synth.MotionScene(62, h, w, static=True)]
    burst = synth.MotionScene(63, h, w, rect=30, speed=11)
    streams = [StreamConfig(name=f"cam{i}", roi_polygons=polys if i == 0 else None, motion_filter=True, motion_threshold=0.02,
                            downsample_ratio=1.0 if i == 0 else 0.75, adaptive_fps=True, target_fps=25, min_target_fps=5,
                            idle_frame_tolerance=3) for i in range(2)]

    def head(i, t):
        n_obj = 5 if ((i == 0 or 8 <= t <= 12) and t < 14) else 0
        return synth.synth_head(7000 + 10 * t + i, 20, 256, n_obj, dup=2, input_hw=(ih, iw))[None]

    def frame(i, t):
        return (burst if (i == 1 and 8 <= t <= 12) else scenes[i]).frame(t)

    assert (ih, iw) == IN_HW
    eng = OracleEngine(streams, CONF, IOU, (3, 0.5, 1), head)
    col = TickCollector(eng, max_wait_s=5.0)
    rec, log = Recorder(), []
    proc = make_process_packet(lambda wk: col)
    workers = [types.SimpleNamespace(ctx=types.SimpleNamespace(metrics=rec, kafka=rec, health=Health(log, s.name)),
                                     _frame_index=0, _maybe_save_snapshot=lambda *a, **k: None, _process_every=1,
                                     _idle_frames=0) for s in streams]
    n = int(z["pipe_n"][0])
    n_frames = n // len(streams)

    async def drive():
        for t in range(n_frames):
            n_calls = len(rec.calls)
            await asyncio.gather(*[proc(wk, _Packet(s, frame(i, t), t)) for i, (s, wk) in enumerate(zip(streams, workers))])
            calls = rec.calls[n_calls:]
            for i, (s, wk) in enumerate(zip(streams, workers)):
                k = t * len(streams) + i
                zi, zt, processed, pe, idle = z[f"pipe_{k}_hdr"].tolist()
                assert (zi, zt) == (i, t)
                assert [G.sha(frame(i, t)), G.sha(head(i, t))] == z[f"pipe_{k}_sha"].tolist(), "synthetic generator drifted"
                want = {kk: z[f"pipe_{k}_t{kk}"] for kk in ("id", "cls", "conf", "box", "age", "hits")}
                sent = [c for c in calls if c[0] == "kafka" and c[1] == s.name]
                metrics = [c for c in calls if c[0] == "metrics" and c[1] == s.name]
                assert len(metrics) == 1 and metrics[0][2] == 1, (t, s.name)
                assert len(sent) == int(processed), (t, s.name)
                if processed:
                    assert sent[0][2] == t and metrics[0][4] == len(want["id"])
                    for kk, v in want.items():
                        assert np.array_equal(sent[0][3][kk], v), (t, s.name, kk)
                assert (wk._process_every, wk._idle_frames, wk._frame_index) == (pe, idle, t + 1), (t, s.name)
        assert col.ticks == n_frames and col.frames == n
        await col.close()

    asyncio.run(drive())
    assert all(all(b) for b in eng.batches)
    assert log == [("health_ok", s.name) for _ in range(n_frames) for s in streams]


def test_collector_partial_ticks_errors_and_retired_streams():
    """A late stream does not hold a tick back longer than max_wait_s, an engine failure reaches every waiting worker
    (and is counted by its health tracker), and a retired stream is not waited for."""
    names = ["a", "b", "c"]
    streams = [types.SimpleNamespace(name=n) for n in names]

    class Engine:
        def __init__(self):
            self.streams, self.seen, self.fail = streams, [], False

        def tick(self, frames, ids):
            if self.fail:
                raise ValueError("boom")
            self.seen.append([f is not None for f in frames])
            return [types.SimpleNamespace(stream_name=s.name, processed=True, n_detections=1, n_tracks=2, tracks=[], frame_id=i,
                                          adaptive_state=None) for s, f, i in zip(streams, frames, ids) if f is not None]

    eng = Engine()
    col = TickCollector(eng, max_wait_s=0.05)
    log, rec = [], Recorder()
    proc = make_process_packet(lambda w: col)
    workers = [types.SimpleNamespace(ctx=types.SimpleNamespace(metrics=rec, kafka=rec, health=Health(log, n)), _frame_index=0,
                                     _maybe_save_snapshot=lambda *a, **k: None, _process_every=1, _idle_frames=0) for n in names]

    async def drive():
        # tick 1: only a and b deliver -> fires after max_wait_s without c
        await asyncio.gather(*[proc(workers[i], _Packet(streams[i], np.zeros((2, 2, 3), np.uint8), 1)) for i in (0, 1)])
        assert eng.seen == [[True, True, False]]
        # c retires: a tick of a and b is now "full" immediately
        col.retire("c")
        col.max_wait_s = 30.0
        await asyncio.wait_for(asyncio.gather(*[proc(workers[i], _Packet(streams[i], np.zeros((2, 2, 3), np.uint8), 2))
                                                for i in (0, 1)]), timeout=5.0)
        assert eng.seen[-1] == [True, True, False]
        # a second packet of the same stream before the tick is refused (one outstanding packet per worker)
        eng.fail = True
        res = await asyncio.gather(*[proc(workers[i], _Packet(streams[i], np.zeros((2, 2, 3), np.uint8), 3)) for i in (0, 1)],
                                   return_exceptions=True)
        assert all(isinstance(r, ValueError) for r in res)
        eng.fail = False
        with pytest.raises(KeyError):
            await col.process("nope", _Packet(streams[0], None, 0))
        await col.close()
        with pytest.raises(RuntimeError):
            await col.process("a", _Packet(streams[0], None, 0))

    asyncio.run(drive())
    assert [c for c in log if c[0] == "health_err"] == [("health_err", "a"), ("health_err", "b")]
    assert sum(1 for c in log if c[0] == "health_ok") == 4 and col.ticks == 2


@pytest.mark.gpu
def test_collector_over_the_gpu_engine_matches_the_oracle_pipeline():
    import torch
    from realtime_video_analytics_32streams_b200 import (DetectorConfig, HotPathEngine, StreamConfig, TrackerConfig,
                                                         _native)

    h = _native.Handle(device=0, max_batch=N_STREAMS, max_anchors=256, max_candidates=256, max_dets=64,
                       max_streams=N_STREAMS, max_tracks=128)
    try:
        streams = [StreamConfig(**_stream_kwargs(i)) for i in range(N_STREAMS)]
        tick = {"t": 0}
        eng = HotPathEngine(streams, DetectorConfig(confidence_threshold=CONF, iou_threshold=IOU),
                            TrackerConfig(max_age=3, max_iou_distance=0.5, min_hits=1),
                            infer=lambda tensor: torch.from_numpy(
                                np.concatenate([_head(i, tick["t"]) for i in eng.active_streams])).to(h.device),
                            handle=h, input_hw=IN_HW)
        ora = OracleEngine(streams, CONF, IOU, (3, 0.5, 1), _head)
        col = TickCollector(eng, max_wait_s=5.0)
        scenes = [_scene(i) for i in range(N_STREAMS)]

        async def drive():
            for t in range(N_FRAMES):
                tick["t"] = t
                frames = [scenes[i].frame(t) for i in range(N_STREAMS)]
                got = await asyncio.gather(*[col.process(s.name, _Packet(s, frames[i], t)) for i, s in enumerate(streams)])
                want = ora.tick(frames, [t] * N_STREAMS)
                for g, w in zip(got, want):
                    assert (g.stream_name, g.processed, g.skip_reason, g.n_detections, g.n_tracks, g.adaptive_state) == \
                           (w.stream_name, w.processed, w.skip_reason, w.n_detections, w.n_tracks, w.adaptive_state), (t, g.stream_name)
                    ga, wa = G.tracks_arrays(g.tracks), G.tracks_arrays(w.tracks)
                    for k in wa:
                        assert np.array_equal(ga[k], wa[k]), (t, g.stream_name, k)
            assert col.ticks == N_FRAMES
            await col.close()

        asyncio.run(drive())
        h.poll_status()
    finally:
        h.close()
