"""The Ultralytics backend batched against the per-stream path it replaces, on one GPU: 32 x 1080p streams with a fixed
[32, 84, 5040] decoded head standing in for the model (LetterBox(auto=True) gives 1080p a 384 x 640 input).

    python tools/bench_ultralytics.py [--ticks 20] [--reps 5] [--out profiles/ultralytics_batched.json]

1. Per tick of 32 frames: B200UltralyticsDetector.predict + B200IouTracker.update once per stream (what a pipeline on
   `backend: b200_ultralytics` runs without batching) against HotPathEngine.tick in Ultralytics mode, from CUDA frames
   and from pinned host BGR / NV12 frames; host clock around work that ends in a synchronise, with the bytes put on the
   bus per tick (FrameStager.bytes_moved).
2. b200va_tick_ultralytics at schedule 6 against preprocess_geom + postprocess_ultralytics + tracker_update called one
   after another, eager and as replayed CUDA graphs; CUDA events over `--ticks` back-to-back calls.

Every batched arm is compared with its unbatched twin before it is timed.  The card name and power limit are read in
the same run."""
import argparse
import json
import os
import statistics
import subprocess
import sys
import time

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import cv2
import numpy as np
import torch

from realtime_video_analytics_32streams_b200 import (B200IouTracker, B200UltralyticsDetector, DetectorConfig, FramePacket,
                                                     HotPathEngine, StreamConfig, TrackerConfig, _native, synth)

ap = argparse.ArgumentParser()
ap.add_argument("--ticks", type=int, default=20, help="ticks (or calls, or replays) per timed window")
ap.add_argument("--reps", type=int, default=5, help="windows per arm (median reported)")
ap.add_argument("--out", default="")
args = ap.parse_args()

S, HW, IN, IN_HW, A = 32, (1080, 1920), (640, 640), (384, 640), 5040
CONF, IOU, TRK = 0.35, 0.5, (30, 1, 0.5)
if not torch.cuda.is_available():
    sys.exit("bench_ultralytics needs a CUDA device")
dev = torch.device("cuda", 0)


def card():
    limit = None
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=power.limit", "--format=csv,noheader,nounits", "-i", "0"],
                           stdout=subprocess.PIPE, text=True, timeout=30).stdout.strip()
        limit = float(q.splitlines()[0])
    except Exception:
        pass
    return {"device": torch.cuda.get_device_name(0), "power_limit_w": limit}


def handle():
    return _native.Handle(device=0, max_batch=S, max_anchors=8400, max_candidates=4096, max_dets=1024, max_streams=S,
                          max_tracks=512)


HEAD = torch.from_numpy(np.stack([synth.synth_head(500 + s, 84, A, 12, dup=3, input_hw=IN_HW) for s in range(S)])).to(dev)
NV12 = [np.random.default_rng(40 + s).integers(0, 256, size=(HW[0] * 3 // 2, HW[1]), dtype=np.uint8) for s in range(S)]
BGR = [cv2.cvtColor(f, cv2.COLOR_YUV2BGR_NV12) for f in NV12]
FRAMES = {"cuda": [torch.from_numpy(f).to(dev) for f in BGR], "host_bgr": [torch.from_numpy(f).pin_memory() for f in BGR],
          "host_nv12": [torch.from_numpy(f).pin_memory() for f in NV12]}
STREAMS = [StreamConfig(name=f"cam{s}") for s in range(S)]
DCFG = DetectorConfig(confidence_threshold=CONF, iou_threshold=IOU, backend="b200_ultralytics")
TCFG = TrackerConfig(max_age=TRK[0], min_hits=TRK[1], max_iou_distance=TRK[2])


def per_stream_arm(frames):
    """The unbatched path: one predict and one tracker update per stream."""
    h = handle()
    box = {"s": 0}
    det = B200UltralyticsDetector(DCFG, input_hw=IN, handle=h, infer=lambda t: HEAD[box["s"]:box["s"] + 1])
    trk = B200IouTracker(TCFG, handle=h)

    def tick():
        out = []
        for s, f in enumerate(frames):
            box["s"] = s
            out.append(trk.update(STREAMS[s].name, det.predict(FramePacket(STREAMS[s], f, 0))))
        torch.cuda.synchronize()
        return out

    return tick, det._stager, h


def engine_arm(frames):
    h = handle()
    det = B200UltralyticsDetector(DCFG, input_hw=IN, handle=h, infer=lambda t: HEAD[:t.shape[0]])
    eng = HotPathEngine(STREAMS, DCFG, TCFG, infer=None, detector=det)

    def tick():
        res = eng.tick(list(frames))
        return [r.tracks for r in res]

    return tick, eng.stager, h


def host_windows(fn, reps, ticks):
    ms = []
    for _ in range(reps):
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        for _ in range(ticks):
            fn()
        torch.cuda.synchronize()
        ms.append((time.perf_counter() - t0) * 1e3 / ticks)
    return statistics.median(ms)


def rows(tracks):
    return [[(x.track_id, x.class_id, x.confidence, x.bbox_xyxy, x.age, x.hits) for x in st] for st in tracks]


result = {"card": card(), "streams": S, "frame_hw": HW, "in_hw": IN_HW, "head": [S, 84, A], "engine": {}, "tick": {}}
for kind, frames in FRAMES.items():
    ps, ps_stager, h1 = per_stream_arm(frames)
    en, en_stager, h2 = engine_arm(frames)
    assert rows(ps()) == rows(en()), f"{kind}: the engine differs from the per-stream path"
    for _ in range(2):  # warm up every shape
        ps()
        en()
    b0, e0 = ps_stager.bytes_moved, en_stager.bytes_moved
    ps()
    en()
    bus_ps, bus_en = ps_stager.bytes_moved - b0, en_stager.bytes_moved - e0
    t_ps_l, t_en_l = [], []
    for _ in range(args.reps):  # the two arms alternated
        t_ps_l.append(host_windows(ps, 1, max(args.ticks // 4, 1)))
        t_en_l.append(host_windows(en, 1, args.ticks))
    t_ps, t_en = statistics.median(t_ps_l), statistics.median(t_en_l)
    result["engine"][kind] = {"per_stream_ms_per_tick": round(t_ps, 3), "engine_ms_per_tick": round(t_en, 3),
                              "per_stream_frames_per_s": round(S * 1e3 / t_ps, 1),
                              "engine_frames_per_s": round(S * 1e3 / t_en, 1),
                              "per_stream_bus_bytes_per_tick": int(bus_ps), "engine_bus_bytes_per_tick": int(bus_en)}
    print(kind, result["engine"][kind], flush=True)
    h1.close()
    h2.close()

# ---- b200va_tick_ultralytics against the three calls ----------------------------------------------------------------
for nv12 in (False, True):
    h = handle()
    h.tracker_set_next_id(1)
    m = _native.letterbox_meta_ultralytics(*HW, *IN, True, 32)[0]
    src = [torch.from_numpy(f).to(dev) for f in (NV12 if nv12 else BGR)]
    net = torch.zeros((S, 3, *IN_HW), dtype=torch.float32, device=dev)
    dets, tracks = h.alloc_dets(S), h.alloc_tracks(S)
    plan = h.plan_tick(frames=src, net_out=net, dst_hw=IN_HW, head=HEAD, conf_thr=CONF, iou_thr=IOU, filter_conf=CONF,
                       dets=dets, slots=list(range(S)), tracker_cfg=TRK, schedule=_native.SCHEDULE_AUTO, tracks=tracks,
                       ultralytics=dict(geoms=[m] * S, frame_hw=[HW] * S, in_hw=IN_HW))
    h2 = handle()
    h2.tracker_set_next_id(1)
    net2 = torch.zeros_like(net)
    dets2, tracks2 = h2.alloc_dets(S), h2.alloc_tracks(S)
    fb = _native.Nv12Batch(src) if nv12 else _native.FrameBatch(src)
    slots = _native._int_array(range(S))

    def separate():
        h2.preprocess_geom(fb, [m] * S, IN_HW, out=net2)
        h2.postprocess_ultralytics(HEAD, [HW] * S, IN_HW, CONF, IOU, filter_conf=CONF, out=dets2)
        h2.tracker_update(slots, dets2, *TRK, out=tracks2)

    h.tick(plan)
    separate()
    torch.cuda.synchronize()
    for k in ("count", "cls", "conf", "bbox_xyxy"):
        assert torch.equal(dets[k], dets2[k]), k
    for k in ("count", "track_id", "bbox_xyxy", "hits"):
        assert torch.equal(tracks[k], tracks2[k]), k
    assert torch.equal(net, net2)
    graphs = []
    side = torch.cuda.Stream()
    side.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(side):
        for fn in (lambda: h.tick(plan), separate):
            g = torch.cuda.CUDAGraph()
            with torch.cuda.graph(g, stream=side):
                fn()
            graphs.append(g)
    torch.cuda.current_stream().wait_stream(side)
    torch.cuda.synchronize()
    arms = {"tick_eager": lambda: h.tick(plan), "separate_eager": separate, "tick_graph": graphs[0].replay,
            "separate_graph": graphs[1].replay}
    got = {k: [] for k in arms}
    for fn in arms.values():
        fn()
    for _ in range(args.reps):
        for k, fn in arms.items():
            a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            a.record()
            for _ in range(args.ticks):
                fn()
            b.record()
            b.synchronize()
            got[k].append(a.elapsed_time(b) * 1e3 / args.ticks)
    result["tick"]["nv12" if nv12 else "bgr"] = {k: round(statistics.median(v), 1) for k, v in got.items()}
    print("tick us", "nv12" if nv12 else "bgr", result["tick"]["nv12" if nv12 else "bgr"], flush=True)
    h.poll_status()
    h2.poll_status()
    h.close()
    h2.close()

print(json.dumps(result))
if args.out:
    with open(args.out, "w") as f:
        json.dump(result, f, indent=1)
