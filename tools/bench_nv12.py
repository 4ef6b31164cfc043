"""NV12 frames against BGR frames on one GPU: the letterbox per launch, the graph-replayed tick, HotPathEngine end to
end from pinned host frames, and the host-side cv2.cvtColor a caller holding NV12 no longer runs.

    python tools/bench_nv12.py [--steps 40] [--reps 7] [--out profiles/nv12.json]

Every arm is compared for equality (bytes / float bit patterns) with its BGR twin on cv2.cvtColor(frame,
COLOR_YUV2BGR_NV12) before anything is timed.  Letterbox arms: `--steps` back-to-back launches per CUDA-event window over
rotating input sets whose total is larger than L2 (126 MB), NV12 and BGR windows alternated; the median window is
reported per launch.  Algorithmic bytes per frame into 640 x 640 float32 (tapped source rows + the 4,915,200-byte
output), from oracle.cv_restate.linear_taps: 1080p 6,988,800 (BGR) / 6,297,600 (NV12), 4K 13,209,600 / 9,062,400;
the fraction is of the 6.45 TB/s copy peak measured on a B200 (tools/membw.cu).  The card name and power limit are
read in the same run."""
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

from realtime_video_analytics_32streams_b200 import _native, synth

ap = argparse.ArgumentParser()
ap.add_argument("--steps", type=int, default=40, help="back-to-back launches (or replays, or engine ticks) per window")
ap.add_argument("--reps", type=int, default=7, help="windows per arm")
ap.add_argument("--out", default="")
args = ap.parse_args()

S, IN_HW = 32, (640, 640)
PEAK = 6.45e12
ALG = {"1080p": {"bgr": 6_988_800, "nv12": 6_297_600}, "4k": {"bgr": 13_209_600, "nv12": 9_062_400}}
SIZES = {"1080p": (1080, 1920), "4k": (2160, 3840)}
dev = torch.device("cuda", 0)


def card():
    name = torch.cuda.get_device_name(0)
    limit = None
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=power.limit", "--format=csv,noheader,nounits", "-i", "0"],
                           stdout=subprocess.PIPE, text=True, timeout=30).stdout.strip()
        limit = float(q.splitlines()[0])
    except Exception:
        pass
    return {"device": name, "power_limit_w": limit}


def bgr_of(nv12):
    """The BGR twin of an NV12 frame: the conversion the NV12 entry points are byte-identical to."""
    return cv2.cvtColor(nv12, cv2.COLOR_YUV2BGR_NV12)


def nv12_frames(seed, n, h, w):
    rng = np.random.default_rng(seed)
    return [rng.integers(0, 256, size=(h * 3 // 2, w), dtype=np.uint8) for _ in range(n)]


def timed(fn, steps):
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record()
    for k in range(steps):
        fn(k)
    b.record()
    b.synchronize()
    return a.elapsed_time(b) / steps


def alternate(arms, steps, reps):
    """{name: median ms per step}, the arms' windows interleaved."""
    for fn in arms.values():  # warm every shape
        timed(fn, 2)
    got = {k: [] for k in arms}
    for _ in range(reps):
        for k, fn in arms.items():
            got[k].append(timed(fn, steps))
    return {k: statistics.median(v) for k, v in got.items()}


def same(a, b):
    return a.shape == b.shape and torch.equal(a.contiguous().view(torch.uint8), b.contiguous().view(torch.uint8))


def letterbox(h, size):
    H, W = SIZES[size]
    per_set = S * H * W * 3
    n_sets = max(2, -(-300_000_000 // per_set))  # BGR sets: > 2 x L2 in all
    nv = [[torch.from_numpy(f).to(dev) for f in nv12_frames(10 + k, S, H, W)] for k in range(n_sets)]
    bgr = [[torch.from_numpy(bgr_of(f.cpu().numpy())).to(dev) for f in fs] for fs in nv]
    nb = [_native.Nv12Batch(fs) for fs in nv]
    bb = [_native.FrameBatch(fs) for fs in bgr]
    out_n = torch.empty((S, 3, *IN_HW), dtype=torch.float32, device=dev)
    out_b = torch.empty_like(out_n)
    for k in range(n_sets):
        h.preprocess(nb[k], IN_HW, _native.OUT_F32_RGB_NCHW, out=out_n)
        h.preprocess(bb[k], IN_HW, _native.OUT_F32_RGB_NCHW, out=out_b)
        assert same(out_n, out_b), (size, k)
    ms = alternate({"nv12": lambda i: h.preprocess(nb[i % n_sets], IN_HW, _native.OUT_F32_RGB_NCHW, out=out_n),
                    "bgr": lambda i: h.preprocess(bb[i % n_sets], IN_HW, _native.OUT_F32_RGB_NCHW, out=out_b)},
                   args.steps, args.reps)
    res = {"input_sets": n_sets, "outputs_equal": True}
    for k, v in ms.items():
        bps = S * ALG[size][k] / (v * 1e-3)
        res[k] = {"us_per_launch": round(v * 1e3, 2), "algorithmic_GBps": round(bps / 1e9, 1),
                  "fraction_of_copy_peak": round(bps / PEAK, 3)}
    res["nv12_over_bgr_time"] = round(ms["nv12"] / ms["bgr"], 3)
    return res


def tick(h):
    H, W = SIZES["1080p"]
    nv = [torch.from_numpy(f).to(dev) for f in nv12_frames(40, S, H, W)]
    bgr = [torch.from_numpy(bgr_of(f.cpu().numpy())).to(dev) for f in nv]
    head = torch.from_numpy(np.stack([synth.synth_head(60 + s, 84, 8400, 12, dup=3) for s in range(S)])).to(dev)
    metas = [_native.letterbox_meta(H, W, *IN_HW) for _ in range(S)]
    res, nets, rows, graphs = {}, {}, {}, {}
    for kind, frames in (("nv12", nv), ("bgr", bgr)):
        net = torch.zeros((S, 3, *IN_HW), dtype=torch.float32, device=dev)
        h.tracker_set_next_id(1)
        for s in range(S):
            h.tracker_reset(s)
        plan = h.plan_tick(frames=frames, net_out=net, dst_hw=IN_HW, head=head, metas=metas, conf_thr=0.35, iou_thr=0.5,
                           filter_conf=0.35, slots=list(range(S)), tracker_cfg=(30, 1, 0.5))
        h.tick(plan)
        torch.cuda.synchronize()
        nets[kind], rows[kind] = net.clone(), plan.tracks["_flat"].clone()
        side = torch.cuda.Stream()
        side.wait_stream(torch.cuda.current_stream())
        with torch.cuda.stream(side):
            g = torch.cuda.CUDAGraph()
            with torch.cuda.graph(g, stream=side):
                h.tick(plan)
        torch.cuda.current_stream().wait_stream(side)
        torch.cuda.synchronize()
        graphs[kind] = (g, plan, net)
    assert same(nets["nv12"], nets["bgr"]) and torch.equal(rows["nv12"], rows["bgr"])
    ms = alternate({k: (lambda i, g=g: g[0].replay()) for k, g in graphs.items()}, args.steps, args.reps)
    for k, v in ms.items():
        res[k] = {"us_per_tick": round(v * 1e3, 2)}
    res["outputs_equal"] = True
    return res


def engine(h, config):
    from realtime_video_analytics_32streams_b200 import DetectorConfig, HotPathEngine, StreamConfig, TrackerConfig

    H, W = SIZES["1080p" if config == "bench" else "4k"]
    streams = []
    for s in range(S):
        kw = {}
        if config == "4k_roi_motion":
            kw = dict(roi_polygons=synth.synth_polygons(600 + s, H, W), motion_filter=True, motion_threshold=0.0)
        streams.append(StreamConfig(name=f"cam{s:02d}", **kw))
    head = torch.from_numpy(np.stack([synth.synth_head(80 + s, 84, 8400, 12, dup=3) for s in range(S)])).to(dev)
    n_sets = 2
    nv_host = [[torch.from_numpy(f).pin_memory() for f in nv12_frames(90 + k, S, H, W)] for k in range(n_sets)]
    bgr_host = [[torch.from_numpy(bgr_of(f.numpy())).pin_memory() for f in fs] for fs in nv_host]
    res = {}
    engines, results = {}, {}
    for kind, sets in (("nv12", nv_host), ("bgr", bgr_host)):
        h.tracker_set_next_id(1)
        eng = HotPathEngine(streams, DetectorConfig(confidence_threshold=0.35, iou_threshold=0.5),
                            TrackerConfig(max_age=30, max_iou_distance=0.5, min_hits=1),
                            infer=lambda t: head[:t.shape[0]], handle=h, input_hw=IN_HW)
        results[kind] = [[(r.processed, r.n_detections, r.n_tracks, r.track_arrays["track_id"].tolist())
                          for r in eng.tick(sets[k])] for k in range(n_sets)]
        engines[kind] = (eng, sets)
        for s in streams:
            eng.tracker.reset(s.name)
    assert results["nv12"] == results["bgr"], config
    for kind, (eng, sets) in engines.items():
        for k in range(2):
            eng.tick(sets[k])  # warm
        torch.cuda.synchronize()
        b0 = eng.stager.bytes_moved
        times = []
        for _ in range(args.reps):
            t0 = time.perf_counter()
            for i in range(args.steps // 4):
                eng.tick(sets[i % n_sets])
            torch.cuda.synchronize()
            times.append((time.perf_counter() - t0) / (args.steps // 4))
        ticks = args.reps * (args.steps // 4)
        dt = statistics.median(times)
        res[kind] = {"ms_per_tick": round(dt * 1e3, 3), "frames_per_s": round(S / dt, 1),
                     "bus_bytes_per_tick": (eng.stager.bytes_moved - b0) // ticks}
    res["outputs_equal"] = True
    return res


def cvtcolor():
    res = {"cpu_cores": os.cpu_count(), "cv2_threads": cv2.getNumThreads()}
    for size, (H, W) in SIZES.items():
        f = nv12_frames(5, 1, H, W)[0]
        for k in range(3):
            cv2.cvtColor(f, cv2.COLOR_YUV2BGR_NV12)
        n = 30
        t0 = time.perf_counter()
        for _ in range(n):
            cv2.cvtColor(f, cv2.COLOR_YUV2BGR_NV12)
        dt = (time.perf_counter() - t0) / n
        res[size] = {"ms_per_frame": round(dt * 1e3, 3), "ms_per_32_frames": round(32 * dt * 1e3, 2)}
    return res


def main():
    h = _native.Handle(device=0, max_batch=S, max_anchors=8400, max_candidates=2048, max_dets=512, max_streams=2 * S,
                       max_tracks=1024)
    res = {"card": card(), "steps": args.steps, "reps": args.reps}
    res["letterbox_32x1080p"] = letterbox(h, "1080p")
    res["letterbox_32x4k"] = letterbox(h, "4k")
    res["tick_32x1080p_graph"] = tick(h)
    res["engine_bench_config"] = engine(h, "bench")
    res["engine_32x4k_roi_motion"] = engine(h, "4k_roi_motion")
    res["host_cvtcolor_nv12_to_bgr"] = cvtcolor()
    h.poll_status()
    h.close()
    print(json.dumps(res))
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            json.dump(res, f, indent=1)


if __name__ == "__main__":
    main()
