"""The Kafka preview downscale on NV12 frames against the ways a caller could reach it before: INTER_AREA per launch for
32 frames, and one PreviewRenderer.render end to end from a host 4K frame.

    python tools/bench_nv12_preview.py [--steps 40] [--reps 7] [--out profiles/nv12_preview.json]

Arms (32 frames per launch):
  4k_to_1080p      nv12: b200va_resize_area_u8_nv12 (the 2 x 2 vector kernel);  bgr: b200va_resize_area_u8 on frames
                   already converted with cv2.cvtColor;  round_trip: resize (INTER_LINEAR) at the frame's own size, which
                   is cvtColor on the device, into a BGR frame, then b200va_resize_area_u8 (two launches per step)
  1440p_to_1080p   the general (fractional) path, NV12 and BGR
  1080p_same_size  1 x 1 blocks, which is cvtColor itself, NV12 and BGR
  render_4k        PreviewRenderer.render of a host 4K NV12 frame (upload 1.5 B/px, one call) against host
                   cv2.cvtColor + render of the BGR frame (upload 3 B/px); host clock around each call, which ends in a
                   device synchronise; the preview images are compared before timing

Every arm's output is compared for equality with the others before anything is timed.  Kernel arms: `--steps`
back-to-back launches per CUDA-event window over rotating input sets larger than L2 (126 MB) in all, the arms' windows
alternated; the median window is reported per launch.  The launches are issued through the C ABI with argument arrays
built once, so the window times the device, not Python.  Algorithmic bytes per frame: source planes read once plus the
BGR output written once (4K -> 1080p: 12,441,600 + 6,220,800 NV12, 24,883,200 + 6,220,800 BGR; the round trip adds the
full-size BGR frame written and read again); the fraction is of the 6.45 TB/s copy peak measured on a B200
(tools/membw.cu).  The card name and power limit are read in the same run."""
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

from realtime_video_analytics_32streams_b200 import _native, sinks, synth

ap = argparse.ArgumentParser()
ap.add_argument("--steps", type=int, default=40, help="back-to-back launches (or render calls) per window")
ap.add_argument("--reps", type=int, default=7, help="windows per arm")
ap.add_argument("--out", default="")
args = ap.parse_args()

S = 32
PEAK = 6.45e12
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


def nv12_set(seed, h, w):
    """S uniform-random NV12 frames [3H/2, W] on the device, and their cvtColor twins (BGR, converted on the host)."""
    rng = np.random.default_rng(seed)
    host = [rng.integers(0, 256, size=(h * 3 // 2, w), dtype=np.uint8) for _ in range(S)]
    return ([torch.from_numpy(f).to(dev) for f in host],
            [torch.from_numpy(cv2.cvtColor(f, cv2.COLOR_YUV2BGR_NV12)).to(dev) for f in host])


def timed(fn, steps):
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record()
    for k in range(steps):
        fn(k)
    b.record()
    b.synchronize()
    return a.elapsed_time(b) / steps


def alternate(arms, steps, reps, clock=timed):
    """{name: median ms per step}, the arms' windows interleaved."""
    for fn in arms.values():  # warm every shape
        clock(fn, 2)
    got = {k: [] for k in arms}
    for _ in range(reps):
        for k, fn in arms.items():
            got[k].append(clock(fn, steps))
    return {k: statistics.median(v) for k, v in got.items()}


def report(ms, alg_bytes):
    res = {}
    for k, v in ms.items():
        bps = S * alg_bytes[k] / (v * 1e-3)
        res[k] = {"us_per_launch": round(v * 1e3, 2), "algorithmic_bytes_per_frame": alg_bytes[k],
                  "algorithmic_GBps": round(bps / 1e9, 1), "fraction_of_copy_peak": round(bps / PEAK, 3)}
    return res


class Launch:
    """One prepared resize_area call (NV12 or BGR frames -> S BGR outputs) issued straight through the C ABI."""

    def __init__(self, h, frames, dst_hw, outs):
        self.h, self.outs = h, outs
        self.fb = h._batch(frames, nv12_ok=True)
        self.dst = _native._ptr_array([o.data_ptr() for o in outs])
        self.dh, self.dw = _native._int_array([dst_hw[0]] * S), _native._int_array([dst_hw[1]] * S)
        self.st = h._stream()

    def __call__(self, _=0):
        h, fb = self.h, self.fb
        if isinstance(fb, _native.Nv12Batch):
            h._check(h.lib.b200va_resize_area_u8_nv12(h._h, fb.nv, fb.hs, fb.ws, S, self.dst, self.dh, self.dw, self.st))
        else:
            h._check(h.lib.b200va_resize_area_u8(h._h, fb.ptrs, fb.hs, fb.ws, fb.pitch, S, self.dst, self.dh, self.dw,
                                                 self.st))


class LinearLaunch:
    """resize (INTER_LINEAR) of NV12 frames at their own size: cvtColor on the device, into persistent BGR frames."""

    def __init__(self, h, frames, outs):
        self.h, self.outs = h, outs
        self.fb = h._batch(frames, nv12_ok=True)
        self.dst = _native._ptr_array([o.data_ptr() for o in outs])
        self.st = h._stream()

    def __call__(self, _=0):
        h, fb = self.h, self.fb
        h._check(h.lib.b200va_resize_linear_u8_nv12(h._h, fb.nv, fb.hs, fb.ws, S, None, self.dst, fb.hs, fb.ws, self.st))


def same(a, b):
    return all(torch.equal(x, y) for x, y in zip(a, b))


def outputs(dst_hw):
    return [torch.empty((*dst_hw, 3), dtype=torch.uint8, device=dev) for _ in range(S)]


def kernel_arms(h, src_hw, dst_hw, round_trip=False):
    H, W = src_hw
    nv_bytes, bgr_bytes, out_bytes = H * W * 3 // 2, H * W * 3, dst_hw[0] * dst_hw[1] * 3
    n_sets = max(2, -(-300_000_000 // (S * nv_bytes)))  # NV12 sets alone: > 2 x L2 in all
    sets = [nv12_set(100 * H + k, H, W) for k in range(n_sets)]
    o_nv, o_bgr, o_rt = outputs(dst_hw), outputs(dst_hw), outputs(dst_hw)
    nv = [Launch(h, s[0], dst_hw, o_nv) for s in sets]
    bgr = [Launch(h, s[1], dst_hw, o_bgr) for s in sets]
    arms = {"nv12": lambda i: nv[i % n_sets](), "bgr": lambda i: bgr[i % n_sets]()}
    alg = {"nv12": nv_bytes + out_bytes, "bgr": bgr_bytes + out_bytes}
    if round_trip:
        full = outputs(src_hw)
        lin = [LinearLaunch(h, s[0], full) for s in sets]
        rt = Launch(h, full, dst_hw, o_rt)

        def rt_step(i):
            lin[i % n_sets]()
            rt()

        arms["round_trip"] = rt_step
        alg["round_trip"] = nv_bytes + 2 * bgr_bytes + out_bytes
    for k in range(n_sets):
        for fn in arms.values():
            fn(k)
        torch.cuda.synchronize()
        assert same(o_nv, o_bgr), (src_hw, k)
        if round_trip:
            assert same(o_nv, o_rt), (src_hw, k)
    res = {"input_sets": n_sets, "outputs_equal": True}
    res.update(report(alternate(arms, args.steps, args.reps), alg))
    if round_trip:
        res["nv12_over_bgr_time"] = round(res["nv12"]["us_per_launch"] / res["bgr"]["us_per_launch"], 3)
        res["nv12_over_round_trip_time"] = round(res["nv12"]["us_per_launch"] / res["round_trip"]["us_per_launch"], 3)
    return res


def host_clock(fn, steps):
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    for k in range(steps):
        fn(k)
    torch.cuda.synchronize()
    return (time.perf_counter() - t0) * 1e3 / steps


def render(h):
    """One PreviewRenderer.render of a 4K frame with four tracks (GPU drawing path), from host memory."""
    bgr_scene = synth.MotionScene(7, 2160, 3840).frame(0)
    i420 = cv2.cvtColor(bgr_scene, cv2.COLOR_BGR2YUV_I420)
    y, u, v = i420[:2160], i420[2160:2700].reshape(1080, 1920), i420[2700:].reshape(1080, 1920)
    nv = np.concatenate([y, np.stack([u, v], axis=2).reshape(1080, 3840)])
    tracks = [{"track_id": 3 + k, "class_id": k, "bbox_xyxy": (200.0 + 900 * k, 300.0, 700.0 + 900 * k, 900.0)} for k in range(4)]
    r_nv, r_bgr = sinks.PreviewRenderer(h), sinks.PreviewRenderer(h)
    arms = {"nv12": lambda i: r_nv.render(nv, tracks),
            "host_cvtcolor_bgr": lambda i: r_bgr.render(cv2.cvtColor(nv, cv2.COLOR_YUV2BGR_NV12), tracks)}
    assert np.array_equal(arms["nv12"](0), arms["host_cvtcolor_bgr"](0))
    ms = alternate(arms, max(args.steps // 4, 4), args.reps, clock=host_clock)
    res = {"outputs_equal": True, "cpu_cores": os.cpu_count(), "cv2_threads": cv2.getNumThreads()}
    for k, v in ms.items():
        res[k] = {"ms_per_frame": round(v, 3)}
    res["nv12_over_bgr_time"] = round(ms["nv12"] / ms["host_cvtcolor_bgr"], 3)
    return res


def main():
    h = _native.Handle(device=0, max_batch=S, max_anchors=256, max_candidates=256, max_dets=64, max_streams=8, max_tracks=64)
    res = {"card": card(), "steps": args.steps, "reps": args.reps, "frames_per_launch": S, "copy_peak_Bps": PEAK}
    res["4k_to_1080p"] = kernel_arms(h, (2160, 3840), (1080, 1920), round_trip=True)
    torch.cuda.empty_cache()
    res["1440p_to_1080p"] = kernel_arms(h, (1440, 2560), (1080, 1920))
    torch.cuda.empty_cache()
    res["1080p_same_size"] = kernel_arms(h, (1080, 1920), (1080, 1920))
    res["render_4k"] = render(h)
    h.poll_status()
    h.close()
    print(json.dumps(res))
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            json.dump(res, f, indent=1)


if __name__ == "__main__":
    main()
