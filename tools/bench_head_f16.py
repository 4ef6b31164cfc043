"""float16 heads on one GPU: the decode reading an fp16 head in place (B200VA_HEAD_F16) against today's conversion
pass (head.float()) followed by the float32 decode, and the 32 x 1080p tick with either head.

    python tools/bench_head_f16.py [--steps 24] [--reps 9] [--out profiles/head_f16.json]

Workload: 32 heads of [84, 8400] from synth.DenseScene (bench.py's), 4 rotating input sets.  Every timed window
starts with a 512 MB fill, so L2 holds no head and is full of dirty lines (as after a real tick's letterbox).  Arms,
alternated within every repetition:
  (a) fp32 head, float32 decode;
  (b) fp16 head, head.float() + float32 decode (one event pair around both);
  (c) fp16 head decoded in place.
Each window is `--steps` back-to-back b200va_postprocess calls with a confidence threshold no score reaches (the full
decode pass; the NMS launch finds no candidate and returns), as bench.py's decode roofline does.  The decode phase
alone (b200va_set_profiling events around the decode launch) is reported for (a) and (c).  The tick is bench.py's
(letterbox || decode -> NMS -> tracker, default schedule) replayed from one CUDA graph per input set, with the fp32
and the fp16 head alternated.  Algorithmic bytes of one decode pass: 32 * 84 * 8400 * 4 = 90,316,800 B (fp32) and
45,158,400 B (fp16).  Detections of (a), (b) and (c) at the real thresholds are compared bit for bit first."""
import argparse
import json
import os
import subprocess
import sys

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import numpy as np
import torch

from realtime_video_analytics_32streams_b200 import _native, synth

ap = argparse.ArgumentParser()
ap.add_argument("--steps", type=int, default=24, help="back-to-back calls (or tick replays) per timed window")
ap.add_argument("--reps", type=int, default=9, help="windows per arm")
ap.add_argument("--out", default="")
args = ap.parse_args()

STREAMS, C, A, N_SETS = 32, 84, 8400, 4
H, W, IN_HW = 1080, 1920, (640, 640)
CONF, IOU = 0.35, 0.5
TRK = (30, 1, 0.5)  # max_age, min_hits, max_iou_distance
dev = torch.device("cuda", 0)


def card():
    """Device name and power limit, read in this run."""
    name = torch.cuda.get_device_name(0)
    limit = None
    try:
        import pynvml

        pynvml.nvmlInit()
        limit = pynvml.nvmlDeviceGetPowerManagementLimit(pynvml.nvmlDeviceGetHandleByIndex(0)) / 1000.0
    except Exception:
        try:
            q = subprocess.run(["nvidia-smi", "--query-gpu=power.limit", "--format=csv,noheader,nounits", "-i", "0"],
                               stdout=subprocess.PIPE, text=True, timeout=30).stdout.strip()
            limit = float(q.splitlines()[0])
        except Exception:
            pass
    return {"device": name, "power_limit_w": limit}


def tables(d):
    return {k: v.cpu().numpy().copy() for k, v in d.items() if not k.startswith("_")}


def same(a, b):
    if not np.array_equal(a["count"], b["count"]):
        return False
    for i, n in enumerate(a["count"]):
        for key in ("bbox_xyxy", "conf", "cls"):
            if not np.array_equal(a[key][i, :n].view(np.uint8), b[key][i, :n].view(np.uint8)):
                return False
    return True


def main():
    info = card()
    heads_np = np.stack([np.stack([synth.DenseScene(7000 + s, n_objects=24, dup=3, n_obj_classes=10).head(t)
                                   for s in range(STREAMS)]) for t in range(N_SETS)])  # [sets, 32, C, A]
    # the fp32 arm decodes the float32 widening of the fp16 head: one model output in two dtypes
    h16 = [torch.from_numpy(heads_np[k].astype(np.float16)).to(dev) for k in range(N_SETS)]
    h32 = [x.float() for x in h16]
    h = _native.Handle(device=0, max_batch=STREAMS, max_anchors=A, max_candidates=2048, max_dets=512,
                       max_streams=2 * STREAMS, max_tracks=4096)
    metas = (_native.Letterbox * STREAMS)(*[_native.letterbox_meta(H, W, *IN_HW) for _ in range(STREAMS)])
    dets = h.alloc_dets(STREAMS)
    filler = torch.empty(512 << 20, dtype=torch.uint8, device=dev)

    arms = {
        "a_fp32_decode": lambda k, thr: h.postprocess(h32[k % N_SETS], metas, thr, IOU, filter_conf=CONF, out=dets),
        "b_fp16_float_then_fp32_decode": lambda k, thr: h.postprocess(h16[k % N_SETS].float(), metas, thr, IOU,
                                                                      filter_conf=CONF, out=dets),
        "c_fp16_decode_in_place": lambda k, thr: h.postprocess(h16[k % N_SETS], metas, thr, IOU, filter_conf=CONF,
                                                               out=dets),
    }
    # identical detections of the three arms, every input set, real thresholds
    identical = True
    for k in range(N_SETS):
        got = {}
        for name, fn in arms.items():
            fn(k, CONF)
            torch.cuda.synchronize()
            got[name] = tables(dets)
        identical &= all(same(got["a_fp32_decode"], v) for v in got.values())
    n_dets = int(got["c_fp16_decode_in_place"]["count"].sum())
    h.poll_status()

    # back-to-back windows, arms alternated within each repetition
    for name, fn in arms.items():  # warm-up
        for k in range(4):
            fn(k, 2.0)
    torch.cuda.synchronize()
    b2b = {name: [] for name in arms}
    for r in range(args.reps):
        for name, fn in arms.items():
            filler.fill_(r & 1)
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            for k in range(args.steps):
                fn(k, 2.0)
            e1.record()
            torch.cuda.synchronize()
            b2b[name].append(e0.elapsed_time(e1) / args.steps)
    # the decode phase alone (events around the decode launch), (a) and (c) alternated
    h.set_profiling(True)
    h.phase_times()
    phase = {"a_fp32_decode": [], "c_fp16_decode_in_place": []}
    for r in range(args.reps * 4):
        for name in phase:
            filler.fill_(r & 1)
            arms[name](r, 2.0)
            phase[name].append(h.phase_times()["decode"])
    h.set_profiling(False)
    h.poll_status()

    # the 32 x 1080p tick by graph replay, fp32 against fp16 head
    g = torch.Generator(device=dev)
    g.manual_seed(1234)
    frame_sets = [torch.randint(0, 256, (STREAMS, H, W, 3), dtype=torch.uint8, device=dev, generator=g)
                  for _ in range(N_SETS)]
    batches = [_native.FrameBatch(list(fs.unbind(0))) for fs in frame_sets]
    nets = [torch.empty((STREAMS, 3, *IN_HW), dtype=torch.float32, device=dev) for _ in range(N_SETS)]
    tracks = h.alloc_tracks(STREAMS)
    slots = _native._int_array(list(range(STREAMS)))

    def capture(heads):
        plans = [h.plan_tick(frames=batches[k], net_out=nets[k], dst_hw=IN_HW, head=heads[k], metas=metas,
                             conf_thr=CONF, iou_thr=IOU, filter_conf=CONF, dets=dets, slots=slots, tracker_cfg=TRK,
                             tracks=tracks) for k in range(N_SETS)]
        for k in range(N_SETS):  # warm every plan eagerly first
            h.tick(plans[k])
        torch.cuda.synchronize()
        side = torch.cuda.Stream()
        side.wait_stream(torch.cuda.current_stream())
        graphs = []
        with torch.cuda.stream(side):
            for plan in plans:
                gr = torch.cuda.CUDAGraph()
                with torch.cuda.graph(gr, stream=side):
                    h.tick(plan)
                graphs.append(gr)
        torch.cuda.current_stream().wait_stream(side)
        torch.cuda.synchronize()
        return plans, graphs

    tick_arms = {"tick_fp32_head": capture(h32), "tick_fp16_head": capture(h16)}
    for _, graphs in tick_arms.values():
        for k in range(2 * N_SETS):
            graphs[k % N_SETS].replay()
    torch.cuda.synchronize()
    tick = {name: [] for name in tick_arms}
    for r in range(args.reps):
        for name, (_, graphs) in tick_arms.items():
            filler.fill_(r & 1)
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            for k in range(args.steps):
                graphs[k % N_SETS].replay()
            e1.record()
            torch.cuda.synchronize()
            tick[name].append(e0.elapsed_time(e1) / args.steps)
    h.poll_status()
    h.close()

    def stat(v):
        return {"median_us": round(float(np.median(v)) * 1e3, 2), "min_us": round(float(np.min(v)) * 1e3, 2),
                "max_us": round(float(np.max(v)) * 1e3, 2)}

    bytes32, bytes16 = STREAMS * C * A * 4, STREAMS * C * A * 2
    res = {"metric": "fp16 head decode", **info, "shape": [STREAMS, C, A], "input_sets": N_SETS,
           "steps_per_window": args.steps, "windows": args.reps, "l2": "512 MB fill before every window",
           "algorithmic_bytes": {"fp32_head": bytes32, "fp16_head": bytes16},
           "identical_detections": bool(identical), "detections_in_set": n_dets,
           "per_call_back_to_back": {k: stat(v) for k, v in b2b.items()},
           "decode_phase": {k: stat(v) for k, v in phase.items()},
           "tick_graph_replay": {k: stat(v) for k, v in tick.items()}}
    for k, nbytes in (("a_fp32_decode", bytes32), ("c_fp16_decode_in_place", bytes16)):
        res["decode_phase"][k]["GBps"] = round(nbytes / (float(np.median(phase[k])) * 1e-3) / 1e9, 1)
    print(json.dumps(res))
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            json.dump(res, f, indent=1)
    if not identical:
        raise SystemExit("bench_head_f16: the arms' detections differ")


if __name__ == "__main__":
    main()
