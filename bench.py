#!/usr/bin/env python
"""Benchmark of the pre + post + track hot path (BASELINE.json metric).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl reference] [--schedule 0..6] [--no-graph] [--no-cpu]
                    [--dump-outputs DIR]

Workload at every N: each GPU serves 32 streams of 1080p BGR frames with a synthetic decoded
YOLOv8 head [32, 84, 8400] (config 3 of BASELINE.json, the one the metric is quoted on); with
N > 1 every rank (one process per GPU, torchrun) serves its own 32 streams -- weak scaling, no
data-path collective.  One "step" is one tick: letterbox preprocess of the 32 frames, head decode +
NMS of the 32 heads, tracker update of the 32 streams -- one prepared `b200va_tick` call (letterbox on
the caller's stream, decode -> NMS -> tracker on the library's second stream, fork and join inside the
call).  The detector forward is outside the measured path (north_star): the head tensors stand in
for its output.

`value`   : frames/s with frames and heads already resident in HBM (CUDA events around exactly K timed
            steps, max over ranks).  The tick is replayed from a CUDA graph per input set.  Four rotating
            input sets keep every step's reads out of the 126 MB L2.
`--dump-outputs DIR`: after the K timed steps, rank 0 writes what the last of them handed its caller
            (letterbox tensor as a fixed seeded sample, detection and track tables) as DIR/<name>.npy in
            float32 / float64.  Inputs depend only on the arguments, so two builds compare output for output.
`roofline`: the letterbox kernel's algorithmic bytes / its event-timed duration vs the measured HBM peak.
`e2e`     : the same tick through the public API (HotPathEngine.submit / collect, two ticks in flight)
            with HOST buffers: pinned frames and heads are copied to the device and the result tables
            are read back inside the timed region.
`cpu_baseline` / `--impl reference`: the reference's own OpenCV/NumPy call sequence (oracle, cv2
            back end) on the host cores of the same box (one thread / one process per core).
Informational keys: value_eager_tick, value_three_serial_calls (the unfused call sequence),
value_pad_rows_written_once (B200VA_OUT_FLAG_PADS_VALID), value_32_streams_total_strong_scaling (N > 1).
"""

from __future__ import annotations

import argparse
import json
import os
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

from realtime_video_analytics_32streams_b200 import synth  # noqa: E402

METRIC = "pre+post+track frames/sec (32x1080p)"
STREAMS = 32
H, W = 1080, 1920
IN_HW = (640, 640)
C, A = 84, 8400
CONF, IOU = 0.35, 0.5
TRK = dict(max_age=30, max_iou_distance=0.5, min_hits=1)
N_SETS = 4  # rotating input sets: every step reads frames / heads that left L2 long ago
OBJECTS, DUP = 24, 3
# algorithmic HBM bytes of the letterbox kernel per 1080p frame (SURVEY.md §8d): the 360 tapped
# source rows (every third row carries weight 2048, the rest 0) + the fp32 NCHW output
LETTERBOX_BYTES_PER_FRAME = 360 * 1920 * 3 + 3 * 640 * 640 * 4


def workload_config(n_gpus: int) -> dict:
    return {"workload": "32 streams x 1080p BGR per GPU -> letterbox 640x640 fp32 + YOLOv8 head [32,84,8400] decode/NMS "
                        "+ IoU tracker (BASELINE.json configs[2] shape, 32 streams on every GPU)",
            "streams_per_gpu": STREAMS, "streams_total": STREAMS * n_gpus, "frame": [H, W, 3], "head": [C, A],
            "objects_per_frame": OBJECTS * DUP, "conf_thr": CONF, "iou_thr": IOU, "tracker": TRK,
            "cache": f"{N_SETS} rotating input sets (199 MB frames + 90 MB heads each) > 126 MB L2",
            "sharding": "by stream id, no collective"}


def make_heads(stream: int, n_sets: int) -> np.ndarray:
    scene = synth.DenseScene(7000 + stream, n_objects=OBJECTS, dup=DUP, n_obj_classes=10)
    return np.stack([scene.head(t) for t in range(n_sets)])


# --------------------------------------------------------------------------------------------
# clocks
# --------------------------------------------------------------------------------------------
class ClockSampler:
    def __init__(self, device_index: int, period_s: float = 0.002):
        self.samples, self.reasons, self.max_mhz = [], set(), None
        self.period_s = period_s
        self._stop = threading.Event()
        self._thread = None
        try:
            import pynvml

            pynvml.nvmlInit()
            # honour CUDA_VISIBLE_DEVICES when mapping the torch ordinal to an NVML index
            vis = os.environ.get("CUDA_VISIBLE_DEVICES")
            idx = device_index
            if vis:
                try:
                    idx = int(vis.split(",")[device_index])
                except (ValueError, IndexError):
                    idx = device_index
            self.nv = pynvml
            self.dev = pynvml.nvmlDeviceGetHandleByIndex(idx)
            self.max_mhz = pynvml.nvmlDeviceGetMaxClockInfo(self.dev, pynvml.NVML_CLOCK_SM)
        except Exception:  # pragma: no cover
            self.nv = None

    def _poll(self):
        nv = self.nv
        names = {"hw_slowdown": 0x8, "sw_power_cap": 0x4, "hw_thermal_slowdown": 0x40, "sw_thermal_slowdown": 0x20,
                 "hw_power_brake_slowdown": 0x80}
        while not self._stop.is_set():
            try:
                self.samples.append(nv.nvmlDeviceGetClockInfo(self.dev, nv.NVML_CLOCK_SM))
                try:
                    r = nv.nvmlDeviceGetCurrentClocksEventReasons(self.dev)
                except Exception:
                    r = nv.nvmlDeviceGetCurrentClocksThrottleReasons(self.dev)
                for k, bit in names.items():
                    if r & bit:
                        self.reasons.add(k)
            except Exception:
                pass
            self._stop.wait(self.period_s)

    def start(self):
        if self.nv is not None:
            self._stop.clear()
            self._thread = threading.Thread(target=self._poll, daemon=True)
            self._thread.start()

    def stop(self):
        if self._thread is not None:
            self._stop.set()
            self._thread.join()
            self._thread = None

    def summary(self) -> dict:
        med = float(np.median(self.samples)) if self.samples else None
        return {"sm_mhz": med, "sm_max_mhz": self.max_mhz, "reasons": sorted(self.reasons), "samples": len(self.samples)}


# --------------------------------------------------------------------------------------------
# CPU arm: the reference's OpenCV / NumPy call sequence (oracle, cv2 back end)
# --------------------------------------------------------------------------------------------
_W = {}


def _cpu_worker_init(stream_ids, n_sets):
    import cv2

    from oracle import hotpath as O

    cv2.setNumThreads(1)
    _W["O"] = O
    _W["frames"] = {s: synth.synth_frame(3000 + s, H, W) for s in stream_ids}
    _W["heads"] = {s: make_heads(s, n_sets) for s in stream_ids}
    _W["tracker"] = O.IouTracker(TRK["max_age"], TRK["max_iou_distance"], TRK["min_hits"])


def _cpu_tick(args):
    stream_ids, t = args
    O = _W["O"]
    n_tracks = 0
    for s in stream_ids:
        tensor, meta = O.preprocess(_W["frames"][s], IN_HW, False, backend="cv2")
        heads = _W["heads"][s]
        dets = O.postprocess(heads[t % len(heads)][None], meta, CONF, IOU)
        dets = O.filter_detections(dets, CONF)
        n_tracks += len(_W["tracker"].update(f"s{s}", dets))
    return n_tracks


def cpu_single_core_sample(budget_s: float = 10.0, n_streams: int = 4) -> dict:
    """Bounded single-thread sample of the same workload (rank 0, N=1 only)."""
    ids = list(range(n_streams))
    _cpu_worker_init(ids, N_SETS)
    _cpu_tick((ids, 0))  # warm-up
    t0 = time.perf_counter()
    ticks = 0
    while True:
        _cpu_tick((ids, ticks + 1))
        ticks += 1
        if time.perf_counter() - t0 > budget_s or ticks >= 2000:
            break
    dt = time.perf_counter() - t0
    return {"value": round(ticks * n_streams / dt, 2), "unit": "frames/s", "cores": 1, "kind": "port",
            "sample": f"{ticks} ticks x {n_streams} streams of the bench workload (1080p letterbox + [84,8400] decode/NMS + "
                      f"tracker), oracle with the cv2 back end (the reference's own OpenCV/NumPy call sequence), "
                      f"1 thread, {dt:.1f} s"}


def run_reference(args) -> None:
    """--impl reference: the CPU path on every host core (rank 0 only under torchrun)."""
    rank = int(os.environ.get("RANK", 0))
    if rank != 0:
        return
    import multiprocessing as mp

    cores = len(os.sched_getaffinity(0)) if hasattr(os, "sched_getaffinity") else (os.cpu_count() or 1)
    procs = max(1, min(cores, STREAMS))
    # a step = one tick of a bounded number of streams, spread evenly over the worker processes
    streams_per_proc = 1 if procs >= 8 else 2
    groups = [[p * streams_per_proc + k for k in range(streams_per_proc)] for p in range(procs)]
    n_frames = procs * streams_per_proc
    ctx = mp.get_context("fork")
    pools = [ctx.Pool(1, initializer=_cpu_worker_init, initargs=(g, N_SETS)) for g in groups]

    def tick(t):
        res = [pool.apply_async(_cpu_tick, ((g, t),)) for pool, g in zip(pools, groups)]
        for r in res:
            r.get()

    for t in range(args.warmup):
        tick(t)
    t0 = time.perf_counter()
    for t in range(args.steps):
        tick(args.warmup + t)
    dt = time.perf_counter() - t0
    for pool in pools:
        pool.terminate()
    value = n_frames * args.steps / dt
    sample = (f"each step = one tick of {n_frames} of the {STREAMS} streams ({streams_per_proc} per process, {procs} processes, "
              f"1 OpenCV thread each); same frames/heads/thresholds as the GPU arm")
    line = {"impl": "reference", "metric": METRIC, "value": round(value, 2), "unit": "frames/s", "n_gpus": args.gpus,
            "steps": args.steps, "warmup": args.warmup, "ms_per_step": round(1e3 * dt / args.steps, 3),
            "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "u8/f32", "data": "synthetic",
            "config": workload_config(args.gpus),
            "cpu_baseline": {"value": round(value, 2), "unit": "frames/s", "cores": procs, "kind": "port", "sample": sample},
            "e2e": {"value": round(value, 2), "unit": "frames/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}
    print(json.dumps(line), flush=True)


# --------------------------------------------------------------------------------------------
# GPU arm
# --------------------------------------------------------------------------------------------
WINDOWS = 15          # K-step windows of the N > 1 strong-scaling variant; its median window is reported
KERNEL_SAMPLES = 24   # eager ticks with per-kernel CUDA-event pairs (b200va_set_profiling), whatever --steps is
HEAD_BYTES_PER_FRAME = C * A * 4
DUMP_NET_SAMPLES = 1 << 21  # letterbox elements --dump-outputs writes (of 32 x 3 x 640 x 640)


def dump_outputs(out_dir: str, net, dets: dict, tracks: dict) -> None:
    """The arrays one tick hands its caller, as float32 / float64 .npy files: the letterbox tensor as a fixed
    seeded sample of its elements (with their flat indices), every field of the detection and track tables.
    Table rows past a stream's `count` hold nothing a caller may read and are written as 0."""
    import torch

    os.makedirs(out_dir, exist_ok=True)
    flat = net.reshape(-1)
    idx = np.sort(np.random.default_rng(0).choice(flat.numel(), DUMP_NET_SAMPLES, replace=False))
    arrays = {"letterbox_sample": flat[torch.from_numpy(idx).to(flat.device)].cpu().numpy(),
              "letterbox_sample_index": idx.astype(np.float64)}
    for prefix, table in (("dets", dets), ("tracks", tracks)):
        host = {k: v.cpu().numpy() for k, v in table.items() if not k.startswith("_")}
        for name, v in host.items():
            v = v.astype(np.float32 if v.dtype == np.float32 else np.float64)
            if v.ndim > 1:  # [streams, rows(, width)]
                v[np.arange(v.shape[1])[None, :] >= host["count"][:, None]] = 0
            arrays[f"{prefix}_{name}"] = v
    for name, v in arrays.items():
        np.save(os.path.join(out_dir, f"{name}.npy"), v)


def _capture(torch, h, plans):
    """One CUDA graph per prepared tick (fork / join and programmatic dependent launches included)."""
    side = torch.cuda.Stream()
    side.wait_stream(torch.cuda.current_stream())
    graphs = []
    l0 = h.launch_count
    with torch.cuda.stream(side):
        for plan in plans:
            gr = torch.cuda.CUDAGraph()
            with torch.cuda.graph(gr, stream=side):
                plan.set_events(None, None)
                h.tick(plan)
            graphs.append(gr)
    torch.cuda.current_stream().wait_stream(side)
    return graphs, (h.launch_count - l0) // max(len(plans), 1)


def parity_check(torch, h, frame_sets, heads_np, plans, nets, tracks, dets) -> dict:
    """Two ticks from an empty tracker (input sets 0 and 1) compared with the CPU oracle: every network-input tensor
    bit for bit, every detection table, every track table (ids, classes, boxes, hits).  The oracle is only the checker
    here; nothing it computes is timed or shipped."""
    from oracle import hotpath as O

    for s in range(STREAMS):
        h.tracker_reset(s)
    h.tracker_set_next_id(1)
    ora = O.IouTracker(TRK["max_age"], TRK["max_iou_distance"], TRK["min_hits"])
    checked = {"ticks": 2, "streams": STREAMS, "letterbox_tensors": 0, "detections": 0, "tracks": 0}
    for t in range(2):
        h.tick(plans[t])
        torch.cuda.synchronize()
        got_net = nets[t].cpu().numpy()
        d = {k: v.cpu().numpy() for k, v in dets.items() if not k.startswith("_")}
        tr = {k: v.cpu().numpy() for k, v in tracks.items() if not k.startswith("_")}
        frames = frame_sets[t].cpu().numpy()
        for s in range(STREAMS):
            tensor, meta = O.preprocess(frames[s], IN_HW, False, backend="cv2")
            if not np.array_equal(got_net[s].view(np.uint8), tensor[0].view(np.uint8)):
                raise SystemExit(f"bench parity: letterbox tensor of stream {s}, tick {t} differs from the oracle")
            want_d = O.filter_detections(O.postprocess(heads_np[t][s][None], meta, CONF, IOU), CONF)
            n = int(d["count"][s])
            if n != len(want_d) or not np.array_equal(
                    d["bbox_xyxy"][s, :n], np.array([w.bbox_xyxy for w in want_d], dtype=np.float32).reshape(n, 4)) \
                    or d["cls"][s, :n].tolist() != [w.class_id for w in want_d] \
                    or not np.array_equal(d["conf"][s, :n], np.array([w.confidence for w in want_d], dtype=np.float32)):
                raise SystemExit(f"bench parity: detections of stream {s}, tick {t} differ from the oracle")
            want_t = ora.update(f"s{s}", want_d)
            m = int(tr["count"][s])
            if m != len(want_t) or tr["track_id"][s, :m].tolist() != [w.track_id for w in want_t] \
                    or tr["cls"][s, :m].tolist() != [w.class_id for w in want_t] \
                    or tr["hits"][s, :m].tolist() != [w.hits for w in want_t] \
                    or not np.array_equal(tr["bbox_xyxy"][s, :m],
                                          np.array([w.bbox_xyxy for w in want_t], dtype=np.float32).reshape(m, 4)):
                raise SystemExit(f"bench parity: track table of stream {s}, tick {t} differs from the oracle")
            checked["letterbox_tensors"] += 1
            checked["detections"] += n
            checked["tracks"] += m
    return checked


def run_gpu(args) -> None:
    import torch
    import torch.distributed as dist

    from realtime_video_analytics_32streams_b200 import (DetectorConfig, HotPathEngine, StreamConfig, TrackerConfig,
                                                         _native)

    rank = int(os.environ.get("RANK", 0))
    world = int(os.environ.get("WORLD_SIZE", 1))
    local = int(os.environ.get("LOCAL_RANK", 0))
    if world != args.gpus:
        raise SystemExit(f"--gpus {args.gpus} but WORLD_SIZE={world}: launch with torchrun --nproc-per-node {args.gpus}")
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    numa_cores = None
    if world > 1 and not args.no_bind:
        from realtime_video_analytics_32streams_b200.runtime import bind_process_to_gpu

        numa_cores = bind_process_to_gpu(local)  # before any pinned allocation: first touch on the GPU's NUMA node
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def gather(values):
        """[world][len(values)] float64: every rank's list, on every rank."""
        mine = torch.tensor(list(values), dtype=torch.float64, device=dev)
        if world == 1:
            return [mine.cpu().tolist()]
        out = [torch.empty_like(mine) for _ in range(world)]
        dist.all_gather(out, mine)
        return [o.cpu().tolist() for o in out]

    K = args.steps
    warm = max(args.warmup, 3)
    # max_tracks 4096: SURVEY.md's sizing note (a stream's table, counted before the prune, must fit)
    h = _native.Handle(device=local, max_batch=STREAMS, max_anchors=A, max_candidates=2048, max_dets=512,
                       max_streams=2 * STREAMS, max_tracks=4096)
    # ---- synthetic inputs, resident in HBM --------------------------------------------------
    g = torch.Generator(device=dev)
    g.manual_seed(1234 + rank)
    frame_sets = [torch.randint(0, 256, (STREAMS, H, W, 3), dtype=torch.uint8, device=dev, generator=g)
                  for _ in range(N_SETS)]
    heads_np = np.stack([make_heads(rank * STREAMS + s, N_SETS) for s in range(STREAMS)], axis=1)  # [sets, 32, C, A]
    head_sets = [torch.from_numpy(heads_np[k]).to(dev) for k in range(N_SETS)]
    metas = (_native.Letterbox * STREAMS)(*[_native.letterbox_meta(H, W, *IN_HW) for _ in range(STREAMS)])
    # the network-input tensor rotates with the input sets (4 x 157 MB): a step's writes never land on lines that
    # are still dirty in L2 from the step before
    nets = [torch.empty((STREAMS, 3, *IN_HW), dtype=torch.float32, device=dev) for _ in range(N_SETS)]
    dets = h.alloc_dets(STREAMS)
    tracks = h.alloc_tracks(STREAMS)
    slots = _native._int_array(list(range(STREAMS)))
    trk_cfg = (TRK["max_age"], TRK["min_hits"], TRK["max_iou_distance"])
    # argument arrays are built once per input set: the per-step host work is one foreign call
    batches = [_native.FrameBatch(list(fs.unbind(0))) for fs in frame_sets]

    def make_plans(fmt=_native.OUT_F32_RGB_NCHW, m=STREAMS, p_dets=dets, p_tracks=tracks, p_slots=slots, p_metas=metas):
        return [h.plan_tick(frames=batches[k] if m == STREAMS else _native.FrameBatch(list(frame_sets[k][:m].unbind(0))),
                            net_out=nets[k][:m], dst_hw=IN_HW, fmt=fmt, head=head_sets[k][:m], metas=p_metas,
                            conf_thr=CONF, iou_thr=IOU, filter_conf=CONF, dets=p_dets, slots=p_slots, tracker_cfg=trk_cfg,
                            tracks=p_tracks, schedule=args.schedule) for k in range(N_SETS)]

    # one prepared b200va_tick per input set: decode -> NMS -> tracker on the library's second stream, letterbox on the
    # caller's (schedule 6 = 3 for this sparse workload: launched beside the decode kernel, overlapping NMS + tracker)
    plans = make_plans()

    # ---- parity of the timed computation (before anything is timed) -------------------------
    parity = None
    if not args.no_parity:
        if rank == 0:
            parity = parity_check(torch, h, frame_sets, heads_np, plans, nets, tracks, dets)
        barrier()
    for s in range(STREAMS):
        h.tracker_reset(s)

    def step(k):
        h.tick(plans[k % N_SETS])

    def serial_step(k):
        h.preprocess(batches[k % N_SETS], IN_HW, _native.OUT_F32_RGB_NCHW, out=nets[k % N_SETS])
        h.postprocess(head_sets[k % N_SETS], metas, CONF, IOU, filter_conf=CONF, out=dets)
        h.tracker_update(slots, dets, *trk_cfg, out=tracks)

    for k in range(warm):
        step(k)
    barrier()
    h.poll_status()
    graphs, kernels_per_graph = None, 0
    if not args.no_graph:
        try:
            graphs, kernels_per_graph = _capture(torch, h, plans)
            for k in range(warm):
                graphs[k % N_SETS].replay()
        except Exception as exc:  # pragma: no cover - capture refused: every step is launched eagerly instead
            print(f"bench: CUDA graph capture failed ({type(exc).__name__}: {exc}); running eagerly", file=sys.stderr)
            graphs, kernels_per_graph = None, 0
            torch.cuda.synchronize()
        barrier()

    def run_step(k):
        if graphs is None:
            step(k)
        else:
            graphs[k % N_SETS].replay()

    def windows(fn, n_windows, frames_per_step=STREAMS):
        """`n_windows` timed windows of EXACTLY K steps each, every one bracketed by barrier + synchronize on both
        sides and timed with CUDA events on the launching stream.  Per window the job time is the max over ranks;
        returns (median window ms, stats).  The headline calls it with one window, so its timed region is exactly K
        steps; the informational variants after it take the median of several windows."""
        for k in range(warm):
            fn(k)
        per = []
        for w in range(n_windows):
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            barrier()
            e0.record()
            for k in range(K):
                fn(w * K + k)
            e1.record()
            barrier()
            per.append(e0.elapsed_time(e1))
        allr = np.array(gather(per))          # [world, windows]
        job = allr.max(axis=0)                # max over ranks, per window
        med = float(np.median(job))
        stats = {"windows": n_windows, "steps_per_window": K,
                 "job_ms_per_step": {"min": round(float(job.min()) / K, 5), "median": round(med / K, 5),
                                     "max": round(float(job.max()) / K, 5)},
                 "per_rank_ms_per_step": [{"rank": r, "min": round(float(allr[r].min()) / K, 5),
                                           "median": round(float(np.median(allr[r])) / K, 5),
                                           "max": round(float(allr[r].max()) / K, 5)} for r in range(world)]}
        return med, stats

    # ---- the timed region --------------------------------------------------------------------
    clocks = ClockSampler(local, period_s=0.010)
    launches0 = h.launch_count
    clocks.start()
    ms, win_stats = windows(run_step, 1)
    clocks.stop()
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, nets[(K - 1) % N_SETS], dets, tracks)
    launches_per_step = kernels_per_graph if graphs is not None else (h.launch_count - launches0) / (K + warm)
    value = world * STREAMS * K / (ms * 1e-3)
    n_tracks = int(tracks["count"].sum().item())
    h.poll_status()
    # clocks under the same load, sampled densely in a window of their own (the thread above polls every 10 ms so
    # that it does not compete with the launching thread inside the short timed windows)
    load_clocks = ClockSampler(local, period_s=0.002)
    barrier()
    load_clocks.start()
    t_end = time.perf_counter() + 0.25
    k = 0
    while time.perf_counter() < t_end:
        run_step(k)
        k += 1
        if k % 64 == 0:
            torch.cuda.synchronize()
    torch.cuda.synchronize()
    load_clocks.stop()
    barrier()

    # ---- live per-kernel device times: eager ticks, one CUDA-event pair per phase on the launching stream -----
    # (a 512 MB fill runs ahead of every sampled tick: the host has enqueued the whole tick before the GPU reaches it, so
    # an event pair never contains a host launch gap, and the fill also evicts the tick's inputs from L2)
    h.set_profiling(True)
    samples = {}
    filler = torch.empty(512 << 20, dtype=torch.uint8, device=dev)
    for k in range(KERNEL_SAMPLES + 4):
        filler.fill_(k & 1)
        step(k)
        pt = h.phase_times()
        if k >= 4:
            for name, v in pt.items():
                samples.setdefault(name, []).append(v)
    h.set_profiling(False)
    # an event pair around ONE launch also holds the front end's event / launch latencies (an empty kernel between two
    # events reads ~6 us on this GPU, tools/membw.cu), which is a fifth of a 36 us kernel.  The letterbox's average
    # launch duration is therefore ALSO taken over 24 back-to-back launches (rotating inputs and outputs) inside one
    # event pair -- kernel + inter-launch gap, event latencies amortised -- and that figure feeds `roofline`.
    def back_to_back(fn, n=24, reps=5):
        out = []
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        for r in range(reps):
            filler.fill_(r & 1)
            e0.record()
            for k in range(n):
                fn(k)
            e1.record()
            torch.cuda.synchronize()
            out.append(e0.elapsed_time(e1) / n)
        return float(np.median(out))

    lb_b2b_ms = back_to_back(lambda k: h.preprocess(batches[k % N_SETS], IN_HW, _native.OUT_F32_RGB_NCHW, out=nets[k % N_SETS]))
    post_b2b_ms = back_to_back(lambda k: h.postprocess(head_sets[k % N_SETS], metas, CONF, IOU, filter_conf=CONF, out=dets))
    # the decode kernel has no entry point of its own: with a confidence threshold no score can reach, b200va_postprocess
    # is the full decode pass over the 32 heads (every row is read and scored, nothing is emitted) plus an NMS launch
    # that finds no candidates and returns at once
    dec_b2b_ms = back_to_back(lambda k: h.postprocess(head_sets[k % N_SETS], metas, 2.0, IOU, out=dets))
    pair = []
    for r in range(9):
        filler.fill_(r & 1)
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        h.tracker_reset(2 * STREAMS - 1)  # a one-thread kernel
        e1.record()
        torch.cuda.synchronize()
        pair.append(e0.elapsed_time(e1))
    pair_overhead_ms = float(np.median(pair))
    del filler
    kern_ms = {name: float(np.median(v)) for name, v in samples.items()}
    h.poll_status()
    barrier()

    # ---- informational variants (5 windows each) --------------------------------------------
    eager_ms, _ = windows(step, 5)
    serial_ms, _ = windows(serial_step, 5)
    # the same tick with B200VA_OUT_FLAG_PADS_VALID -- the 280 pad rows of every 640 x 640 input (44 % of the letterbox
    # output) were written by the earlier steps into the same persistent buffers and are not written again.  Not the
    # headline: `value` rewrites the whole tensor every step, like the reference does.
    pads_ms = None
    if graphs is not None:
        p_graphs, _ = _capture(torch, h, make_plans(fmt=_native.OUT_F32_RGB_NCHW | _native.OUT_FLAG_PADS_VALID))
        pads_ms, _ = windows(lambda k: p_graphs[k % N_SETS].replay(), 5)
        h.poll_status()
    # BASELINE.json's deployment shape: 32 streams IN TOTAL, 32 / N per GPU (strong scaling); at N = 1 this is the
    # headline itself.  One tick of 32 / N streams per GPU, same kernels, same graph replay.
    strong = None
    if STREAMS % world == 0:
        m = STREAMS // world
        if world == 1:
            strong = {"streams_total": STREAMS, "streams_per_gpu": m, "value": round(value, 1), "unit": "frames/s",
                      "ms_per_tick": round(ms / K, 5)}
        elif graphs is not None:
            s_dets, s_tracks = h.alloc_dets(m), h.alloc_tracks(m)
            s_slots = _native._int_array([STREAMS + i for i in range(m)])
            s_metas = (_native.Letterbox * m)(*[metas[i] for i in range(m)])
            s_graphs, _ = _capture(torch, h, make_plans(m=m, p_dets=s_dets, p_tracks=s_tracks, p_slots=s_slots,
                                                        p_metas=s_metas))
            s_ms, s_stats = windows(lambda k: s_graphs[k % N_SETS].replay(), WINDOWS)
            strong = {"streams_total": STREAMS, "streams_per_gpu": m, "value": round(STREAMS * K / (s_ms * 1e-3), 1),
                      "unit": "frames/s", "ms_per_tick": round(s_ms / K, 5),
                      "per_rank_ms_per_tick": s_stats["per_rank_ms_per_step"]}
            h.poll_status()

    # ---- end to end through the public API with host buffers ---------------------------------
    streams = [StreamConfig(name=f"r{rank}s{s}") for s in range(STREAMS)]
    host_frames = [torch.empty((H, W, 3), dtype=torch.uint8).pin_memory() for _ in range(STREAMS)]
    for s, hf in enumerate(host_frames):
        hf.copy_(frame_sets[0][s])
    host_heads = [torch.from_numpy(heads_np[k]).pin_memory() for k in range(N_SETS)]
    tick_no = [0]
    heads_from_host = [True]

    def infer(tensor):  # the detector forward is out of scope: its output arrives from pinned host memory
        k = tick_no[0] % N_SETS
        return host_heads[k].to(dev, non_blocking=True) if heads_from_host[0] else head_sets[k]

    eng = HotPathEngine(streams, DetectorConfig(confidence_threshold=CONF, iou_threshold=IOU),
                        TrackerConfig(**TRK), infer=infer, handle=h, input_hw=IN_HW, depth=2)
    e2e_steps = max(3, min(K, 100))

    def e2e_run(objects: bool):
        """`e2e_steps` ticks, tick k+1 submitted before tick k is collected (uploads overlap the
        host-side handling of results).  Every tick's H2D and D2H copies are inside the timed region."""
        eng.reset_tracks()
        checksum = 0
        for k in range(3):
            tick_no[0] = k
            eng.tick(host_frames)
        barrier()
        moved0 = eng.stager.bytes_moved
        t0 = time.perf_counter()
        prev = None
        for k in range(e2e_steps):
            tick_no[0] = 3 + k
            cur = eng.submit(host_frames)
            if prev is not None:
                for r in eng.collect(prev):
                    checksum += (len(r.tracks) + len(r.detections)) if objects else (r.n_tracks + r.n_detections)
            prev = cur
        for r in eng.collect(prev):
            checksum += (len(r.tracks) + len(r.detections)) if objects else (r.n_tracks + r.n_detections)
        torch.cuda.synchronize()
        dt = time.perf_counter() - t0
        dt = float(np.max(gather([dt])))
        assert checksum > 0
        return world * STREAMS * e2e_steps / dt, dt, (eng.stager.bytes_moved - moved0) // e2e_steps

    e2e_value, e2e_s, frame_bytes_per_step = e2e_run(objects=False)
    e2e_objects, _, _ = e2e_run(objects=True)
    heads_from_host[0] = False
    e2e_dev_heads, _, _ = e2e_run(objects=False)
    ctx0 = eng._ctxs[0]
    d2h = int(ctx0.host_dets_t["_flat"].numel() * ctx0.host_dets_t["_flat"].element_size()
              + ctx0.host_tracks_t["_flat"].numel() * ctx0.host_tracks_t["_flat"].element_size())
    h.poll_status()
    h.close()

    # ---- the other BASELINE.json configurations, driver-run (N = 1 only; a few steps each) ---------------
    configs_block = None
    used_graphs = graphs is not None
    if world == 1 and not args.no_configs:
        try:
            sys.path.insert(0, os.path.join(ROOT, "tools"))
            import bench_configs

            del frame_sets, head_sets, nets, batches, plans, graphs
            torch.cuda.empty_cache()
            configs_block = bench_configs.run_all(("1", "2", "5", "4", "D", "E", "P"), steps=max(10, min(K, 30)))
        except Exception as exc:  # pragma: no cover - informational block: never lose the headline line over it
            configs_block = {"error": f"{type(exc).__name__}: {exc}"}

    if rank == 0:
        peaks_path = os.path.join(ROOT, "MEASURED_PEAKS.json")
        if os.path.exists(peaks_path):
            with open(peaks_path) as fh:
                peak, peak_src = float(json.load(fh)["hbm_gbs"]), "MEASURED_PEAKS.json hbm_gbs (measured copy, burst)"
        else:
            peak, peak_src = 6650.0, "fallback 6.65 TB/s (B200_PROFILING.md)"
        traffic = {}
        tpath = os.path.join(ROOT, "profiles", "roofline_traffic.json")
        if os.path.exists(tpath):
            with open(tpath) as fh:
                traffic = json.load(fh)

        def roof(kernel, bytes_per_launch, ms_launch, traffic_key, note=None):
            ach = bytes_per_launch / (ms_launch * 1e-3) / 1e9
            tr = traffic.get(traffic_key)
            r = {"bound": "hbm", "kernel": kernel, "achieved": round(ach, 1), "peak": peak, "unit": "GB/s",
                 "frac": round(ach / peak, 4), "traffic": tr,
                 "frac_dram": round(tr / (ms_launch * 1e-3) / 1e9 / peak, 4) if tr else None,
                 "kernel_ms": round(ms_launch, 5), "algorithmic_bytes_per_launch": int(bytes_per_launch),
                 "samples": KERNEL_SAMPLES}
            if note:
                r["note"] = note
            return r

        roofline = roof("k_letterbox<F32_RGB_NCHW> (32 x 1080p per launch)", LETTERBOX_BYTES_PER_FRAME * STREAMS, lb_b2b_ms,
                        "k_letterbox_dram_bytes_per_launch")
        roofline["peak_source"] = peak_src
        roofline["samples"] = 5 * 24
        roofline["kernel_ms_event_pair_in_tick"] = round(kern_ms["preprocess"], 5)
        roofline["frac_event_pair_in_tick"] = round(LETTERBOX_BYTES_PER_FRAME * STREAMS / (kern_ms["preprocess"] * 1e-3) / 1e9 / peak, 4)
        roofline["event_pair_around_one_thread_kernel_ms"] = round(pair_overhead_ms, 5)
        roofline["how"] = ("kernel_ms: average launch duration over 24 back-to-back b200va_preprocess launches (4 rotating input "
                           "sets and outputs, 512 MB fill ahead so the host is never the limit) inside ONE CUDA-event pair on the "
                           "launching stream, median of 5 such runs; kernel_ms_event_pair_in_tick: median of %d eager ticks with "
                           "an event pair around the single letterbox launch (b200va_set_profiling) -- that pair also holds the "
                           "front end's event and launch latencies, see event_pair_around_one_thread_kernel_ms; `traffic` = "
                           "dram__bytes_read + dram__bytes_write of one launch from the ncu --set full capture summarised in "
                           "profiles/ (static, not re-measured in this run); frac_dram = traffic / kernel_ms / peak" % KERNEL_SAMPLES)
        roofline_kernels = [roofline]
        dec = roof("k_decode_cm<4> (32 heads [84, 8400] per launch, read-only)", HEAD_BYTES_PER_FRAME * STREAMS, dec_b2b_ms,
                   "k_decode_dram_bytes_per_launch",
                   "kernel_ms: 24 back-to-back b200va_postprocess calls with an unreachable confidence threshold (the full decode "
                   "pass + an NMS launch that returns at once) in one event pair.  A 90 MB read-only kernel is launch / ramp "
                   "bound on this GPU: tools/membw.cu times a pure 90 MB read at 18.4 us between events (4.9 TB/s) against "
                   "6.9 TB/s for 1 GB; profiles/r2_membw.log")
        dec["samples"] = 5 * 24
        if "decode" in kern_ms:
            dec["kernel_ms_event_pair_in_tick"] = round(kern_ms["decode"], 5)
        roofline_kernels.append(dec)
        for c in configs_block if isinstance(configs_block, list) else []:
            if str(c.get("config", "")).startswith("4:"):
                roofline_kernels.append(roof("k_motion_tile + ROI (32 x 4K per launch)", c["motion_algorithmic_bytes"],
                                             c["motion(+roi)"], "k_motion_tile_dram_bytes_per_launch"))
                roofline_kernels.append(roof("k_letterbox<F32_RGB_NCHW, masked> (32 x 4K + ROI per launch)",
                                             c["preprocess_algorithmic_bytes"], c["preprocess(+roi)"],
                                             "k_letterbox_4k_masked_dram_bytes_per_launch"))
            if str(c.get("config", "")).startswith("8f-3"):
                roofline_kernels.append(roof("k_area_fast (INTER_AREA 32 x 4K -> 1080p per call)", c["algorithmic_bytes"],
                                             c["resize_area"], "k_area_fast_dram_bytes_per_launch"))
            if str(c.get("config", "")).startswith("a14"):
                roofline_kernels.append(roof("k_dfl_decode (32 raw heads [144, 8400] per launch)", c["algorithmic_bytes"],
                                             c["dfl_decode"], "k_dfl_decode_dram_bytes_per_launch"))
        tick_bytes = (LETTERBOX_BYTES_PER_FRAME + HEAD_BYTES_PER_FRAME) * STREAMS

        def fps(ms_window):
            return round(world * STREAMS * K / (ms_window * 1e-3), 1)

        sched = {0: "serial", 1: "letterbox after decode, overlapping NMS + tracker (b200va_tick)",
                 2: "letterbox overlapping decode + NMS + tracker (b200va_tick)",
                 3: "letterbox launched beside the decode kernel (programmatic dependent launch), NMS + tracker "
                    "on the second stream (b200va_tick)",
                 5: "letterbox launched as a programmatic dependent of the decode kernel and waiting for it to drain "
                    "(griddepcontrol.wait), NMS + tracker on the second stream (b200va_tick)",
                 4: "software-pipelined b200va_tick: decode + letterbox of step k beside NMS + tracker of step k-1",
                 6: "automatic (b200va_tick schedule 6): >= 24 sparse frames -> letterbox launched beside the decode kernel as "
                    "its programmatic dependent, NMS + tracker on the second stream; small batches and dense scenes -> "
                    "letterbox after decode"}
        line = {"metric": METRIC, "value": round(value, 1), "unit": "frames/s", "n_gpus": world, "steps": K,
                "warmup": warm, "ms_per_step": round(ms / K, 5), "higher_is_better": True,
                "scaling": "weak", "vs_baseline": None, "dtype": "u8/f32", "data": "synthetic",
                "config": workload_config(world),
                "timing": dict(win_stats, how="CUDA events around the K timed steps, barrier + synchronize on both sides, "
                                              "max over ranks"),
                "parity_checked": parity is not None, "parity": parity,
                "roofline": roofline, "roofline_kernels": roofline_kernels,
                "tick_hbm": {"algorithmic_bytes_per_tick": tick_bytes,
                             "floor_ms_at_peak": round(tick_bytes / peak / 1e6, 5),
                             "frac": round(tick_bytes / peak / 1e6 / (ms / K), 4)},
                "kernel_ms": dict({k_: round(v, 5) for k_, v in kern_ms.items()},
                                  preprocess_back_to_back=round(lb_b2b_ms, 5), postprocess_back_to_back=round(post_b2b_ms, 5),
                                  decode_back_to_back=round(dec_b2b_ms, 5),
                                  how="event pair per phase in eager ticks; *_back_to_back: 24 launches in one pair"),
                "e2e": {"value": round(e2e_value, 1), "unit": "frames/s",
                        "h2d_bytes_per_step": int(frame_bytes_per_step + STREAMS * C * A * 4), "d2h_bytes_per_step": d2h,
                        "h2d_frame_bytes_per_step": int(frame_bytes_per_step), "h2d_head_bytes_per_step": STREAMS * C * A * 4,
                        "steps": e2e_steps, "ms_per_step": round(1e3 * e2e_s / e2e_steps, 3),
                        "value_with_python_objects": round(e2e_objects, 1),
                        "value_heads_resident_on_device": round(e2e_dev_heads, 1),
                        "api": "HotPathEngine.submit/collect (= tick, two ticks in flight) with pinned host frames -> "
                               "FrameResult host arrays (counts, boxes, ids); only the frame rows the letterbox reads "
                               "are uploaded (1 in 3 at 1080p); in `value` the head tensors are ALSO copied from "
                               "pinned host memory every step (conservative: a GPU-resident detector would leave "
                               "them on the device, see value_heads_resident_on_device); value_with_python_objects "
                               "additionally builds every Detection / Track object"},
                "gpu_launches": int(round(launches_per_step * K)), "launches_per_step": launches_per_step,
                "schedule": sched[args.schedule],
                "launch": ("CUDA graph replay of the prepared b200va_tick (one graph per input set)"
                           if used_graphs else "eager b200va_tick every step"),
                "value_eager_tick": fps(eager_ms), "value_three_serial_calls": fps(serial_ms),
                "value_pad_rows_written_once": fps(pads_ms) if pads_ms is not None else None,
                "strong_scaling_32_streams_total": strong,
                "clocks": dict(load_clocks.summary(), during_timed_windows=clocks.summary(),
                               how="sm_mhz: median of 2 ms NVML polls while the same graph replay loop runs for 0.25 s right "
                                   "after the timed windows; during_timed_windows: 10 ms polls while the windows ran"),
                "tracks_alive": n_tracks,
                "cpu_affinity": (f"rank 0 pinned to {len(numa_cores)} NUMA-local cores" if numa_cores else "unchanged"),
                "configs": configs_block}
        if world == 1 and not args.no_cpu:
            line["cpu_baseline"] = cpu_single_core_sample()
        else:
            line["cpu_baseline"] = None
        print(json.dumps(line), flush=True)
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()


def main() -> None:
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=200)
    ap.add_argument("--warmup", type=int, default=20)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--schedule", type=int, default=6, choices=[0, 1, 2, 3, 4, 5, 6],
                    help="b200va_tick schedule: 0 serial, 1 letterbox after decode, 2 fully parallel, 3 / 5 letterbox as the "
                         "decode kernel's programmatic dependent, 4 software-pipelined, 6 automatic (default; see include/b200va.h)")
    ap.add_argument("--no-graph", action="store_true", help="launch every step eagerly instead of replaying CUDA graphs")
    ap.add_argument("--no-bind", action="store_true", help="N > 1: do not pin each rank to its GPU's NUMA-local cores")
    ap.add_argument("--no-cpu", action="store_true", help="skip the single-core CPU sample")
    ap.add_argument("--no-configs", action="store_true", help="skip the `configs` block (BASELINE.json configs 1, 2, 4, 5)")
    ap.add_argument("--no-parity", action="store_true", help="skip the oracle comparison of two ticks before the timed region")
    ap.add_argument("--dump-outputs", metavar="DIR", help="write the outputs of the last timed step as DIR/<name>.npy")
    args = ap.parse_args()
    if args.dump_outputs and args.impl == "reference":
        ap.error("--dump-outputs writes the outputs of the GPU path; it does not apply to --impl reference")
    if args.impl == "reference":
        run_reference(args)
    else:
        run_gpu(args)


if __name__ == "__main__":
    main()
