"""Every tracker path against the sequential float64 IoU tracker (``oracle.hotpath.IouTracker``, tracker.py:36-147).

The device tracker splits the reference's order-dependent loop over threads in many ways (tracker_body.cuh): three
entry kernels (k_tracker, k_post_track<false|true>, k_dense_resolve_track), a small / shared-memory / global-scratch
working table, a pair list or 64-row units in phase A, the kCand fall-back to the sequential scan, phase B for
conflicted detections, phase C for new-track numbering and last-writer boxes, a prune of several rounds and the
last-CTA id patch.  Each case runs the same per-frame detection lists through the oracle and through one entry point,
and every frame is compared bit for bit: per stream the count and the row order, per track id, class, hits and age,
and conf and the four box doubles as int64 patterns (NaN positions and signed zeros count).

Entry points: ``tracker_update`` with float32 rows and ``det_scale`` (ratios 0.5 and 0.3), with float64 rows, and
``B200IouTracker.update``; and ``tick`` with only the head half: the fused sparse kernel k_post_track<false>, the
Ultralytics tick (k_post_track<true>), k_sort_nms followed by k_tracker (B200VA_FUSE_POST_TRACK=0), and
k_dense_resolve_track (B200VA_DENSE_IMPL=2).  A tick case builds its heads from the intended detections (one anchor
per detection, objectness 1, class score = conf, exact centres and sizes, identity letterbox, NMS threshold 1.0,
distinct scores in the intended order) and first checks that the NumPy post-process returns exactly that list.  A
detection with x1 = x2 = NaN comes from a head anchor with a NaN centre x; it survives NMS only as the first box of its
class (a NaN IoU suppresses), so such cases run the tick with class-aware NMS and skip the Ultralytics entry.  The
k_post_track entries take frames of at most 256 detections (more would switch the handle to its dense kernels): the
creation frame of a large scene goes through k_tracker instead, and only there (run_case asserts it).
``tracker_paths.predict`` restates the kernel's path choices; the path-matrix cases assert the path they are built for.
"""
import os

import numpy as np
import pytest

import tracker_paths as P
from oracle import hotpath as O
from oracle import ultralytics_restate as U

pytestmark = pytest.mark.gpu

FRAME = 4096  # identity letterbox: frame and network input are FRAME x FRAME
NC = 4  # head classes (the scenes use 0-2; class 3 carries the NaN-centre detections)
CONF = 0.25
I32_MIN, I32_MAX = -2 ** 31, 2 ** 31 - 1
NAN, INF = float("nan"), float("inf")
KERNELS = ("k_tracker", "k_post_track<false>", "k_post_track<true>", "k_dense_resolve_track")
SEEN = set()  # tracker kernels observed by the profiler in this module
UPDATE_ENTRIES = ("f32-0.5", "f32-0.3", "f64", "update")
TICK_ENTRIES = ("post", "ultra", "sortnms", "dense")
ENTRY_ENV = {"sortnms": (("B200VA_FUSE_POST_TRACK", "0"),), "dense": (("B200VA_DENSE_IMPL", "2"),)}
_HANDLES = {}


@pytest.fixture(scope="module", autouse=True)
def _handles():
    yield
    for h in _HANDLES.values():
        h.close()
    _HANDLES.clear()


def handle(env=()):
    """A handle created with the B200VA_* knobs `env` set (they are read when the handle is created)."""
    key = tuple(sorted(env))
    if key not in _HANDLES:
        from realtime_video_analytics_32streams_b200 import _native as N

        old = {k: os.environ.get(k) for k, _ in key}
        os.environ.update(dict(key))
        try:
            _HANDLES[key] = N.Handle(device=0, max_batch=128, max_anchors=4096, max_candidates=4096, max_dets=4096,
                                     max_streams=128, max_tracks=4096)
        finally:
            for k, v in old.items():
                if v is None:
                    del os.environ[k]
                else:
                    os.environ[k] = v
    return _HANDLES[key]


def cu(a):
    import torch

    return torch.from_numpy(np.ascontiguousarray(a)).cuda()


def kernel_of(name):
    if "k_dense_resolve_track" in name:
        return "k_dense_resolve_track"
    if "k_post_track" in name:
        return "k_post_track<true>" if ("<true>" in name or "ILb1E" in name) else "k_post_track<false>"
    if "k_tracker(" in name or "k_trackerE" in name:
        return "k_tracker"
    return None


def profiled(fn, expect=None):
    """Run fn under torch.profiler; record which tracker kernels it launched, and assert that `expect` is among them.
    Every tracker step launches a tracker kernel, so a trace without any (in a long pytest process the profiler now
    and then delivers an empty trace) says nothing about the step and is not held against it; the last test of the
    module asserts that every entry kernel was seen."""
    import torch
    from torch.profiler import ProfilerActivity, profile

    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        out = fn()
        torch.cuda.synchronize()
    ran = {kernel_of(e.name) for e in prof.events()} - {None}
    SEEN.update(ran)
    if expect is not None and ran:
        assert expect in ran, (expect, sorted(ran))
    return out


# ---- cases -------------------------------------------------------------------------------------------------------

class Case:
    """frames[t][s]: the detections (cls, conf, (x1, y1, x2, y2)) of stream s at frame t, or None when the stream
    skips the frame (``tracker.update(stream, [])``).  cfg: (max_age, min_hits, max_iou_distance), one for every
    frame or a list with one per frame."""

    def __init__(self, name, frames, cfg=(30, 0, 0.5), next_id=1, aware=False):
        self.name = name
        self.aware = aware  # tick with class-aware NMS
        self.frames = [f if (f and isinstance(f[0], (list, type(None)))) else [f] for f in frames]
        self.streams = len(self.frames[0])
        self.cfgs = cfg if isinstance(cfg, list) else [cfg] * len(self.frames)
        self.next_id = next_id

    def tickable(self, ultra=False):
        """Every box can be decoded exactly from a head (half-integer coordinates inside the frame, or x1 = x2 = NaN
        from a NaN centre when the tick uses class-aware NMS and the box leads its class alone), every class is a
        head class and every confidence is finite."""
        for fr in self.frames:
            for dets in fr:
                for c, f, b in dets or ():
                    if not (0 <= c < NC and np.isfinite(f)):
                        return False
                    if np.isnan(b[0]) and np.isnan(b[2]):
                        if ultra or not self.aware or sum(d[0] == c for d in dets) != 1:
                            return False
                        b = (0.0, b[1], 0.0, b[3])
                    if not all(np.isfinite(v) and v * 2 == int(v * 2) and 0 <= v <= FRAME - 1 for v in b):
                        return False
                    if b[2] < b[0] or b[3] < b[1]:
                        return False
        return True


def grid_box(k, w=12.0, h=12.0, dx=0.0, dy=0.0):
    """Box k of a lattice of 20-pixel cells: boxes of different cells never overlap."""
    x, y = 20.0 * (k % 200) + 4, 20.0 * (k // 200) + 4
    return (x + dx, y + dy, x + w + dx, y + h + dy)


def rank_conf(j):
    return (8192 - j) / 8192.0  # distinct, exact in float32, above CONF for j < 6144


# ---- running -----------------------------------------------------------------------------------------------------

def canon(a):
    a = np.array(a, dtype=np.float64).reshape(-1)
    a[np.isnan(a)] = np.nan
    return a.view(np.int64)


def check_stream(got, want, where):
    """got: (id, cls, conf, box, age, hits) arrays of one stream's rows; want: the oracle's Trk list."""
    ids, cls, conf, box, age, hits = got
    assert len(ids) == len(want), (where, len(ids), len(want))
    assert list(ids) == [w.track_id for w in want], where
    assert list(cls) == [w.class_id for w in want], where
    assert list(hits) == [w.hits for w in want], where
    assert list(age) == [w.age for w in want], where
    assert np.array_equal(canon(conf), canon([w.confidence for w in want])), where
    assert np.array_equal(canon(box), canon([w.bbox_xyxy for w in want])), where


def rows_of(host, b):
    n = int(host["count"][b])
    return (host["track_id"][b, :n].tolist(), host["cls"][b, :n].tolist(), host["conf"][b, :n],
            host["bbox_xyxy"][b, :n], host["age"][b, :n].tolist(), host["hits"][b, :n].tolist())


def soa_host(out):
    from realtime_video_analytics_32streams_b200 import B200IouTracker

    return B200IouTracker.soa_to_host(out)


def dets_f32(frame):
    return [[O.Det(int(c), float(np.float32(f)), tuple(float(np.float32(v)) for v in b)) for c, f, b in dets or ()]
            for dets in frame]


def dets_f64(frame):
    return [[O.Det(int(c), float(f), tuple(float(v) for v in b)) for c, f, b in dets or ()] for dets in frame]


def update_soa(dets, f64, md=None):
    B = len(dets)
    md = md or max(64, max(len(d) for d in dets))
    ft = np.float64 if f64 else np.float32
    box = np.zeros((B, md, 4), ft)
    conf = np.zeros((B, md), ft)
    cl = np.zeros((B, md), np.int32)
    cnt = np.zeros((B,), np.int32)
    for s, ds in enumerate(dets):
        cnt[s] = len(ds)
        for i, d in enumerate(ds):
            box[s, i], conf[s, i], cl[s, i] = d.bbox_xyxy, d.confidence, d.class_id
    return {"bbox_xyxy": cu(box), "conf": cu(conf), "cls": cu(cl), "count": cu(cnt)}


def tick_frame(h, frame, cfg, ultra, skip, tracks, aware=False):
    """One tick with only the head half; returns the detections the tracker was given (intended lists)."""
    from realtime_video_analytics_32streams_b200 import _native as N

    B = len(frame)
    A = max(64, max(len(d or ()) for d in frame))
    C = 4 + NC if ultra else 5 + NC
    head = np.zeros((B, C, A), np.float32)
    intended = []
    for s, dets in enumerate(frame):
        want = []
        for j, (c, _, b) in enumerate(dets or ()):
            f = rank_conf(j)
            head[s, 0, j], head[s, 1, j] = (b[0] + b[2]) / 2, (b[1] + b[3]) / 2
            head[s, 2, j], head[s, 3, j] = b[2] - b[0], b[3] - b[1]
            if np.isnan(b[0]):  # a NaN centre x decodes to x1 = x2 = NaN
                head[s, 2, j] = 10.0
            if ultra:
                head[s, 4 + c, j] = f
            else:
                head[s, 4, j] = 1.0
                head[s, 5 + c, j] = f
            want.append(O.Det(int(c), f, tuple(float(v) for v in b)))
        # the NumPy post-process must hand the tracker exactly this list
        if ultra:
            got = [O.Det(c, f, b) for c, f, b in U.postprocess(head[s], (FRAME, FRAME), (FRAME, FRAME), CONF, 1.0)]
        else:
            meta = {"orig_shape": (FRAME, FRAME), "scale": 1.0, "pad": (0, 0)}
            got = O.postprocess(head[s][None], meta, CONF, 1.0, class_aware=aware)
        got = O.filter_detections(got, CONF)
        assert [(d.class_id, d.confidence) for d in got] == [(d.class_id, d.confidence) for d in want], s
        assert np.array_equal(canon([d.bbox_xyxy for d in got]), canon([d.bbox_xyxy for d in want])), s
        intended.append(want if dets is not None else [])
    kw = {}
    if ultra:
        kw["ultralytics"] = dict(frame_hw=[(FRAME, FRAME)] * B, in_hw=(FRAME, FRAME))
    else:
        kw["metas"] = [N.Letterbox(FRAME, FRAME, FRAME, FRAME, 0, 0, 1.0)] * B
        if aware:
            kw["nms_mode"] = N.NMS_CLASS_AWARE
    plan = h.plan_tick(head=cu(head), conf_thr=CONF, iou_thr=1.0, filter_conf=CONF, slots=list(range(B)),
                       tracker_cfg=cfg, skip=skip, tracks=tracks, schedule=1, **kw)
    h.tick(plan)
    return intended


def run_case(case, entry, env=(), profile=False, expect=None):
    """Runs every frame of `case` through `entry` and compares each frame with the oracle."""
    from realtime_video_analytics_32streams_b200 import B200IouTracker, TrackerConfig

    h = handle(tuple(env) + ENTRY_ENV.get(entry, ()))
    B = case.streams
    names = [f"s{s}" for s in range(B)]
    ora = O.IouTracker()
    ora._ids = iter(range(case.next_id, case.next_id + 10 ** 7))
    trk = None
    if entry == "update":
        trk = B200IouTracker(TrackerConfig(), handle=h)
        for n in names:
            trk.slot_of(n)
    for s in range(B):
        h.tracker_reset(s)
    h.tracker_set_next_id(case.next_id)
    tracks = h.alloc_tracks(B)
    try:
        for t, frame in enumerate(case.frames):
            max_age, min_hits, thr = cfg = case.cfgs[t]
            ora.max_age, ora.min_hits, ora.max_iou_distance = cfg
            skip = [d is None for d in frame]
            where = (case.name, entry, t)

            def step():
                if entry == "update":
                    trk.config = TrackerConfig(max_age=max_age, min_hits=min_hits, max_iou_distance=thr)
                    given = dets_f64(frame)
                    return given, [trk.update(n, d) for n, d in zip(names, given)]
                if entry in TICK_ENTRIES:
                    if max(len(d or ()) for d in frame) <= 256 or entry in ("sortnms", "dense"):
                        given = tick_frame(h, frame, cfg, entry == "ultra", skip, tracks, case.aware)
                        return given, soa_host(tracks)
                    # k_post_track entries: only a scene's creation frame is too large for the sparse tick
                    assert t == 0, (where, "more than 256 detections in a checked frame of a k_post_track case")
                f64 = entry == "f64"
                given = dets_f64(frame) if f64 else dets_f32(frame)
                scale = None
                if entry.startswith("f32-"):
                    ratio = float(entry[4:])
                    scale = [1.0 / max(ratio, 1e-6)] * B
                    given = [O.rescale_detections(d, ratio) for d in given]
                raw = dets_f64(frame) if f64 else dets_f32(frame)
                out = h.tracker_update(list(range(B)), update_soa(raw, f64), max_age, min_hits, thr, det_scale=scale,
                                       skip=skip, out=tracks, f64=f64)
                return given, soa_host(out)

            given, got = profiled(step, expect) if (profile or expect) else step()
            for s in range(B):
                want = ora.update(names[s], given[s] if frame[s] is not None else [])
                if entry == "update":
                    g = got[s]
                    rows = ([x.track_id for x in g], [x.class_id for x in g], [x.confidence for x in g],
                            [x.bbox_xyxy for x in g], [x.age for x in g], [x.hits for x in g])
                else:
                    rows = rows_of(got, s)
                check_stream(rows, want, where + (s,))
        h.poll_status()
    finally:
        if trk is not None:
            trk.close()


def run_all(case, entries=UPDATE_ENTRIES + TICK_ENTRIES, env=()):
    for e in entries:
        if e in TICK_ENTRIES and not case.tickable(ultra=e == "ultra"):
            continue
        run_case(case, e, env)


# ---- path matrix -------------------------------------------------------------------------------------------------

def scene(t0, d, seed, thr=0.5, cls_mix=3, frames=3):
    """Frame 0 creates t0 tracks on the lattice; frame 1 has d detections: re-detections (shifted by half or one
    pixel), shifted duplicates of earlier detections (conflicts and detection-detection edges), re-detections in
    another class and new boxes; frame 2 re-detects every other track, so the rest age (and are pruned with
    max_age 0)."""
    rng = np.random.default_rng(seed)
    f0 = [(k % cls_mix, rank_conf(k), grid_box(k)) for k in range(t0)]
    f1 = []
    for j in range(d):
        r = int(rng.integers(0, 6))
        if r <= 1 and t0:
            k = int(rng.integers(0, t0))
            f1.append((k % cls_mix, 0.0, grid_box(k, dx=float(rng.choice([0.5, 1.0, -1.0])), dy=float(rng.choice([0.0, 0.5])))))
        elif r == 2 and f1:
            c, _, b = f1[int(rng.integers(0, len(f1)))]
            f1.append((c, 0.0, (b[0] + 0.5, b[1], b[2] + 0.5, b[3] + 0.5)))
        elif r == 3 and t0:
            k = int(rng.integers(0, t0))
            f1.append(((k + 1) % cls_mix, 0.0, grid_box(k, dx=0.5)))
        else:
            f1.append((j % cls_mix, 0.0, grid_box(t0 + j)))
    f1 = [(c, rank_conf(j), b) for j, (c, _, b) in enumerate(f1)]
    f2 = [(k % cls_mix, rank_conf(i), grid_box(k, dx=0.5)) for i, k in enumerate(range(0, t0, 2))][:256]
    return [f0, f1, f2][:frames]


MATRIX = [
    # (name, t0, d, env, entries, path check: (entry kind, smem_tracks, threads, fused, chunk (tc, nd) or None, want))
    ("small-staged", 40, 20, (), ("post", "f64"), (512, 256, True, None, P.Path("small-staged", "shared", "few", 256))),
    ("small-unstaged", 300, 6, (), ("post", "ultra", "f32-0.3"), (512, 256, True, None, P.Path("small", "shared", "few", 256))),
    ("few-pairs", 60, 20, (), ("f32-0.5", "f64", "sortnms"), (512, 512, False, None, P.Path("general", "shared", "few", 256))),
    ("units-G8-64", 200, 64, (), UPDATE_ENTRIES + TICK_ENTRIES, (512, 512, False, None, P.Path("general", "shared", "units-G8", 512))),
    ("units-G8-31", 300, 31, (), ("f32-0.3", "f64", "post"), (3072, 512, False, None, P.Path("general", "shared", "units-G8", 512))),
    ("units-G4-33", 500, 33, (), ("f32-0.5", "post", "dense"), (3072, 512, False, None, P.Path("general", "shared", "units-G4", 512))),
    ("units-G4-63", 800, 63, (), ("f64", "update", "ultra"), (3072, 512, False, None, P.Path("general", "shared", "units-G4", 512))),
    ("units-G2-129", 1000, 129, (), ("f32-0.3", "f64", "post", "dense"), (3072, 512, False, None, P.Path("general", "shared", "units-G2", 512))),
    ("units-G2-1-w256", 2100, 65, (("B200VA_TRK_THREADS", "256"),), ("f64", "post"),
     (3072, 256, False, (2100 + 8, 1), P.Path("general", "shared", "units-G2", 256))),
    ("global-natural", 3000, 100, (), ("f64", "dense"), (3072, 512, False, None, P.Path("general", "global", "units-G2", 512))),
    ("global-smem8", 300, 40, (("B200VA_TRK_SMEM_TRACKS", "8"),), ("f32-0.5", "post", "dense"),
     (8, 256, True, None, P.Path("general", "global", "units-G8", 256))),
    ("global-smem8-few", 60, 20, (("B200VA_TRK_SMEM_TRACKS", "8"),), ("f64", "sortnms"),
     (8, 512, False, None, P.Path("general", "global", "few", 256))),
]


@pytest.mark.parametrize("name,t0,d,env,entries,path", MATRIX, ids=[m[0] for m in MATRIX])
def test_path_matrix(name, t0, d, env, entries, path):
    smem, threads, fused, chunk, want = path
    tc, nd = chunk if chunk else (None, None)
    assert P.predict(t0, d, smem, threads, fused, tc, nd) == want, name
    for k, cfg in enumerate(((1, 0, 0.5), (0, 1, 0.3))):
        case = Case(name, scene(t0, d, seed=t0 * 1000 + d), cfg=cfg)
        for e in entries:
            run_case(case, e, env, profile=k == 0)


def test_pair_list_overflow_without_fallback():
    """One chunk of 64 wide staggered boxes against 100 staggered tracks: every pair overlaps (6400 + 2016 listed
    pairs > 2048, the rest is evaluated on the spot), but only neighbours pass the 0.99 threshold: each detection
    ties between two tracks (the earlier wins) and shares them with its neighbours (phase B)."""
    tracks = [(0, rank_conf(i), (8.0 * i, 0.0, 8.0 * i + 1000, 1000.0)) for i in range(100)]
    dets = [(0, rank_conf(j), (8.0 * j + 4, 0.0, 8.0 * j + 1004, 1000.0)) for j in range(64)]
    assert P.predict(100, 64, 512, 512).phase_a == "units-G8"
    assert 64 * 100 + 64 * 63 // 2 > P.TRK_PAIRS
    assert O.iou_f64(tracks[5][2], dets[5][2]) == O.iou_f64(tracks[6][2], dets[5][2]) >= 0.99
    assert O.iou_f64(dets[4][2], dets[5][2]) < 0.99
    run_all(Case("pairlist", [tracks, dets], cfg=(5, 0, 0.99)), ("f32-0.5", "f64", "update", "post", "sortnms", "dense"))


def strips():
    """Ten strips across a 100 x 100 box: IoU 0.2 with the box, at most 0.111 between any two of them."""
    h = [(0, 0.0, (1000.0, 1000.0 + 20 * k, 1100.0, 1020.0 + 20 * k)) for k in range(5)]
    v = [(0, 0.0, (1000.0 + 20 * k, 1000.0, 1020.0 + 20 * k, 1100.0)) for k in range(5)]
    return [(c, rank_conf(j), b) for j, (c, _, b) in enumerate(h + v)]


@pytest.mark.parametrize("pad", [0, 60, 200])
def test_kcand_fallback(pad):
    """More than kCand = 6 candidates: ten tracks under one detection, and ten earlier detections of the same chunk
    under one detection.  `pad` unrelated tracks (and up to 20 re-detections of them) move the fused kernel from its
    small instantiation to the general one (`kinds`), whose fall-back scan is inlined instead of called."""
    centre = (1000.0, 1000.0, 1100.0, 1100.0)
    s = strips()
    assert all(O.iou_f64(b, centre) >= 0.15 for _, _, b in s)
    assert max(O.iou_f64(a[2], b[2]) for a in s for b in s if a is not b) < 0.15
    filler = [(1, 0.5, grid_box(k)) for k in range(pad)]
    again = [(1, 0.5, grid_box(k, dx=0.5)) for k in range(min(pad, 20))]
    frames_trk = [s + filler, [(0, 0.9, centre)] + again]
    frames_det = [filler, s + [(0, 0.9, centre)] + again]
    # pad 0: small in both; 60: small with ten track candidates, general with ten detection candidates; 200: general
    kinds = {0: ("small-staged", "small-staged"), 60: ("small-staged", "general"), 200: ("general", "general")}[pad]
    assert P.predict(len(s) + pad, 1 + len(again), 512, 256, fused=True).kind == kinds[0]
    assert P.predict(pad, len(s) + 1 + len(again), 512, 256, fused=True).kind == kinds[1]
    for frames in (frames_trk, frames_det):
        run_all(Case(f"kcand-{pad}", frames, cfg=(3, 0, 0.15)))


def test_prune_several_rounds():
    """1300 tracks, most unmatched: the prune compacts the table in 512-row rounds (1024 on the dense kernel)."""
    f0 = [(k % 2, rank_conf(k), grid_box(k)) for k in range(1300)]
    f1 = [(k % 2, rank_conf(i), grid_box(k, dx=1.0)) for i, k in enumerate(range(0, 1300, 7))]
    f2 = [(k % 2, rank_conf(i), grid_box(k, dx=0.5)) for i, k in enumerate(range(0, 1300, 11))]
    for cfg in ((0, 0, 0.5), (1, 2, 0.5), (-1, 0, 0.5)):
        run_all(Case("prune", [f0, f1, f2, []], cfg=cfg), ("f32-0.5", "f64", "post", "dense"))


def test_graph_tick_grows_past_captured_rows():
    """A tick captured in a CUDA graph freezes the size of its shared-memory table (512 rows on a fresh handle);
    replays whose streams need more rows (live tracks + detections) work in the global scratch."""
    import torch
    from realtime_video_analytics_32streams_b200 import _native as N

    h = N.Handle(device=0, max_batch=2, max_anchors=256, max_candidates=4096, max_dets=4096, max_streams=2,
                 max_tracks=4096)
    try:
        B = 2
        head = torch.zeros((B, 5 + NC, 256), dtype=torch.float32, device="cuda")
        tracks = h.alloc_tracks(B)
        plan = h.plan_tick(head=head, metas=[N.Letterbox(FRAME, FRAME, FRAME, FRAME, 0, 0, 1.0)] * B, conf_thr=CONF,
                           iou_thr=1.0, filter_conf=CONF, slots=list(range(B)), tracker_cfg=(30, 0, 0.5),
                           tracks=tracks, schedule=1)
        side = torch.cuda.Stream()
        side.wait_stream(torch.cuda.current_stream())
        graph = torch.cuda.CUDAGraph()
        with torch.cuda.stream(side):
            with torch.cuda.graph(graph, stream=side):
                h.tick(plan)
        torch.cuda.current_stream().wait_stream(side)
        torch.cuda.synchronize()
        for s in range(B):
            h.tracker_reset(s)
        h.tracker_set_next_id(1)
        ora = O.IouTracker(30, 0.5, 0)
        needs = []
        for t in range(5):  # 235 new boxes per frame and stream, 15 re-detections of the previous frame's boxes
            hn = np.zeros((B, 5 + NC, 256), np.float32)
            frame = []
            for s in range(B):
                rows = [(s, grid_box(1200 * s + 240 * t + j)) for j in range(235)]
                rows += [(s, grid_box(1200 * s + 240 * (t - 1) + j, dx=1.0)) for j in range(0, 240, 16) if t]
                want = []
                for j, (c, b) in enumerate(rows):
                    hn[s, :4, j] = ((b[0] + b[2]) / 2, (b[1] + b[3]) / 2, b[2] - b[0], b[3] - b[1])
                    hn[s, 4, j], hn[s, 5 + c, j] = 1.0, rank_conf(j)
                    want.append(O.Det(c, rank_conf(j), b))
                frame.append(want)
            needs.append(len(ora._tracks.get("s0", [])) + len(frame[0]))
            head.copy_(torch.from_numpy(hn))
            graph.replay()
            torch.cuda.synchronize()
            host = soa_host(tracks)
            for s in range(B):
                check_stream(rows_of(host, s), ora.update(f"s{s}", frame[s]), ("graph", t, s))
        assert needs[0] <= 512 < needs[-1], needs  # the last replays needed more rows than were captured
        assert P.predict(needs[-1] - 250, 250, 512, 256, fused=True).table == "global"
        h.poll_status()
    finally:
        h.close()


# ---- value and semantics families ---------------------------------------------------------------------------------

def test_threshold_exact_and_one_ulp_either_side():
    track, det = (10.0, 10.0, 30.0, 30.0), (12.0, 11.0, 31.0, 29.5)
    v = O.iou_f64(track, det)
    for thr, match in ((v, True), (float(np.nextafter(v, -1.0)), True), (float(np.nextafter(v, 2.0)), False)):
        case = Case("thr-ulp", [[(0, 0.9, track)], [(0, 0.8, det)]], cfg=(30, 0, thr))
        want = O.IouTracker(30, thr, 0)
        want.update("s", [O.Det(0, 0.9, track)])
        assert (len(want.update("s", [O.Det(0, 0.8, det)])) == 1) == match
        run_all(case, ("f32-0.5", "f64", "update", "post", "dense"))


@pytest.mark.parametrize("thr", [0.0, -0.5, 1.0, 1.5, NAN])
def test_thresholds(thr):
    f0 = [(0, 0.9, (0.0, 0.0, 10.0, 10.0)), (0, 0.8, (20.0, 0.0, 30.0, 10.0)), (1, 0.7, (40.0, 0.0, 50.0, 10.0))]
    f1 = [(0, 0.9, (0.0, 0.0, 10.0, 10.0)),     # IoU 1
          (0, 0.8, (30.0, 0.0, 40.0, 10.0)),    # touches track 2: IoU 0
          (1, 0.7, (45.0, 0.0, 55.0, 10.0)),    # IoU 1/3
          (0, 0.6, (25.0, 0.0, 30.0, 10.0))]    # inside track 2: IoU 0.5
    run_all(Case(f"thr-{thr}", [f0, f1, f1], cfg=(30, 0, thr)))


def _mirror(gap, swap):
    a, b = (90.0, 100.0, 190.0, 200.0), (110.0, 100.0, 210.0, 200.0)
    first, last = (b, a) if swap else (a, b)
    f0 = [(0, 0.9, first)] + [(0, 0.5, grid_box(400 + k)) for k in range(gap - 1)] + [(0, 0.8, last)]
    return [f0, [(0, 0.7, (100.0, 100.0, 200.0, 200.0))]]


@pytest.mark.parametrize("gap", [1, 31, 32, 64])
def test_tie_mirror_earliest_track_wins(gap):
    for swap in (False, True):
        run_all(Case(f"tie-{gap}-{swap}", _mirror(gap, swap), cfg=(30, 0, 0.75)))


def test_tie_with_track_created_in_the_same_chunk():
    f0 = [(0, 0.9, (90.0, 100.0, 190.0, 200.0))]
    f1 = [(0, 0.8, (110.0, 100.0, 210.0, 200.0)), (0, 0.7, (100.0, 100.0, 200.0, 200.0))]
    for pad in (0, 62):  # the pair at the end of a full chunk
        fill = [(1, 0.5, grid_box(300 + k)) for k in range(pad)]
        run_all(Case(f"tie-new-{pad}", [f0, fill + f1], cfg=(30, 0, 0.75)))


def test_tie_through_phase_b_detection_edge():
    u, t = (90.0, 100.0, 190.0, 200.0), (112.0, 100.0, 212.0, 200.0)
    e, i = (110.0, 100.0, 210.0, 200.0), (100.0, 100.0, 200.0, 200.0)
    assert O.iou_f64(u, i) == O.iou_f64(e, i) and O.iou_f64(t, i) >= 0.75 > O.iou_f64(u, e)
    for order in ((u, t), (t, u)):
        f0 = [(0, 0.9, order[0]), (0, 0.8, order[1])]
        run_all(Case("tie-phaseB", [f0, [(0, 0.7, e), (0, 0.6, i)]], cfg=(30, 0, 0.75)))


@pytest.mark.parametrize("pad", [0, 63])
def test_phase_b_chains(pad):
    """e takes t, and a later i must see e's box on t; e simple / conflicted; a track re-boxed twice (last writer);
    i's match to t's chunk-start box is gone after e moved it.  `pad`: e at index 63, i in the next chunk."""
    p = (100.0, 100.0, 200.0, 200.0)
    chains = [[(110.0, 100.0, 210.0, 200.0), (120.0, 100.0, 220.0, 200.0)],   # e simple, i matches through e
              [(104.0, 100.0, 204.0, 200.0), (112.0, 100.0, 212.0, 200.0)],   # e conflicted (i claims t too)
              [(110.0, 100.0, 210.0, 200.0), (95.0, 100.0, 195.0, 200.0)],    # after e, i no longer matches t
              [(102.0, 100.0, 202.0, 200.0), (104.0, 100.0, 204.0, 200.0), (106.0, 100.0, 206.0, 200.0)]]
    fill = [(1, 0.5, grid_box(300 + k)) for k in range(pad)]
    for k, chain in enumerate(chains):
        f1 = fill + [(0, rank_conf(j), b) for j, b in enumerate(chain)]
        run_all(Case(f"chain-{k}-{pad}", [[(0, 0.9, p)], f1, f1[pad:]], cfg=(30, 0, 0.75)))


def test_signed_zero_negative_inverted_zero_area():
    f0 = [(0, 0.9, (0.0, -0.0, 10.0, 10.0)), (0, 0.8, (-50.0, -40.0, -10.0, -5.0)), (0, 0.7, (30.0, 30.0, 10.0, 10.0)),
          (0, 0.6, (5.0, 5.0, 5.0, 10.0)), (1, 0.5, (-0.0, -0.0, -0.0, -0.0))]
    f1 = [(0, 0.9, (-0.0, 0.0, 10.0, 10.0)), (0, 0.8, (-49.0, -40.0, -10.0, -5.0)), (0, 0.7, (30.0, 30.0, 10.0, 10.0)),
          (0, 0.6, (10.0, 10.0, 30.0, 30.0)), (0, 0.5, (5.0, 5.0, 5.0, 10.0)), (1, 0.4, (0.0, 0.0, 0.0, 0.0))]
    run_all(Case("zeros", [f0, f1, f1], cfg=(30, 0, 0.3)))


def test_subnormal_and_low_word_coordinates():
    sub = 1e-310
    f0 = [(0, 0.9, (0.0, 0.0, sub, 1.0)), (0, 0.8, (0.0, 10.0, 1e-40, 11.0)), (0, 0.7, (0.0, 20.0, 100.0, 120.0))]
    x = 100.0 + 1e-9  # differs from 100.0 in the low word only: the overlap keys are equal
    assert np.float64(x).view(np.int64) >> 32 == np.float64(100.0).view(np.int64) >> 32
    det = (0.0, 20.0, x, 120.0)
    v = O.iou_f64(f0[2][2], det)
    assert 0 < 1 - v < 1e-9
    f1 = [(0, 0.9, (0.0, 0.0, sub, 1.0)), (0, 0.8, (0.0, 10.0, 1e-40, 11.0)), (0, 0.7, det)]
    for thr in (v, float(np.nextafter(v, 2.0))):
        run_all(Case("subnormal-lowword", [f0, f1], cfg=(30, 0, thr)), UPDATE_ENTRIES)


def test_huge_and_infinite_coordinates():
    big = 1e300
    f0 = [(0, 0.9, (0.0, 0.0, big, big)), (0, 0.8, (-INF, 0.0, INF, 10.0)), (1, 0.7, (0.0, 0.0, 10.0, INF)),
          (2, 0.6, (-big, -big, 0.0, 0.0))]
    f1 = [(0, 0.9, (0.0, 0.0, big, big)), (0, 0.8, (0.0, 0.0, big, 1.0)), (0, 0.7, (-INF, 0.0, INF, 10.0)),
          (0, 0.6, (0.0, 0.0, 10.0, 10.0)), (1, 0.5, (0.0, 0.0, 10.0, INF)), (2, 0.4, (-big, -big, 0.0, 0.0))]
    for thr in (0.5, 0.0):
        run_all(Case("huge", [f0, f1, f1], cfg=(30, 0, thr)), UPDATE_ENTRIES)


NAN_DETS = [(NAN, 0.0, 8.0, 10.0), (0.0, NAN, 10.0, 8.0), (2.0, 0.0, NAN, 10.0), (0.0, 2.0, 10.0, NAN),
            (NAN, 0.0, NAN, 5.0), (NAN, NAN, NAN, NAN), (NAN, 0.0, 10.0, 10.0)]


def test_oracle_matches_nan_detections_through_builtin_min_max():
    ref = O.IouTracker(30, 0.5, 0)
    ref.update("s", [O.Det(0, 0.9, (0.0, 0.0, 10.0, 10.0))])
    tr = ref.update("s", [O.Det(0, 0.8, (NAN, 0.0, NAN, 5.0))])
    assert len(tr) == 1 and tr[0].hits == 2


@pytest.mark.parametrize("thr", [0.5, 1.5])
def test_nan_detection_coordinates(thr):
    """Python's min / max keep the track's coordinate where the detection's is NaN: such a detection can match (with
    IoU above 1 even).  One stream per NaN pattern, each with a track (0, 0, 10, 10) to match; frame 2 offers the
    track's box again: the tracks that took a NaN box cannot match it any more (NaN on the track side)."""
    track = (0.0, 0.0, 10.0, 10.0)
    f0 = [[(0, 0.9, track)] for _ in NAN_DETS]
    f1 = [[(0, 0.8, b)] for b in NAN_DETS]
    f2 = [[(0, 0.7, track)] for _ in NAN_DETS]
    run_all(Case(f"nan-{thr}", [f0, f1, f2, f2], cfg=(30, 0, thr)), UPDATE_ENTRIES)


def test_nan_track_box_and_nan_confidence():
    f0 = [(0, NAN, (0.0, 0.0, 10.0, 10.0)), (0, 0.9, (NAN, 20.0, 30.0, 30.0))]
    f1 = [(0, 0.5, (0.0, 0.0, 10.0, 10.0)), (0, NAN, (20.0, 20.0, 30.0, 30.0)), (0, NAN, (0.0, 0.0, 10.0, 10.0))]
    run_all(Case("nan-conf", [f0, f1, f1], cfg=(30, 0, 0.3)), UPDATE_ENTRIES)


def test_nan_detection_on_the_units_path():
    """A NaN-centre re-detection (x1 = x2 = NaN, y inside the track's) among 64 detections against 201 tracks: phase A
    takes the 64-row units (det_keys, the unit's key test, overlaps()), on k_tracker and on the general instantiation
    of k_post_track; the NaN box matches its track (IoU 1) as tracker.py's min / max have it."""
    f0, f1, f2 = scene(200, 64, seed=77)
    track = grid_box(900)
    nan_det = (NAN, track[1] + 3.0, NAN, track[3] - 3.0)
    assert O.iou_f64(track, nan_det) == 1.0
    f0 = f0 + [(3, rank_conf(len(f0)), track)]
    for i in (40, 63):
        g1 = list(f1)
        g1[i] = (3, g1[i][1], nan_det)
        frames = [f0, g1, f2 + [(3, rank_conf(len(f2)), track)]]
        assert P.predict(201, 64, 512, 512).phase_a == "units-G8"
        assert P.predict(201, 64, 512, 256, fused=True) == P.Path("general", "shared", "units-G8", 256)
        case = Case(f"nan-units-{i}", frames, cfg=(3, 0, 0.5), aware=True)
        assert case.tickable() and not case.tickable(ultra=True)
        for e in ("f32-0.5", "f64", "update", "sortnms"):
            run_case(case, e)
        run_case(case, "post", expect="k_post_track<false>")
        run_case(case, "dense", expect="k_dense_resolve_track")


@pytest.mark.parametrize("pad", [0, 200])
def test_nan_detection_in_the_kcand_fallback(pad):
    """A NaN-centre detection over the ten strips (y inside them) has IoU 4 with the five vertical strips and 1 with
    two horizontal ones: seven candidates, so the chunk takes the sequential scan (overlaps() + iou64), in the small
    (pad 0) and the general (pad 200) instantiation; the five-way tie goes to the earliest vertical strip.  As ten
    earlier detections of the chunk (k_tracker entries only: a NaN box behind boxes of its class does not survive
    NMS)."""
    s = strips()
    nan_det = (NAN, 1010.0, NAN, 1090.0)
    assert sorted(O.iou_f64(b, nan_det) for _, _, b in s) == [0.0] * 3 + [1.0] * 2 + [4.0] * 5
    filler = [(1, 0.5, grid_box(k)) for k in range(pad)]
    again = [(1, 0.5, grid_box(k, dx=0.5)) for k in range(min(pad, 20))]
    kind = "small-staged" if pad == 0 else "general"
    assert P.predict(len(s) + pad, 1 + len(again), 512, 256, fused=True).kind == kind
    case = Case(f"nan-kcand-trk-{pad}", [s + filler, [(0, 0.9, nan_det)] + again, s[:1]], cfg=(3, 0, 0.15), aware=True)
    assert case.tickable()
    for e in ("f32-0.3", "f64", "update", "sortnms", "dense"):
        run_case(case, e)
    run_case(case, "post", expect="k_post_track<false>")
    case = Case(f"nan-kcand-det-{pad}", [filler, s + [(0, 0.9, nan_det)] + again], cfg=(3, 0, 0.15), aware=True)
    assert not case.tickable()
    run_all(case, UPDATE_ENTRIES)


def test_extreme_classes():
    box = (0.0, 0.0, 10.0, 10.0)
    f0 = [(c, 0.9, box) for c in (I32_MIN, -1, 0, I32_MAX)]
    f1 = [(c, 0.8, (0.0, 0.0, 10.0, 11.0)) for c in (I32_MAX, 0, -1, I32_MIN, 7)]
    run_all(Case("classes", [f0, f1, f1], cfg=(30, 0, 0.5)), UPDATE_ENTRIES)


@pytest.mark.parametrize("max_age,min_hits", [(-1, 0), (0, 1), (1000, 0), (2, 50), (3, 1)])
def test_age_hits_and_skips(max_age, min_hits):
    """Three streams; stream 1 skips frames 2-4 (host skip), stream 2 sees no detections in frames 1-3: ages
    accumulate and the prune follows max_age / min_hits."""
    a = [(0, 0.9, grid_box(k)) for k in range(5)]
    b = [(0, 0.8, grid_box(k, dx=1.0)) for k in range(0, 5, 2)]
    frames = [[a, a, a], [b, b, []], [b, None, []], [a, None, []], [b, None, a], [a, a, b]]
    run_all(Case(f"state-{max_age}-{min_hits}", frames, cfg=(max_age, min_hits, 0.5)))


def test_device_skip_mask_ages_like_host_skip():
    import torch

    h = handle()
    a = [(0, 0.9, grid_box(k)) for k in range(5)]
    case = Case("skipmask", [[a, a], [a, a], [a, a], [a, a]], cfg=(1, 0, 0.5))
    host = Case("skipmask", [[a, a], [a, None], [a, None], [a, a]], cfg=(1, 0, 0.5))
    # the device mask stands in for the host flags of `host`: run the host-flag case once to get the oracle rows,
    # then the mask case frame by frame against the same oracle
    ora = O.IouTracker(1, 0.5, 0)
    for s in range(2):
        h.tracker_reset(s)
    h.tracker_set_next_id(1)
    mask = torch.zeros(2, dtype=torch.uint8, device="cuda")
    try:
        h.set_skip_mask(mask)
        for t, frame in enumerate(case.frames):
            mask.copy_(torch.tensor([0, 1 if host.frames[t][1] is None else 0], dtype=torch.uint8))
            out = h.tracker_update([0, 1], update_soa(dets_f64(frame), True), 1, 0, 0.5, f64=True)
            got = soa_host(out)
            for s in range(2):
                check_stream(rows_of(got, s), ora.update(f"s{s}", dets_f64(host.frames[t])[s]), ("skipmask", t, s))
    finally:
        h.set_skip_mask(None)


def test_hundred_streams_one_launch():
    """100 streams in one k_tracker launch (ids are drawn in batch order by the last CTA), with empty streams and
    skips; the fused tick at 64 streams."""
    rng = np.random.default_rng(3)
    frames = []
    for t in range(3):
        fr = []
        for s in range(100):
            if s % 9 == 4 and t == 1:
                fr.append(None)
            elif s % 7 == 3:
                fr.append([])
            else:
                n = int(rng.integers(0, 6))
                fr.append([(k % 2, rank_conf(k), grid_box(k + 5 * (s % 3), dx=0.5 * t)) for k in range(n)])
        frames.append(fr)
    run_all(Case("streams100", frames, cfg=(1, 0, 0.5)), UPDATE_ENTRIES)
    run_all(Case("streams64", [fr[:64] for fr in frames], cfg=(1, 0, 0.5)), TICK_ENTRIES)


def test_ids_above_32_bits():
    f = [(0, rank_conf(k), grid_box(k)) for k in range(70)]
    g = [(0, rank_conf(k), grid_box(k + 100)) for k in range(3)]
    run_all(Case("id62", [[f, g], [g, f]], cfg=(30, 0, 0.5), next_id=2 ** 62), ("f64", "post", "sortnms", "dense"))


def test_id_base():
    """With id_base, stream b numbers its new tracks id_base[b] + creation ordinal and the shared counter is not
    touched."""
    h = handle()
    a = [(0, 0.9, grid_box(k)) for k in range(4)]
    b = [(0, 0.8, grid_box(k, dx=1.0)) for k in range(0, 6)]
    for s in range(2):
        h.tracker_reset(s)
    h.tracker_set_next_id(7)
    ora = O.IouTracker(30, 0.5, 0)
    ids = {}
    bases = [[1000, 2 ** 40], [5000, 2 ** 40 + 100]]
    for t, frame in enumerate([[a, b], [b, a]]):
        out = h.tracker_update([0, 1], update_soa(dets_f64(frame), True), 30, 0, 0.5, id_base=bases[t], f64=True)
        got = soa_host(out)
        for s in range(2):
            want = ora.update(f"s{s}", dets_f64(frame)[s])
            new = [w for w in want if w.track_id not in ids]
            for k, w in enumerate(new):
                ids[w.track_id] = bases[t][s] + k
            rows = rows_of(got, s)
            assert rows[0] == [ids[w.track_id] for w in want], (t, s)
            check_stream((list(range(len(want))),) + rows[1:], [O.Trk(k, w.class_id, w.confidence, w.bbox_xyxy, w.age,
                                                                      w.hits) for k, w in enumerate(want)], (t, s))
    out = h.tracker_update([0], update_soa([[O.Det(2, 0.5, (0.0, 0.0, 1.0, 1.0))]], True), 30, 0, 0.5, f64=True)
    assert soa_host(out)["track_id"][0, -1] == 7  # the shared counter is where it was set


def test_more_than_32768_detections_are_refused():
    """``last_det`` is 16 bits wide: one update takes at most 32768 detections per stream.  32,800 (a duplicate pile
    of 32700, then re-detections of 100 tracks) are refused and leave the tracker as it was: the same tracker then
    takes a small update, exactly 32768 detections whose last re-detects a track, and a small update again, each equal
    to the oracle's.  The C entry points refuse a detection table of 32769 rows per stream."""
    from realtime_video_analytics_32streams_b200 import B200IouTracker, TrackerConfig
    from realtime_video_analytics_32streams_b200 import _native as N

    h = handle()
    seed = [O.Det(0, 0.9, grid_box(k)) for k in range(100)]
    pile = [O.Det(1, 0.5, (3000.0, 3000.0, 3050.0, 3050.0))]
    small = [O.Det(0, 0.7, grid_box(k, dx=0.5)) for k in range(0, 100, 25)] + [O.Det(2, 0.6, grid_box(300))]
    trk = B200IouTracker(TrackerConfig(max_age=30, max_iou_distance=0.5, min_hits=0), handle=h)
    ora = O.IouTracker(30, 0.5, 0)
    try:
        def check(dets, t):
            got, want = trk.update("s", dets), ora.update("s", dets)
            check_stream(([x.track_id for x in got], [x.class_id for x in got], [x.confidence for x in got],
                          [x.bbox_xyxy for x in got], [x.age for x in got], [x.hits for x in got]), want, ("32768", t))

        check(seed, 0)
        big = pile * 32700 + [O.Det(0, 0.8, grid_box(k, dx=1.0)) for k in range(100)]
        assert len(big) == 32800
        with pytest.raises(N.B200VAError) as e:
            trk.update("s", big)
        assert e.value.status == N.ERR_INVALID
        check(small, 1)
        check(pile * 32767 + [O.Det(0, 0.8, grid_box(7, dx=1.0))], 2)
        check(small, 3)
    finally:
        trk.close()
    h.tracker_reset(0)
    for f64 in (False, True):
        ft = np.float64 if f64 else np.float32
        soa = {"bbox_xyxy": cu(np.zeros((1, 32769, 4), ft)), "conf": cu(np.zeros((1, 32769), ft)),
               "cls": cu(np.zeros((1, 32769), np.int32)), "count": cu(np.array([1], np.int32))}
        with pytest.raises(N.B200VAError) as e:
            h.tracker_update([0], soa, 30, 0, 0.5, f64=f64)
        assert e.value.status == N.ERR_INVALID


def test_tick_nan_centre_after_tracking():
    """End to end: a frame whose leading box has a NaN centre x after its object was tracked.  The post-process hands
    that box to the tracker (x1 = x2 = NaN), and tracker.py's min / max match it to the track."""
    import torch
    from realtime_video_analytics_32streams_b200 import _native as N

    for entry in ("post", "dense", "sortnms"):
        h = handle(ENTRY_ENV.get(entry, ()))
        h.tracker_reset(0)
        h.tracker_set_next_id(1)
        meta = {"orig_shape": (FRAME, FRAME), "scale": 1.0, "pad": (0, 0)}
        ora = O.IouTracker(30, 0.5, 0)
        tracks = h.alloc_tracks(1)
        for t, (cx, hh) in enumerate(((100.0, 10.0), (NAN, 6.0), (100.0, 10.0))):
            head = np.zeros((1, 5 + NC, 64), np.float32)
            head[0, :4, 0] = (cx, 100.0, 20.0, hh)
            head[0, 4, 0], head[0, 5, 0] = 1.0, 0.9
            head[0, :4, 1] = (300.0, 300.0, 10.0, 10.0)
            head[0, 4, 1], head[0, 5, 1] = 1.0, 0.8
            want_d = O.filter_detections(O.postprocess(head, meta, CONF, 0.5), CONF)
            plan = h.plan_tick(head=cu(head), metas=[N.Letterbox(FRAME, FRAME, FRAME, FRAME, 0, 0, 1.0)], conf_thr=CONF,
                               iou_thr=0.5, filter_conf=CONF, slots=[0], tracker_cfg=(30, 0, 0.5), tracks=tracks,
                               schedule=1)
            profiled(lambda: h.tick(plan))
            d = plan.dets
            m = int(d["count"].cpu()[0])
            assert m == len(want_d), (entry, t)
            assert np.array_equal(canon(d["bbox_xyxy"][0, :m].cpu().numpy()), canon([w.bbox_xyxy for w in want_d]))
            want = ora.update("s", want_d)
            if t == 1:
                assert want[0].hits == 2 and want[0].bbox_xyxy[0] != want[0].bbox_xyxy[0]  # the NaN box matched
            check_stream(rows_of(soa_host(tracks), 0), want, ("nan-tick", entry, t))
        h.poll_status()


def test_zz_every_tracker_kernel_ran():
    """Runs last in this module: every entry kernel was observed by the profiler, in the cases above and in one
    session over a small case through k_tracker, both k_post_track instantiations and k_dense_resolve_track."""
    import torch
    from torch.profiler import ProfilerActivity, profile

    case = Case("coverage", [[(0, 0.9, grid_box(0))], [(0, 0.8, grid_box(0, dx=1.0)), (1, 0.7, grid_box(1))]])
    for _ in range(3):  # (a session whose trace came back empty is run again, see `profiled`)
        with profile(activities=[ProfilerActivity.CUDA]) as prof:
            for e in ("f64", "post", "ultra", "dense"):
                run_case(case, e)
            torch.cuda.synchronize()
        names = sorted({e.name for e in prof.events()})
        ran = {kernel_of(n) for n in names} - {None}
        SEEN.update(ran)
        if ran:
            break
    assert set(KERNELS) <= SEEN, (sorted(set(KERNELS) - SEEN), [n[:80] for n in names])
