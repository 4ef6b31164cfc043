"""Every head-decode kernel against the NumPy decode (oracle.hotpath / oracle.ultralytics_restate) at the shapes and
scores where a decode goes wrong.

The decode step has five kernels, picked by layout, alignment, class count, frames per launch and B200VA_DECODE_IMPL:
k_decode_cm_split<8, 12>, k_decode_cm<4>, k_decode_cm<1>, k_decode_ring (opt-in) and k_decode_am.  One handle per
forced variant (0 auto, 1 register kernels, 2 ring, 3 split), every case family records with torch.profiler which
decode kernel ran and asserts it is the intended one, and the last test asserts that all five ran.

Outputs are compared as bit patterns (classes exactly, confidences and boxes through ``view(np.uint32)``, NaN
positions equal), so -0.0 against +0.0 and a flushed subnormal are differences.  iou_thr = 1.0 keeps almost every
candidate, so the decode itself is what is compared; 0.5 runs the ordinary NMS on top."""

import numpy as np
import pytest

from oracle import hotpath as O
from oracle import ultralytics_restate as U

pytestmark = pytest.mark.gpu

IN_HW = (640, 640)
GEOMS = [(1080, 1920), (720, 1280), (1920, 1080), (480, 640)]  # source frames of the letterbox metas, mixed per batch
KERNELS = ("k_decode_cm_split", "k_decode_cm<4>", "k_decode_cm<1>", "k_decode_ring", "k_decode_am")
SEEN = set()  # decode kernels observed by the profiler in this module


@pytest.fixture(scope="module")
def HS():
    """B200VA_DECODE_IMPL -> handle (the knob is read when the handle is created)."""
    import os

    import torch
    from realtime_video_analytics_32streams_b200 import _native

    assert torch.cuda.is_available()
    handles = {}
    try:
        for impl in ("0", "1", "2", "3"):
            os.environ["B200VA_DECODE_IMPL"] = impl
            try:
                handles[impl] = _native.Handle(device=0, max_batch=128, max_anchors=8400, max_candidates=4096,
                                               max_dets=4096, max_streams=2, max_tracks=64)
            finally:
                del os.environ["B200VA_DECODE_IMPL"]
        yield handles
        for h in handles.values():
            h.poll_status()
    finally:
        for h in handles.values():
            h.close()


# ---- inputs ------------------------------------------------------------------------------------------------------

def _cls0(C, mode):
    return 5 if mode == "ref" and C > 5 else 4


def _unique(rng, n, lo, hi):
    s = np.unique(rng.uniform(lo, hi, 4 * n + 8).astype(np.float32))
    rng.shuffle(s)
    assert len(s) >= n
    return s[:n]


# distances between two equal maxima of one anchor: neighbours, ring groups of four, split parts (per = 2, 3, 12),
# ring stages (17-24 rows), anchor-major lanes (c and c + 32)
DUP_OFFSETS = (1, 2, 3, 4, 5, 8, 12, 16, 17, 20, 21, 24, 31, 32, 33, 64)


def make_head(seed, C, A, n_cand, mode="ref", ties=False, lo=0.3, hi=0.99):
    """Head [C, A]: boxes inside the network input, class rows in [0, 0.2) (under the 0.25 threshold), objectness in
    [0.6, 1] (REF_COMPAT with C > 5).  n_cand anchors carry a maximum -- distinct float32 values, or multiples of 1/8
    with ties=True -- in the first row, the last row, every row, one row, or two / three rows DUP_OFFSETS apart."""
    rng = np.random.default_rng(seed)
    cls0 = _cls0(C, mode)
    n_cls = C - cls0
    h = np.empty((C, A), np.float32)
    h[0] = rng.uniform(0, IN_HW[1], A)
    h[1] = rng.uniform(0, IN_HW[0], A)
    h[2] = rng.uniform(4, 80, A)
    h[3] = rng.uniform(4, 80, A)
    if cls0 == 5:
        h[4] = rng.uniform(0.6, 1.0, A)
    h[cls0:] = rng.uniform(0, 0.2, (n_cls, A))
    n_cand = min(n_cand, A)
    picks = rng.permutation(A)[:n_cand]
    scores = (rng.integers(3, 8, n_cand) / 8).astype(np.float32) if ties else _unique(rng, n_cand, lo, hi)
    for a, s in zip(picks, scores):
        kind = int(rng.integers(6))
        r = int(rng.integers(n_cls))
        if kind == 0:
            rows = [0]
        elif kind == 1:
            rows = [n_cls - 1]
        elif kind == 2:
            rows = list(range(n_cls))
        elif kind == 3:
            rows = [r]
        else:
            d = int(DUP_OFFSETS[rng.integers(len(DUP_OFFSETS))])
            r = int(rng.integers(max(n_cls - d, 1)))
            rows = [r, r + d] if kind == 4 else [r, r + d, r + 2 * d]
        rows = [x for x in rows if x < n_cls]
        h[cls0 + np.asarray(rows), a] = s
    return h


def _dev(a, offset=False):
    """CUDA copy of `a`; offset=True: a contiguous view one float into a larger buffer (a base that is not 16-byte
    aligned)."""
    import torch

    t = torch.from_numpy(np.ascontiguousarray(a)).cuda()
    if not offset:
        return t
    buf = torch.zeros(t.numel() + 1, dtype=torch.float32, device="cuda")
    buf[1:].copy_(t.view(-1))
    v = buf[1:].view(t.shape)
    assert v.is_contiguous() and v.data_ptr() % 16 == 4
    return v


def _metas(B):
    from realtime_video_analytics_32streams_b200 import _native as N

    return [N.letterbox_meta(*GEOMS[b % len(GEOMS)], *IN_HW) for b in range(B)]


def _frame_hw(B):
    return [GEOMS[b % len(GEOMS)] for b in range(B)]


# ---- observation -------------------------------------------------------------------------------------------------

def _profiled(fn, expect):
    """Run fn; with `expect`, record the decode kernels it launched and assert that `expect` was one of them."""
    if expect is None:
        return fn()
    import torch
    from torch.profiler import ProfilerActivity, profile

    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        out = fn()
        torch.cuda.synchronize()
    names = {e.name for e in prof.events() if "k_decode" in e.name}
    ran = {k for k in KERNELS if any(k in n for n in names)}
    SEEN.update(ran)
    assert expect in ran, (expect, sorted(names))
    return out


def _same_bits(got, want):
    got = np.asarray(got, np.float32)
    want = np.asarray(want, np.float32).reshape(got.shape)
    gn, wn = np.isnan(got), np.isnan(want)
    return np.array_equal(gn, wn) and np.array_equal(got[~gn].view(np.uint32), want[~wn].view(np.uint32))


def _check_frame(out, b, cls, conf, box, what):
    n = int(out["count"][b].item())
    assert n == len(cls), (what, b, n, len(cls))
    assert out["cls"][b, :n].cpu().numpy().tolist() == [int(c) for c in cls], (what, b)
    assert _same_bits(out["conf"][b, :n].cpu().numpy(), conf), (what, b)
    assert _same_bits(out["bbox_xyxy"][b, :n].cpu().numpy(), np.asarray(box, np.float32).reshape(-1, 4)), (what, b)
    return n


def run_ref(H, heads, conf, iou, layout="cm", mode="ref", classes=None, aware=False, filt=None, offset=False,
            expect=None, metas=None, skip=()):
    """H.postprocess on heads [B, C, A] (given channel-major; sent as `layout`) against O.postprocess frame by frame.
    Frames in `skip` are gated by the handle's skip mask and must report no detections."""
    from realtime_video_analytics_32streams_b200 import _native as N

    B = heads.shape[0]
    metas = metas or _metas(B)
    host = heads if layout == "cm" else heads.transpose(0, 2, 1)
    dev = _dev(host, offset)
    kw = dict(classes=classes, layout=N.HEAD_CHANNEL_MAJOR if layout == "cm" else N.HEAD_ANCHOR_MAJOR,
              score_mode=N.SCORE_V8_NATIVE if mode == "v8" else N.SCORE_REF_COMPAT,
              nms_mode=N.NMS_CLASS_AWARE if aware else N.NMS_AGNOSTIC)
    if filt is not None:
        kw["filter_conf"] = filt
    out = _profiled(lambda: H.postprocess(dev, metas, conf, iou, **kw), expect)
    total = 0
    with np.errstate(invalid="ignore", over="ignore"):
        for b in range(B):
            if b in skip:
                assert int(out["count"][b].item()) == 0, b
                continue
            ref = O.postprocess(heads[b], metas[b].as_meta(), conf, iou, classes, v8_native=mode == "v8",
                                class_aware=aware, layout="cm")
            if filt is not None:
                ref = O.filter_detections(ref, filt)
            total += _check_frame(out, b, [d.class_id for d in ref], [d.confidence for d in ref],
                                  [d.bbox_xyxy for d in ref], ("ref", layout, mode, conf, iou))
    return total


def run_ultra(H, heads, conf, iou, layout="cm", classes=None, agnostic=False, max_det=300, filt=None, offset=False,
              expect=None, skip=()):
    """H.postprocess_ultralytics against U.postprocess (+ the float64 filter on what it returns)."""
    from realtime_video_analytics_32streams_b200 import _native as N

    B = heads.shape[0]
    fhw = _frame_hw(B)
    host = heads if layout == "cm" else heads.transpose(0, 2, 1)
    dev = _dev(host, offset)
    out = _profiled(lambda: H.postprocess_ultralytics(
        dev, fhw, IN_HW, conf_thr=conf, iou_thr=iou, classes=classes, agnostic=agnostic, max_det=max_det,
        layout=N.HEAD_CHANNEL_MAJOR if layout == "cm" else N.HEAD_ANCHOR_MAJOR, filter_conf=filt), expect)
    total = 0
    with np.errstate(invalid="ignore", over="ignore"):
        for b in range(B):
            if b in skip:
                assert int(out["count"][b].item()) == 0, b
                continue
            want = U.postprocess(heads[b], IN_HW, fhw[b], conf, iou, classes, agnostic, max_det)
            if filt is not None:
                want = [w for w in want if w[1] >= filt]
            total += _check_frame(out, b, [c for c, _, _ in want], [s for _, s, _ in want], [bx for _, _, bx in want],
                                  ("ultra", layout, conf, iou, agnostic))
    return total


def expected_kernel(impl, layout, C, A, mode, frames, offset=False, skip=False):
    """The host's dispatch rule (postprocess_impl), restated."""
    if layout == "am":
        return "k_decode_am"
    n_cls = C - _cls0(C, "v8" if mode == "ultra" else mode)
    vec4 = A % 4 == 0 and not offset
    if vec4 and 16 <= n_cls <= 96 and (impl == "3" or (impl == "0" and frames <= 8)):
        return "k_decode_cm_split"
    if vec4 and A >= 128 and impl == "2" and not skip:
        return "k_decode_ring"
    return "k_decode_cm<4>" if vec4 else "k_decode_cm<1>"


def run(H, impl, heads, mode, conf, iou, layout="cm", offset=False, profile=True, **kw):
    B, C, A = heads.shape
    expect = expected_kernel(impl, layout, C, A, mode, min(B, 64), offset, bool(kw.get("skip"))) if profile else None
    if mode == "ultra":
        return run_ultra(H, heads, conf, iou, layout, offset=offset, expect=expect, **kw)
    return run_ref(H, heads, conf, iou, layout, mode, offset=offset, expect=expect, **kw)


# ---- shapes and argmax -------------------------------------------------------------------------------------------

# (anchors, channels): 1..8400 anchors, 15 / 16 / 17 / 96 / 97 class rows around the split limits (REF_COMPAT;
# one more row each in V8_NATIVE), 3549 and 7581 (416 x 416 and 608 x 608 YOLOv8 exports: A % 4 != 0)
SHAPES = [(1, 5), (3, 6), (5, 20), (256, 20), (127, 21), (128, 21), (128, 22), (132, 84), (3549, 85), (7581, 101),
          (8400, 101), (8400, 102)]


@pytest.mark.parametrize("A,C", SHAPES)
def test_decode_shapes_and_argmax(HS, A, C):
    """Every variant, both layouts, REF_COMPAT / V8_NATIVE / Ultralytics semantics, 2 and 3 frames (tiles and rows
    that end part-way, ring tiles of several frames), duplicated maxima at part / group / stage / lane distances."""
    n_cand = min(A, 150)
    for mode in ("ref", "v8", "ultra"):
        heads = np.stack([make_head(1000 * A + C + 7 * f + {"ref": 0, "v8": 1, "ultra": 2}[mode], C, A, n_cand,
                                    "v8" if mode == "ultra" else mode) for f in range(3 if A > 1000 else 2)])
        for impl in ("0", "1", "2", "3"):
            for iou in (1.0, 0.5):
                run(HS[impl], impl, heads, mode, 0.25, iou, profile=iou == 1.0)
        run(HS["0"], "0", heads, mode, 0.25, 1.0, layout="am")
        run(HS["0"], "0", heads, mode, 0.25, 0.5, layout="am", profile=False)
        if A % 4 == 0:  # a head base one float into its buffer: the unaligned channel-major kernel
            for impl in ("0", "2", "3"):
                run(HS[impl], impl, heads, mode, 0.25, 1.0, offset=True)


def test_decode_all_rows_equal_and_every_row(HS):
    """Per anchor: all class rows equal (np.argmax: row 0), and the maximum alone in each row in turn."""
    for C in (21, 22, 85, 102):
        for mode in ("ref", "v8", "ultra"):
            cls0 = _cls0(C, "v8" if mode == "ultra" else mode)
            n_cls = C - cls0
            rng = np.random.default_rng(C)
            A = 4 * ((2 * n_cls + 3) // 4) + 128
            h = make_head(C, C, A, 0, "v8" if mode == "ultra" else mode)
            s = _unique(rng, A, 0.3, 0.99)
            for a in range(A):
                if a < n_cls:
                    h[cls0 + a, a] = s[a]               # the maximum in row a
                elif a < 2 * n_cls:
                    h[cls0:, a] = s[a]                  # every row equal
                elif a % 3 == 0:
                    h[cls0 + (a % n_cls), a] = s[a]
                    h[cls0 + n_cls - 1, a] = s[a]       # and again in the last row
            heads = h[None]
            for impl in ("0", "1", "2", "3"):
                run(HS[impl], impl, heads, mode, 0.25, 1.0)
            run(HS["0"], "0", heads, mode, 0.25, 1.0, layout="am")


def test_decode_score_ties_across_anchors(HS):
    """Equal scores on different anchors: higher anchor first (reference modes), lower anchor first (Ultralytics)."""
    for A, C in ((3549, 85), (8400, 22), (128, 101)):
        for mode in ("ref", "v8", "ultra"):
            heads = np.stack([make_head(77 + A + f, C, A, 200, "v8" if mode == "ultra" else mode, ties=True)
                              for f in range(2)])
            for impl in ("0", "1", "2", "3"):
                for iou in (1.0, 0.5):
                    run(HS[impl], impl, heads, mode, 0.25, iou, profile=iou == 1.0)
            run(HS["0"], "0", heads, mode, 0.25, 0.5, layout="am")


# ---- non-finite and signed values --------------------------------------------------------------------------------

INF, NAN = np.inf, np.nan
# (objectness, class scores) of C = 9 heads: REF_COMPAT reads column 4 as objectness, V8_NATIVE / Ultralytics as
# class 0 -- the same rows test both
SPECIAL = [
    (1.0, [0.5, NAN, 0.1, 0.1]),       # NaN after the maximum
    (1.0, [NAN, 0.6, 0.1, 0.1]),       # NaN before it
    (1.0, [0.1, 0.1, 0.1, NAN]),       # NaN in the last row
    (NAN, [0.8, 0.1, 0.1, 0.1]),       # NaN objectness
    (0.0, [INF, 0.1, 0.1, 0.1]),       # 0 x inf = NaN
    (INF, [0.5, 0.0, 0.1, 0.1]),       # inf x 0 = NaN
    (1.0, [INF, 0.1, 0.1, 0.1]),
    (1.0, [0.1, INF, INF, 0.2]),
    (1.0, [-INF, -INF, -INF, -INF]),
    (1.0, [0.3, -INF, 0.9, 0.9]),
    (-1.0, [INF, 0.5, 0.6, 0.7]),      # -inf, -0.5, ...: negative scores
    (1.0, [-0.0, 0.0, -0.0, 0.0]),     # equal zeros: row 0, -0.0
    (1.0, [0.0, -0.0, 0.0, -0.0]),
    (-1.0, [0.0, 0.0, 0.0, 0.0]),      # -0.0 products
    (0.0, [-0.5, 0.1, 0.2, 0.3]),      # -0.0, +0.0, ...
    (1.0, [-0.3, -0.2, -0.25, -0.2]),
    (1.0, [-0.6, -0.7, -0.9, -0.8]),
    (1.0, [1e-40, 2e-40, 0.0, 0.0]),   # subnormal scores
    (1e-20, [1e-20, 5e-21, 0.0, 0.0]), # a subnormal product
    (1.0, [3e-45, 0.0, 0.0, 0.0]),
    (1.0, [NAN, NAN, NAN, NAN]),
    (1.0, [0.0, 0.0, 0.0, 1e-38]),
]
# (column, value) written into the box rows of the regular anchors that follow SPECIAL
BOX_EDITS = [[(0, INF)], [(1, -INF)], [(2, INF)], [(3, NAN)], [(0, 1e30)], [(2, 1e30), (3, 1e30)],
             [(0, NAN), (1, NAN), (2, NAN), (3, NAN)], [(2, -50.0)], [(0, -1e30)], [(3, -INF)]]


def special_head(seed, A, mode):
    rng = np.random.default_rng(seed)
    h = make_head(seed, 9, A, 0, mode)
    h[4] = 1.0 if mode == "ref" else 0.05  # objectness 1, or a class row under the regular scores
    k = len(SPECIAL)
    for a, (obj, sc) in enumerate(SPECIAL):
        h[4, a] = obj
        h[5:, a] = sc
    s = _unique(rng, A - k, 0.3, 0.99)
    for j, a in enumerate(range(k, A)):
        h[5 + j % 4, a] = s[j]
    for j, edits in enumerate(BOX_EDITS):
        for col, v in edits:
            h[col, k + 3 * j] = v
    return h


@pytest.mark.parametrize("conf", [0.25, 0.0, -0.25, -1.0, 1e-40, 5e-41, 1e-45, -0.0])
def test_decode_nonfinite_signed_subnormal(HS, conf):
    """NaN scores at and away from the maximum, NaN objectness, 0 x inf, +-inf, +-0 scores, negative scores under
    negative thresholds, subnormal scores and thresholds (no flush to zero), box rows with +-inf, NaN and 1e30."""
    for A in (132, 23):
        for mode in ("ref", "v8", "ultra"):
            heads = np.stack([special_head(5 + A + f, max(A, 64), "ref" if mode == "ref" else "v8")[:, :A]
                              for f in range(2)])
            for impl in ("0", "1", "2", "3"):
                for iou in (1.0, 0.5):
                    run(HS[impl], impl, heads, mode, conf, iou, profile=iou == 1.0 and conf == 0.25)
            run(HS["0"], "0", heads, mode, conf, 1.0, layout="am", profile=conf == 0.25)


def test_signed_zero_scores_rank_equal(HS):
    """Class scores [0, -0, 0, -0, .3, .3, -1, 0] at anchors 0..7 on disjoint boxes: NumPy sees +0.0 and -0.0 as equal
    scores (ordered higher anchor first, 5 4 7 3 2 1 0) and keeps the sign of each; torch's stable descending sort
    orders them lower anchor first."""
    A = 8
    h = np.zeros((6, A), np.float32)
    h[0] = 40 + 70 * np.arange(A)
    h[1] = 300
    h[2] = h[3] = 30
    h[4] = 1.0
    h[5] = np.array([0.0, -0.0, 0.0, -0.0, 0.3, 0.3, -1.0, 0.0], np.float32)
    heads = h[None]
    for impl in ("0", "1", "2", "3"):
        for conf in (0.0, -0.25):
            for mode in ("ref", "v8"):
                for iou in (0.5, 1.0):
                    run(HS[impl], impl, heads, mode, conf, iou)
        run(HS[impl], impl, heads, "ultra", -0.5, 0.5)
    for layout in ("cm", "am"):
        run(HS["0"], "0", heads, "ref", 0.0, 0.5, layout=layout)
        run(HS["0"], "0", heads, "ultra", -0.5, 0.5, layout=layout)
    # the same zeros next to enough anchors that the split, register and ring kernels all see them (A % 4 == 0), with
    # a second zero of the other sign in later rows
    for mode in ("ref", "v8", "ultra"):
        cls0 = 5 if mode == "ref" else 4
        big = make_head(11, 22, 256, 60, "ref" if mode == "ref" else "v8")
        big[4, :8] = 1.0
        big[cls0:, :8] = 0.0
        big[cls0, :8] = h[5]
        big[cls0 + 5, 1] = big[cls0 + 9, 2] = big[cls0 + 4, 0] = -0.0
        big[cls0 + 13, 3] = 0.0
        for impl in ("0", "1", "2", "3"):
            run(HS[impl], impl, big[None], mode, -0.5 if mode == "ultra" else 0.0, 1.0)
        run(HS["0"], "0", big[None], mode, -0.5 if mode == "ultra" else 0.0, 1.0, layout="am")


# ---- threshold edges ---------------------------------------------------------------------------------------------

@pytest.mark.parametrize("thr", [0.45, 0.1, 0.25])
def test_decode_threshold_edges(HS, thr):
    """Scores float32(thr) and one ulp either side: `>=` in the reference modes, strict `>` for Ultralytics, and the
    float64 filter_conf fold (float32(0.45) < 0.45 < float32(0.1) is not: 0.1 rounds up)."""
    t = np.float32(thr)
    edge = [np.nextafter(t, np.float32(0)), t, np.nextafter(t, np.float32(1))]
    A, C = 256, 22
    for mode in ("ref", "v8", "ultra"):
        h = make_head(int(thr * 1000), C, A, 0, "ref" if mode == "ref" else "v8")
        h[4:] = np.minimum(h[4:], np.float32(0.05))
        if mode == "ref":
            h[4] = 1.0
        for a in range(90):
            h[5 + a % 17, a] = edge[a % 3]
        heads = h[None]
        for impl in ("0", "1", "2", "3"):
            for filt in (None, thr):
                assert run(HS[impl], impl, heads, mode, thr, 1.0, filt=filt) > 0
        run(HS["0"], "0", heads, mode, thr, 1.0, layout="am", filt=thr)


# ---- whitelist ---------------------------------------------------------------------------------------------------

def test_whitelist_ids(HS):
    """An empty list (no filter), negative ids, ids >= the class count and duplicates: np.isin."""
    for mode in ("ref", "v8", "ultra"):
        heads = np.stack([make_head(31 + f, 85, 3548, 150, "ref" if mode == "ref" else "v8") for f in range(2)])
        for impl in ("0", "1", "3"):
            for classes in ([], [-1, 3, 3, 500, 7], [79, 80, 81], [-5], [0, 0]):
                run(HS[impl], impl, heads, mode, 0.25, 1.0, classes=classes)
        run(HS["0"], "0", heads, mode, 0.25, 0.5, layout="am", classes=[-1, 3, 3, 500, 7])
    run(HS["0"], "0", heads, "ref", 0.25, 0.5, layout="am", classes=[-1, 3, 3, 500, 7], aware=True)


def _wide_head(mode):
    """2106 channels (2101 / 2102 classes): maxima on classes 0, 5, 2046..2050, 2100 and the last class."""
    C, A = 2106, 128
    cls0 = _cls0(C, mode)
    h = make_head(2106, C, A, 0, mode)
    if cls0 == 5:
        h[4] = 1.0
    rng = np.random.default_rng(7)
    s = _unique(rng, A, 0.3, 0.99)
    targets = [0, 5, 2046, 2047, 2048, 2049, 2050, 2100, C - cls0 - 1]
    for a in range(A):
        h[cls0 + targets[a % len(targets)], a] = s[a]
    return h[None]


def test_whitelist_ids_beyond_2047(HS):
    """Ids 2047, 2048 and 2050 on a head with more than 2048 classes.  The kernels hold the whitelist as a 2048-bit
    map: 2047 filters exactly like np.isin, an id in [2048, class count) is refused with B200VA_ERR_INVALID instead of
    silently matching nothing, an id at or above the class count is accepted (it matches nothing)."""
    from realtime_video_analytics_32streams_b200 import _native as N

    for mode in ("ref", "v8", "ultra"):
        heads = _wide_head("v8" if mode == "ultra" else mode)
        for impl in ("0", "1"):
            assert run(HS[impl], impl, heads, mode, 0.25, 1.0) == 128
            for aware in ((False, True) if mode != "ultra" else (False,)):
                kw = {"aware": aware} if mode != "ultra" else {}
                assert run(HS[impl], impl, heads, mode, 0.25, 0.5, classes=[2047], **kw) > 0
                assert run(HS[impl], impl, heads, mode, 0.25, 1.0, classes=[2047, 3000, 5], **kw) > 0
                for classes in ([2048], [2047, 2050], [2050]):
                    with pytest.raises(N.B200VAError) as e:
                        run(HS[impl], impl, heads, mode, 0.25, 1.0, classes=classes, profile=False, **kw)
                    assert e.value.status == N.ERR_INVALID
        run(HS["0"], "0", heads, mode, 0.25, 1.0, layout="am", classes=[2047, 2200])
        with pytest.raises(N.B200VAError):
            run(HS["0"], "0", heads, mode, 0.25, 1.0, layout="am", classes=[2050], profile=False)
    # a 2050 whitelist entry on an 80-class head matches nothing and is accepted
    heads = np.stack([make_head(9, 85, 3549, 100)])
    run(HS["0"], "0", heads, "ref", 0.25, 1.0, classes=[2050, 3])
    run(HS["0"], "0", heads, "ref", 0.25, 1.0, classes=[2050])


# ---- launch groups, gating and capacity --------------------------------------------------------------------------

def _batch_heads(B, C, A, seed, mode="ref"):
    """B distinct frames: frames 64..69 carry 300 candidates (the dense-scene NMS variants engage after them), the
    rest 20-80."""
    mode = "ref" if mode == "ref" else "v8"
    return np.stack([make_head(seed + b, C, A, 300 if 64 <= b < 70 else 20 + (b * 7) % 61, mode) for b in range(B)])


@pytest.mark.parametrize("B", [64, 65, 128])
def test_launch_groups(HS, B):
    """More than 64 frames: launch groups of 64 offset the metas, output rows and candidate scratch.  Four frame
    geometries mixed; every frame distinct; a follow-up call after frames with more than 256 candidates runs the
    grid / dense NMS variants per group."""
    for impl, (C, A) in (("0", (22, 3549)), ("2", (85, 1024)), ("1", (85, 1024))):
        heads = _batch_heads(B, C, A, 100 * B + int(impl))
        for rep in range(2):
            for iou in (0.5, 1.0):
                run(HS[impl], impl, heads, "ref", 0.25, iou, profile=rep == 0 and iou == 1.0)
        run(HS[impl], impl, heads, "ref", 0.25, 0.5, aware=True, filt=0.6)
        run(HS[impl], impl, _batch_heads(B, C, A, 7 * B + int(impl), "ultra"), "ultra", 0.25, 0.45)
    run(HS["0"], "0", _batch_heads(B, 85, 300, 5), "ref", 0.25, 0.5, layout="am")


def test_launch_groups_skip_mask(HS):
    """set_skip_mask with gated frames in both launch groups: a gated frame reports 0 detections, every other frame
    matches the oracle."""
    import torch

    B = 128
    gated = {0, 5, 63, 64, 65, 100, 127}
    mask = torch.zeros(B, dtype=torch.uint8, device="cuda")
    mask[sorted(gated)] = 1
    for impl, (C, A) in (("0", (22, 3549)), ("2", (85, 1024)), ("3", (22, 1024))):
        heads = _batch_heads(B, C, A, 7 + int(impl))
        H = HS[impl]
        H.set_skip_mask(mask)
        try:
            for iou in (0.5, 1.0):
                run(H, impl, heads, "ref", 0.25, iou, skip=gated)
            run(H, impl, _batch_heads(B, C, A, 9, "ultra"), "ultra", 0.25, 0.45, skip=gated)
            run(H, impl, heads[:8], "ref", 0.25, 0.5, skip={b for b in gated if b < 8})
            run(H, "0", heads, "ref", 0.25, 0.5, layout="am", skip=gated)
        finally:
            H.set_skip_mask(None)
        run(H, impl, heads, "ref", 0.25, 0.5)


def test_candidate_capacity(HS):
    """Exactly max_candidates (4096) candidates: exact output, no flag.  One more: ERR_CAPACITY from poll_status, and
    the flag is cleared by that poll."""
    from realtime_video_analytics_32streams_b200 import _native as N

    H = HS["1"]
    H.poll_status()
    A = 8400
    h = make_head(4096, 22, A, 0)
    h[4] = 1.0
    k = np.arange(4097)
    h[0, :4097] = 8 + (k % 64) * 10.0  # disjoint boxes on a grid
    h[1, :4097] = 8 + (k // 64) * 10.0
    h[2, :4097] = h[3, :4097] = 6.0
    rng = np.random.default_rng(1)
    h[5 + k % 17, k] = _unique(rng, 4097, 0.3, 0.99)
    exact = h.copy()
    exact[5:, 4096] = 0.01  # anchor 4096 falls under the threshold
    assert run(H, "1", exact[None], "ref", 0.25, 1.0) == 4096
    H.poll_status()
    v8 = exact.copy()
    v8[4] = 0.01  # class 0 in V8_NATIVE reading
    run(H, "1", v8[None], "ultra", 0.25, 0.45, max_det=4096)
    H.poll_status()
    H.postprocess(_dev(h[None]), _metas(1), 0.25, 1.0, layout=N.HEAD_CHANNEL_MAJOR)
    with pytest.raises(N.B200VAError) as e:
        H.poll_status()
    assert e.value.status == N.ERR_CAPACITY
    H.poll_status()


def test_every_decode_kernel_ran():
    """The cases above reached all five decode kernels (recorded with torch.profiler)."""
    assert SEEN == set(KERNELS), sorted(SEEN)
