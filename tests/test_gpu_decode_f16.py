"""float16 heads (B200VA_HEAD_F16): every fp16 decode kernel against the same call on ``head.float()`` and against the
NumPy decode on ``head.astype(np.float32)``, at the shapes and scores of test_gpu_decode.py plus the fp16 edges.

Four kernels read an fp16 head in place: k_decode16_cm_split (small batches, 16-96 class rows), k_decode16_cm<8>
(A % 8 == 0, 16-byte aligned base), k_decode16_cm<1> (every other channel-major head) and k_decode16_am.  There is
no fp16 ring: B200VA_DECODE_IMPL=2 selects the register kernels.  One handle per B200VA_DECODE_IMPL value, the kernel
that ran is recorded with torch.profiler, and the last test asserts that all four ran.  Widening is exact, so every
output is compared bit for bit: classes exactly, confidences and boxes as float32 bit patterns."""

import os
import re

import numpy as np
import pytest

import test_gpu_decode as D
from oracle import hotpath as O
from oracle import ultralytics_restate as U

REPO = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
KERNELS16 = ("k_decode16_cm_split", "k_decode16_cm<8>", "k_decode16_cm<1>", "k_decode16_am")
SEEN16 = set()
gpu = pytest.mark.gpu


def test_header_define_matches_python():
    """B200VA_HEAD_F16 in include/b200va.h is _native.HEAD_F16."""
    from realtime_video_analytics_32streams_b200 import _native as N

    text = open(os.path.join(REPO, "include", "b200va.h")).read()
    m = re.search(r"#define\s+B200VA_HEAD_F16\s+(0x[0-9a-fA-F]+|\d+)", text)
    assert m and int(m.group(1), 0) == N.HEAD_F16 == 0x200


@pytest.fixture(scope="module")
def HS():
    """B200VA_DECODE_IMPL -> handle (the knob is read when the handle is created)."""
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


# ---- running and comparing ---------------------------------------------------------------------------------------

def _dev16(a, offset=False):
    """CUDA float16 copy of `a`; offset=True: a contiguous view one half into a larger buffer (2 bytes past a 16-byte
    boundary)."""
    import torch

    t = torch.from_numpy(np.ascontiguousarray(a, dtype=np.float16)).cuda()
    if not offset:
        return t
    buf = torch.zeros(t.numel() + 1, dtype=torch.float16, device="cuda")
    buf[1:].copy_(t.view(-1))
    v = buf[1:].view(t.shape)
    assert v.is_contiguous() and v.data_ptr() % 16 == 2
    return v


def expected16(impl, layout, C, A, mode, frames, offset=False):
    """The host's fp16 dispatch rule (postprocess_impl), restated."""
    if layout == "am":
        return "k_decode16_am"
    n_cls = C - D._cls0(C, "v8" if mode == "ultra" else mode)
    if A % 4 == 0 and not offset and 16 <= n_cls <= 96 and (impl == "3" or (impl == "0" and frames <= 8)):
        return "k_decode16_cm_split"
    return "k_decode16_cm<8>" if A % 8 == 0 and not offset else "k_decode16_cm<1>"


def _profiled16(fn, expect):
    """Run fn; with `expect`, assert that it launched `expect` (a second launch group may pick another fp16 kernel)
    and no float32 decode kernel."""
    if expect is None:
        return fn()
    import torch
    from torch.profiler import ProfilerActivity, profile

    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        out = fn()
        torch.cuda.synchronize()
    names = {e.name for e in prof.events() if "k_decode" in e.name}
    ran = {k for k in KERNELS16 if any(k in n for n in names)}
    SEEN16.update(ran)
    assert expect in ran, (expect, sorted(names))
    assert not any(k in n for k in D.KERNELS for n in names), sorted(names)  # no float32 decode kernel
    return out


def _same_tables(a, b, B):
    """Two detection tables agree bit for bit on every frame's rows."""
    ca, cb = a["count"][:B].cpu().numpy(), b["count"][:B].cpu().numpy()
    assert np.array_equal(ca, cb), (ca, cb)
    for f in range(B):
        n = int(ca[f])
        assert np.array_equal(a["cls"][f, :n].cpu().numpy(), b["cls"][f, :n].cpu().numpy()), f
        assert D._same_bits(a["conf"][f, :n].cpu().numpy(), b["conf"][f, :n].cpu().numpy()), f
        assert D._same_bits(a["bbox_xyxy"][f, :n].cpu().numpy(), b["bbox_xyxy"][f, :n].cpu().numpy()), f


def run16(H, impl, heads, mode, conf, iou, layout="cm", offset=False, profile=True, classes=None, aware=False,
          filt=None, max_det=300, skip=()):
    """heads [B, C, A] (channel-major, any float dtype) are rounded to float16 and sent as `layout`.  The fp16 call
    must equal the same call on head.float() and, frame by frame, the NumPy decode of the widened head.  Returns
    (detections, the fp16 output table)."""
    from realtime_video_analytics_32streams_b200 import _native as N

    h16 = np.asarray(heads).astype(np.float16)
    h32 = h16.astype(np.float32)
    B, C, A = h16.shape
    host = h16 if layout == "cm" else h16.transpose(0, 2, 1)
    dev = _dev16(host, offset)
    lay = N.HEAD_CHANNEL_MAJOR if layout == "cm" else N.HEAD_ANCHOR_MAJOR
    if mode == "ultra":
        fhw = D._frame_hw(B)
        call = lambda d: H.postprocess_ultralytics(d, fhw, D.IN_HW, conf_thr=conf, iou_thr=iou, classes=classes,
                                                   agnostic=not aware, max_det=max_det, layout=lay, filter_conf=filt)
    else:
        metas = D._metas(B)
        call = lambda d: H.postprocess(d, metas, conf, iou, classes=classes, layout=lay, filter_conf=filt,
                                       score_mode=N.SCORE_V8_NATIVE if mode == "v8" else N.SCORE_REF_COMPAT,
                                       nms_mode=N.NMS_CLASS_AWARE if aware else N.NMS_AGNOSTIC)
    expect = expected16(impl, layout, C, A, mode, min(B, 64), offset) if profile else None
    out = _profiled16(lambda: call(dev), expect)
    _same_tables(out, call(dev.float()), B)
    total = 0
    with np.errstate(invalid="ignore", over="ignore"):
        for b in range(B):
            if b in skip:
                assert int(out["count"][b].item()) == 0, b
                continue
            if mode == "ultra":
                want = U.postprocess(h32[b], D.IN_HW, fhw[b], conf, iou, classes, not aware, max_det)
                if filt is not None:
                    want = [w for w in want if w[1] >= filt]
                cls, sc, box = [c for c, _, _ in want], [s for _, s, _ in want], [bx for _, _, bx in want]
            else:
                ref = O.postprocess(h32[b], metas[b].as_meta(), conf, iou, classes, v8_native=mode == "v8",
                                    class_aware=aware, layout="cm")
                if filt is not None:
                    ref = O.filter_detections(ref, filt)
                cls, sc, box = [d.class_id for d in ref], [d.confidence for d in ref], [d.bbox_xyxy for d in ref]
            total += D._check_frame(out, b, cls, sc, box, ("f16", mode, layout, conf, iou))
    return total, out


# ---- shapes and argmax -------------------------------------------------------------------------------------------

# (anchors, channels): 1..8400 anchors (2100, 3549 and 7581 are not multiples of 8 or 4), 15 / 16 / 17 / 79 / 96 / 97
# class rows around the split limits (REF_COMPAT; one more each in V8_NATIVE)
SHAPES16 = [(1, 5), (3, 6), (5, 20), (256, 20), (127, 21), (128, 21), (132, 22), (2100, 84), (3549, 85), (7581, 101),
            (8400, 101), (8400, 102)]


@gpu
@pytest.mark.parametrize("A,C", SHAPES16)
def test_f16_shapes_and_argmax(HS, A, C):
    """Every variant, both layouts, REF_COMPAT / V8_NATIVE / Ultralytics, 2 and 3 frames, duplicated maxima a split
    part / 32 lanes apart, and a head base one half into its buffer."""
    n_cand = min(A, 150)
    for mode in ("ref", "v8", "ultra"):
        heads = np.stack([D.make_head(3000 * A + C + 7 * f + {"ref": 0, "v8": 1, "ultra": 2}[mode], C, A, n_cand,
                                      "v8" if mode == "ultra" else mode) for f in range(3 if A > 1000 else 2)])
        for impl in ("0", "1", "2", "3"):
            for iou in (1.0, 0.5):
                run16(HS[impl], impl, heads, mode, 0.25, iou, profile=iou == 1.0)
        run16(HS["0"], "0", heads, mode, 0.25, 1.0, layout="am")
        for impl in ("0", "3"):
            run16(HS[impl], impl, heads, mode, 0.25, 1.0, offset=True)
        run16(HS["0"], "0", heads, mode, 0.25, 1.0, layout="am", offset=True)


@gpu
def test_f16_ties_and_wide_heads(HS):
    """Equal scores across anchors (multiples of 1/8, exact in fp16) under both tie rules; all rows equal; a head
    of 2101 / 2102 class rows with maxima around class 2048."""
    for A, C in ((3549, 85), (8400, 22), (128, 101)):
        for mode in ("ref", "v8", "ultra"):
            heads = np.stack([D.make_head(91 + A + f, C, A, 200, "v8" if mode == "ultra" else mode, ties=True)
                              for f in range(2)])
            for impl in ("0", "1", "3"):
                for iou in (1.0, 0.5):
                    run16(HS[impl], impl, heads, mode, 0.25, iou, profile=iou == 1.0)
            run16(HS["0"], "0", heads, mode, 0.25, 0.5, layout="am")
    for mode in ("ref", "v8", "ultra"):
        cls0 = D._cls0(85, "v8" if mode == "ultra" else mode)
        h = D.make_head(5, 85, 256, 0, "v8" if mode == "ultra" else mode)
        h[cls0:, :64] = np.float32(0.5)  # every class row equal: np.argmax takes row 0
        heads = h[None]
        for impl in ("0", "1", "3"):
            assert run16(HS[impl], impl, heads, mode, 0.25, 1.0)[0] >= 64
        wide = D._wide_head("v8" if mode == "ultra" else mode)
        for impl in ("0", "1"):
            assert run16(HS[impl], impl, wide, mode, 0.25, 1.0)[0] == 128
        run16(HS["0"], "0", wide, mode, 0.25, 1.0, layout="am")


# ---- non-finite, signed and subnormal values ---------------------------------------------------------------------

SUB = float(np.float16(2.0 ** -24))  # the smallest fp16 subnormal
# (objectness, class scores) rows beyond D.SPECIAL: fp16 subnormals, the fp16 maximum, products that leave fp16 range
SPECIAL16 = D.SPECIAL + [
    (1.0, [SUB, 0.0, 0.0, 0.0]),
    (1.0, [0.0, 3 * SUB, 2.0 ** -15, -SUB]),
    (1.0, [-SUB, -0.0, -2 * SUB, -SUB]),
    (2.0 ** -14, [2.0 ** -14, 1023 * SUB, 0.0, 0.0]),  # min normal x min normal: a float32 normal, not an fp16 one
    (1.0, [65504.0, 0.1, 65504.0, 0.2]),               # equal maxima at the fp16 maximum
    (65504.0, [65504.0, 0.5, 0.25, 0.1]),              # 65504^2 is finite in float32
    (-65504.0, [0.5, 65504.0, 0.0, 0.25]),
    (SUB, [SUB, 0.5, 0.0, 0.0]),                       # products 2^-48 and 2^-25: float32 normals, fp16 would not hold them
]
FP16_BOX = {1e30: 65504.0, -1e30: -65504.0}  # the float32 box edits of D.BOX_EDITS, within fp16 range


def special16_head(seed, A, mode):
    rng = np.random.default_rng(seed)
    h = D.make_head(seed, 9, A, 0, mode)
    h[4] = 1.0 if mode == "ref" else 0.05
    k = len(SPECIAL16)
    for a, (obj, sc) in enumerate(SPECIAL16):
        h[4, a] = obj
        h[5:, a] = sc
    s = D._unique(rng, A - k, 0.3, 0.99)
    for j, a in enumerate(range(k, A)):
        h[5 + j % 4, a] = s[j]
    for j, edits in enumerate(D.BOX_EDITS):
        for col, v in edits:
            h[col, k + 3 * j] = FP16_BOX.get(v, v)
    return h


@gpu
@pytest.mark.parametrize("conf", [0.25, 0.0, -0.25, -0.0, SUB, 2.0 ** -25, -1.0])
def test_f16_nonfinite_signed_subnormal(HS, conf):
    """NaN, 0 x inf, +-inf, +-0, fp16 subnormals (widened to their exact nonzero float32 values), 65504, and box rows
    holding +-inf, NaN and +-65504."""
    import torch

    for A in (136, 37):
        for mode in ("ref", "v8", "ultra"):
            heads = np.stack([special16_head(17 + A + f, max(A, 64), "ref" if mode == "ref" else "v8")[:, :A]
                              for f in range(2)])
            for impl in ("0", "1", "3"):
                for iou in (1.0, 0.5):
                    _, out = run16(HS[impl], impl, heads, mode, conf, iou, profile=iou == 1.0 and conf == 0.25)
                    if mode == "ref" and conf in (0.0, -0.25, -1.0) and iou == 1.0:
                        # anchors 22 and 23 score the fp16 subnormals 2^-24 and 2^-15: emitted as those float32 values
                        n = int(out["count"][0].item())
                        confs = out["conf"][0, :n].cpu().numpy()
                        assert np.any(confs == np.float32(2.0 ** -24)) and np.any(confs == np.float32(2.0 ** -15)), confs
            run16(HS["0"], "0", heads, mode, conf, 1.0, layout="am", profile=conf == 0.25)
    # a subnormal survives the widening on its own: the float32 value of fp16 0x0001
    assert torch.tensor([SUB], dtype=torch.float16).float().item() == 2.0 ** -24


@gpu
@pytest.mark.parametrize("thr", [0.25, 0.45, 0.1, float(np.float16(0.45))])
def test_f16_threshold_edges(HS, thr):
    """Scores one fp16 ulp either side of fp16(thr) and at it; the threshold float32(thr) may lie between two fp16
    values.  `>=` in the reference modes, `>` for Ultralytics, and the float64 filter_conf fold."""
    t = np.float16(thr)
    edge = [np.nextafter(t, np.float16(0)), t, np.nextafter(t, np.float16(1))]
    A, C = 256, 22
    for mode in ("ref", "v8", "ultra"):
        h = D.make_head(int(thr * 1000) + 3, C, A, 0, "ref" if mode == "ref" else "v8")
        h[4:] = np.minimum(h[4:], np.float32(0.05))
        if mode == "ref":
            h[4] = 1.0
        for a in range(90):
            h[5 + a % 17, a] = np.float32(edge[a % 3])
        heads = h[None]
        for impl in ("0", "1", "3"):
            for filt in (None, thr):
                assert run16(HS[impl], impl, heads, mode, thr, 1.0, filt=filt)[0] > 0
        run16(HS["0"], "0", heads, mode, thr, 1.0, layout="am", filt=thr)


# ---- whitelist, class-aware NMS, launch groups, gating -----------------------------------------------------------

@gpu
def test_f16_whitelist_and_class_aware(HS):
    for mode in ("ref", "v8", "ultra"):
        heads = np.stack([D.make_head(41 + f, 85, 3552, 150, "ref" if mode == "ref" else "v8") for f in range(2)])
        for impl in ("0", "1", "3"):
            for classes in ([], [-1, 3, 3, 500, 7], [79, 80, 81], [0, 0]):
                run16(HS[impl], impl, heads, mode, 0.25, 1.0, classes=classes)
            run16(HS[impl], impl, heads, mode, 0.25, 0.5, aware=True, filt=0.6, profile=False)
        run16(HS["0"], "0", heads, mode, 0.25, 0.5, layout="am", classes=[-1, 3, 3, 500, 7], aware=True)


@gpu
@pytest.mark.parametrize("B", [65, 128])
def test_f16_launch_groups(HS, B):
    """Launch groups of 64 offset the fp16 head by base * C * A halves."""
    for impl, (C, A) in (("0", (22, 3549)), ("2", (85, 1024)), ("1", (85, 1000))):
        heads = D._batch_heads(B, C, A, 300 * B + int(impl))
        for iou in (0.5, 1.0):
            run16(HS[impl], impl, heads, "ref", 0.25, iou, profile=iou == 1.0)
        run16(HS[impl], impl, heads, "ref", 0.25, 0.5, aware=True, filt=0.6, profile=False)
        run16(HS[impl], impl, D._batch_heads(B, C, A, 11 * B + int(impl), "ultra"), "ultra", 0.25, 0.45)
    run16(HS["0"], "0", D._batch_heads(B, 85, 300, 5), "ref", 0.25, 0.5, layout="am")


@gpu
@pytest.mark.parametrize("B", [65, 128])
def test_f16_launch_groups_skip_mask(HS, B):
    import torch

    gated = {b for b in (0, 5, 63, 64, 100, 127) if b < B}
    mask = torch.zeros(B, dtype=torch.uint8, device="cuda")
    mask[sorted(gated)] = 1
    for impl, (C, A) in (("0", (22, 3549)), ("1", (85, 1024)), ("3", (22, 1024))):
        heads = D._batch_heads(B, C, A, 13 + int(impl))
        H = HS[impl]
        H.set_skip_mask(mask)
        try:
            run16(H, impl, heads, "ref", 0.25, 0.5, skip=gated)
            run16(H, impl, D._batch_heads(B, C, A, 19, "ultra"), "ultra", 0.25, 0.45, skip=gated)
            run16(H, impl, heads[:8], "ref", 0.25, 0.5, skip={b for b in gated if b < 8})
            run16(H, "0", heads, "ref", 0.25, 0.5, layout="am", skip=gated)
        finally:
            H.set_skip_mask(None)


@gpu
def test_f16_layout_with_unknown_bit_is_refused(HS):
    import torch
    from realtime_video_analytics_32streams_b200 import _native as N

    H = HS["0"]
    head = torch.zeros((1, 84, 256), dtype=torch.float16, device="cuda")
    for layout in (0x400, 0x100, N.HEAD_F16 | 2, 0x1000 | N.HEAD_ANCHOR_MAJOR):
        with pytest.raises(N.B200VAError) as e:
            H.postprocess(head, D._metas(1), 0.25, 0.5, layout=layout)
        assert e.value.status == N.ERR_INVALID
    with pytest.raises(ValueError):
        H.postprocess(head.to(torch.bfloat16), D._metas(1), 0.25, 0.5)


# ---- b200va_tick, the engine, _as_head ---------------------------------------------------------------------------

TB, THW, TCONF, TIOU, TTRK = 6, (540, 960), 0.35, 0.5, (30, 1, 0.5)


def _tick_run(head_dtype, heads16, frames, schedule, graph):
    """Ticks of `schedule` on a fresh handle with the heads as `head_dtype`, eager or replayed from CUDA graphs;
    snapshots of (dets, tracks) after every call (schedule 4 fills tick k's tables in call k + 1)."""
    import torch
    from realtime_video_analytics_32streams_b200 import _native as N

    h = N.Handle(device=0, max_batch=8, max_anchors=8400, max_candidates=2048, max_dets=512, max_streams=8,
                 max_tracks=512)
    try:
        net = torch.empty((TB, 3, *D.IN_HW), dtype=torch.float32, device="cuda")
        metas = [N.letterbox_meta(*THW, *D.IN_HW) for _ in range(TB)]
        dev = [torch.empty((*THW, 3), dtype=torch.uint8, device="cuda") for _ in range(TB)]
        head = torch.empty(heads16[0].shape, dtype=head_dtype, device="cuda")
        plan = h.plan_tick(frames=dev, net_out=net, dst_hw=D.IN_HW, head=head, metas=metas, conf_thr=TCONF,
                           iou_thr=TIOU, filter_conf=TCONF, slots=list(range(TB)), tracker_cfg=TTRK, schedule=schedule)

        def load(t):
            for s in range(TB):
                dev[s].copy_(torch.from_numpy(frames[t][s]))
            head.copy_(torch.from_numpy(heads16[t]).to(head_dtype))

        graphs, start = [], 0
        if graph:
            if schedule == 4:  # prime the pipeline (tick 0 decodes only) so that the captured calls launch a chain
                load(0)
                h.tick(plan)
                torch.cuda.synchronize()
                start = 1
            side = torch.cuda.Stream()
            side.wait_stream(torch.cuda.current_stream())
            with torch.cuda.stream(side):
                for _ in range(2 if schedule == 4 else 1):  # schedule 4 alternates two candidate sets
                    gr = torch.cuda.CUDAGraph()
                    with torch.cuda.graph(gr, stream=side):
                        h.tick(plan)
                    graphs.append(gr)
            torch.cuda.current_stream().wait_stream(side)
            torch.cuda.synchronize()
            if schedule != 4:  # the capture ran nothing; start from clean tracker state anyway
                for s in range(TB):
                    h.tracker_reset(s)
                h.tracker_set_next_id(1)
        snaps = []
        for t in range(start, len(heads16)):
            load(t)
            if graph:
                graphs[(t - start) % len(graphs)].replay()
            else:
                h.tick(plan)
            torch.cuda.synchronize()
            snaps.append(({k: v.clone() for k, v in plan.dets.items() if not k.startswith("_")},
                          {k: v.clone() for k, v in plan.tracks.items() if not k.startswith("_")}))
        h.poll_status()
        return snaps
    finally:
        h.close()


@gpu
@pytest.mark.parametrize("graph", [False, True])
@pytest.mark.parametrize("schedule", [1, 3, 4, 6])
def test_f16_tick_equals_float_tick(schedule, graph):
    """b200va_tick with an fp16 head gives the tables of the same tick on head.float()."""
    import torch
    from realtime_video_analytics_32streams_b200 import synth

    n_ticks = 4
    frames = [[synth.synth_frame(500 + 10 * t + s, *THW) for s in range(TB)] for t in range(n_ticks)]
    heads16 = [np.stack([synth.synth_head(800 + 10 * t + s, 84, 8400, 14, dup=3) for s in range(TB)]).astype(np.float16)
               for t in range(n_ticks)]
    a = _tick_run(torch.float16, heads16, frames, schedule, graph)
    b = _tick_run(torch.float32, heads16, frames, schedule, graph)
    total = 0
    for (da, ta), (db, tb) in zip(a, b):
        _same_tables(da, db, TB)
        total += int(da["count"].sum().item())
        assert np.array_equal(ta["count"].cpu().numpy(), tb["count"].cpu().numpy())
        for k in ("track_id", "cls", "age", "hits"):
            assert np.array_equal(ta[k].cpu().numpy(), tb[k].cpu().numpy()), k
        for k in ("conf", "bbox_xyxy"):
            for s in range(TB):
                n = int(ta["count"][s].item())
                assert D._same_bits(ta[k][s, :n].cpu().numpy(), tb[k][s, :n].cpu().numpy()), (k, s)
    assert total > 0


@gpu
@pytest.mark.parametrize("device_gates", [False, True])
def test_f16_engine_half_equals_float_engine(device_gates):
    """A HotPathEngine with `half: true` whose infer returns fp16 gives the results of one whose infer returns the
    same head as float32; the fp16 head reaches the decode without a conversion."""
    import torch
    from realtime_video_analytics_32streams_b200 import (DetectorConfig, HotPathEngine, StreamConfig, TrackerConfig,
                                                          _native, synth)

    names = [f"cam{i}" for i in range(4)]
    n_ticks = 3
    frames = [[synth.synth_frame(60 + 10 * t + s, *THW) for s in range(4)] for t in range(n_ticks)]
    heads = [torch.from_numpy(np.stack([synth.synth_head(90 + 10 * t + s, 84, 8400, 12, dup=2) for s in range(4)])
                              .astype(np.float16)).cuda() for t in range(n_ticks)]
    results = {}
    for dt in (torch.float16, torch.float32):
        h = _native.Handle(device=0, max_batch=8, max_anchors=8400, max_candidates=2048, max_dets=512, max_streams=8,
                           max_tracks=512)
        seen = []
        box = {}

        def infer(tensor, dt=dt, seen=seen, box=box):
            assert tensor.dtype == torch.float16  # half: true letterboxes into fp16
            head = heads[box["t"]][: tensor.shape[0]].to(dt)
            seen.append(head)
            return head

        eng = HotPathEngine([StreamConfig(name=n) for n in names],
                            DetectorConfig(confidence_threshold=0.3, iou_threshold=0.5, half=True),
                            TrackerConfig(max_age=30, max_iou_distance=0.5, min_hits=1), infer=infer, handle=h,
                            input_hw=(640, 640), device_gates=device_gates)
        out = []
        try:
            for t in range(n_ticks):
                box["t"] = t
                for r in eng.tick(frames[t]):
                    out.append((r.stream_name, r.n_detections, {k: v.copy() for k, v in r.detection_arrays.items()},
                                {k: v.copy() for k, v in r.track_arrays.items()}))
            h.poll_status()
        finally:
            h.close()
        assert all(x.dtype == dt for x in seen)
        results[dt] = out
    a, b = results[torch.float16], results[torch.float32]
    assert len(a) == len(b) and sum(r[1] for r in a) > 0
    for ra, rb in zip(a, b):
        assert ra[:2] == rb[:2]
        for da, db in ((ra[2], rb[2]), (ra[3], rb[3])):
            for k in da:
                assert np.array_equal(da[k].view(np.uint8), db[k].view(np.uint8)), (ra[0], k)


@gpu
def test_f16_as_head_keeps_fp16():
    """_as_head: an fp16 CUDA tensor is returned as is (same data_ptr), a host np.float16 array is uploaded as fp16,
    every other dtype becomes float32."""
    import torch
    from realtime_video_analytics_32streams_b200 import B200Detector, DetectorConfig, _native

    h = _native.Handle(device=0, max_batch=4, max_anchors=8400, max_candidates=1024, max_dets=256, max_streams=2,
                       max_tracks=64)
    try:
        det = B200Detector(DetectorConfig(half=True), handle=h)
        x = torch.randn(2, 84, 512, device="cuda").half()
        y = det._as_head(x)
        assert y.dtype == torch.float16 and y.data_ptr() == x.data_ptr()
        assert det._as_head([x, None]).data_ptr() == x.data_ptr()
        z = det._as_head(x.cpu().numpy())
        assert z.is_cuda and z.dtype == torch.float16 and torch.equal(z, x)
        w = det._as_head(x.transpose(1, 2))  # not contiguous: an fp16 copy
        assert w.dtype == torch.float16 and w.is_contiguous() and torch.equal(w, x.transpose(1, 2))
        for other in (x.to(torch.bfloat16), x.double(), x.cpu().numpy().astype(np.float64)):
            assert det._as_head(other).dtype == torch.float32
    finally:
        h.close()


@gpu
def test_f16_every_decode_kernel_ran():
    """The cases above reached all four fp16 decode kernels (recorded with torch.profiler)."""
    assert SEEN16 == set(KERNELS16), sorted(SEEN16)
