"""The Ultralytics backend on the batched path: ``b200va_preprocess_geom_nv12``, the geometry-aware sparse uploads,
``b200va_tick_ultralytics`` and ``HotPathEngine`` / ``TickCollector`` in Ultralytics mode.

Every batched result must equal what the per-stream path gives: ``B200UltralyticsDetector.predict`` ->
``filter_detections`` -> ``B200IouTracker.update`` in stream order (the same detections bit for bit, the same tracks
and track ids, the same skip decisions), and NV12 results those of ``cv2.cvtColor(frame, COLOR_YUV2BGR_NV12)``."""
import asyncio
import ctypes as C
import os
import types

import numpy as np
import pytest

import nv12_restate as cvr
from oracle import hotpath as O
from oracle import ultralytics_restate as U
from realtime_video_analytics_32streams_b200 import synth

pytestmark = pytest.mark.gpu

IN = (640, 640)
CONF, IOU = 0.35, 0.5
FMTS = ("f32", "f16", "u8_nchw", "u8_nhwc")


def _N():
    from realtime_video_analytics_32streams_b200 import _native

    return _native


def _handle(max_batch=16, dense=False):
    if dense:  # every launch takes the dense-scene kernels (read when the handle is created)
        os.environ["B200VA_DENSE_IMPL"] = "2"
    try:
        return _N().Handle(device=0, max_batch=max_batch, max_anchors=8400, max_candidates=4096, max_dets=1024,
                           max_streams=16, max_tracks=2048 if dense else 256)
    finally:
        os.environ.pop("B200VA_DENSE_IMPL", None)


def _fmt(name):
    N = _N()
    return {"f32": N.OUT_F32_RGB_NCHW, "f16": N.OUT_F16_RGB_NCHW, "u8_nchw": N.OUT_U8_BGR_NCHW, "u8_nhwc": N.OUT_U8_BGR_NHWC}[name]


def _cu(a):
    import torch

    return torch.from_numpy(np.ascontiguousarray(a)).cuda()


def _nv12(seed, h, w):
    return np.random.default_rng(seed).integers(0, 256, size=(h * 3 // 2, w), dtype=np.uint8)


def _same(a, b):
    a, b = np.ascontiguousarray(a), np.ascontiguousarray(b)
    return a.shape == b.shape and np.array_equal(a.view(np.uint8), b.view(np.uint8))


def _anchors(in_hw):
    return sum((in_hw[0] // s) * (in_hw[1] // s) for s in (8, 16, 32))


def _head(seed, in_hw, n_obj=12, dup=4, nc=80, ties=False, t=0):
    """Decoded YOLOv8 head [4 + nc, A] for an `in_hw` input: objects fixed by `seed`, jittered by `t` (tracks persist)."""
    A = _anchors(in_hw)
    rng, jit = np.random.default_rng(seed), np.random.default_rng(seed * 1000 + t)
    h = np.empty((4 + nc, A), dtype=np.float32)
    h[0], h[1] = jit.uniform(0, in_hw[1], A), jit.uniform(0, in_hw[0], A)
    h[2], h[3] = jit.uniform(4, 60, A), jit.uniform(4, 60, A)
    h[4:] = jit.uniform(0, 0.05, (nc, A))
    pick = jit.permutation(A)[:n_obj * dup]
    for o in range(n_obj):
        cx, cy = rng.uniform(40, in_hw[1] - 40) + 2 * t, rng.uniform(40, in_hw[0] - 40)
        w, hh, c = rng.uniform(20, 120), rng.uniform(20, 120), int(rng.integers(0, nc))
        for d in range(dup):
            a = pick[o * dup + d]
            h[:4, a] = (cx + jit.normal(0, 1.5), cy + jit.normal(0, 1.5), w + jit.normal(0, 1.5), hh + jit.normal(0, 1.5))
            s = jit.uniform(0.3, 1.0)
            h[4 + c, a] = np.round(s * 8) / 8 if ties else s
    return h


# ---- b200va_preprocess_geom_nv12 -----------------------------------------------------------------------------------
# the shapes of test_gpu_ultralytics.py::test_preprocess_geom_matches_letterbox_restatement, odd sizes made even
GEOM_SHAPES = [(1080, 1920), (2160, 3840), (720, 1280), (1082, 1920), (360, 640), (1920, 1080), (722, 1000), (480, 854)]


@pytest.mark.parametrize("auto", [False, True])
def test_preprocess_geom_nv12_matches_bgr_on_converted_frames(auto):
    N = _N()
    h = _handle()
    try:
        for i, (fh, fw) in enumerate(GEOM_SHAPES):
            nv = _nv12(40 + i, fh, fw)
            bgr = cvr.nv12_to_bgr(nv)
            m, oh, ow = N.letterbox_meta_ultralytics(fh, fw, *IN, auto, 32)
            mask = h.roi_rasterize(synth.synth_polygons(60 + i, fh, fw), fh, fw) if i % 2 else None
            for name in FMTS:
                got = h.preprocess_geom([_cu(nv)], [m], (oh, ow), _fmt(name), [mask])
                want = h.preprocess_geom([_cu(bgr)], [m], (oh, ow), _fmt(name), [mask])
                assert _same(got.cpu().numpy(), want.cpu().numpy()), (fh, fw, auto, name)
                if name in ("f32", "f16") and mask is None:  # and the LetterBox restatement
                    ref, _ = U.preprocess(bgr, IN, auto=auto, stride=32, half=name == "f16")
                    assert _same(got.cpu().numpy(), ref), (fh, fw, auto, name)
                # B200VA_OUT_FLAG_PADS_VALID: pad rows left as an earlier call of the same geometry wrote them
                other = _nv12(90 + i, fh, fw)
                h.preprocess_geom([_cu(other)], [m], (oh, ow), _fmt(name) | N.OUT_FLAG_PADS_VALID, [mask], out=got)
                fresh = h.preprocess_geom([_cu(other)], [m], (oh, ow), _fmt(name), [mask])
                assert _same(got.cpu().numpy(), fresh.cpu().numpy()), (fh, fw, auto, name)
        # several frames of several sizes in one call, as an Nv12Batch and as (y, uv) pairs
        frames = [_nv12(7 + k, *hw) for k, hw in enumerate(GEOM_SHAPES[:4])]
        geoms = [N.letterbox_meta_ultralytics(*hw, *IN, False, 32)[0] for hw in GEOM_SHAPES[:4]]
        want = h.preprocess_geom([_cu(cvr.nv12_to_bgr(f)) for f in frames], geoms, IN, N.OUT_F32_RGB_NCHW)
        got = h.preprocess_geom(N.Nv12Batch([_cu(f) for f in frames]), geoms, IN, N.OUT_F32_RGB_NCHW)
        pairs = h.preprocess_geom([(_cu(f[:hw[0]]), _cu(f[hw[0]:])) for f, hw in zip(frames, GEOM_SHAPES)], geoms, IN)
        assert _same(got.cpu().numpy(), want.cpu().numpy()) and _same(pairs.cpu().numpy(), want.cpu().numpy())
    finally:
        h.close()


def test_preprocess_geom_nv12_refusals():
    import torch

    N = _N()
    h = _handle()
    try:
        out = torch.empty((1, 3, *IN), dtype=torch.float32, device="cuda")
        y = torch.zeros((1082, 1920), dtype=torch.uint8, device="cuda")
        uv = torch.zeros((541, 1920), dtype=torch.uint8, device="cuda")
        m = N.letterbox_meta_ultralytics(1082, 1920, *IN, False, 32)[0]

        def call(frame, hh, ww, geom=m, dst=IN):
            arr = (N.Nv12Frame * 1)(frame)
            return h.lib.b200va_preprocess_geom_nv12(h._h, arr, N._int_array([hh]), N._int_array([ww]), 1, None,
                                                     (N.Letterbox * 1)(geom), C.c_void_p(out.data_ptr()), dst[0], dst[1],
                                                     N.OUT_F32_RGB_NCHW, None)

        ok = N.Nv12Frame(y.data_ptr(), uv.data_ptr(), 1920, 1920)
        assert call(ok, 1082, 1920) == N.OK
        assert call(N.Nv12Frame(None, uv.data_ptr(), 1920, 1920), 1082, 1920) == N.ERR_INVALID  # NULL plane
        assert call(N.Nv12Frame(y.data_ptr(), None, 1920, 1920), 1082, 1920) == N.ERR_INVALID
        odd = N.letterbox_meta_ultralytics(1081, 1920, *IN, False, 32)[0]
        assert call(ok, 1081, 1920, geom=odd) == N.ERR_INVALID  # odd size
        assert call(ok, 1082, 1920, geom=odd) == N.ERR_INVALID  # geometry of another frame size
        assert call(ok, 1082, 1920, dst=(320, 640)) == N.ERR_INVALID  # does not fit the canvas
        assert call(N.Nv12Frame(y.data_ptr(), uv.data_ptr(), 1000, 1920), 1082, 1920) == N.ERR_INVALID  # pitch < width
        assert h.lib.b200va_preprocess_geom_nv12(h._h, None, N._int_array([1082]), N._int_array([1920]), 1, None,
                                                 (N.Letterbox * 1)(m), C.c_void_p(out.data_ptr()), 640, 640, 0, None) == N.ERR_INVALID
        with pytest.raises(ValueError):  # odd sizes never reach the library from Python
            h.preprocess_geom([torch.zeros((1623, 1921), dtype=torch.uint8, device="cuda")], [m], IN)
    finally:
        h.close()


# ---- geometry-aware sparse uploads ---------------------------------------------------------------------------------
def _tapped_rows(src_h, new_h):
    """Restates linear_tap (preprocess.cu): the source rows with a non-zero vertical weight."""
    need = np.zeros(src_h, bool)
    for d in range(new_h):
        fy = np.float32((d + 0.5) * (src_h / new_h) - 0.5)
        s = int(np.floor(fy))
        fy = np.float32(fy - np.float32(s))
        w0, w1 = int(np.rint((np.float32(1) - fy) * np.float32(2048))), int(np.rint(fy * np.float32(2048)))
        if w0:
            need[min(max(s, 0), src_h - 1)] = True
        if w1:
            need[min(max(s + 1, 0), src_h - 1)] = True
    return need


def _plane_rows(need):
    """Rows an upload copies for one plane: the needed ones, or every row when more than 80 % are needed."""
    n = int(need.sum())
    return n if n * 10 <= len(need) * 8 else len(need)


# (h, w): the Ultralytics new_h (rounded) differs from the reference new_h (truncated) at 640 x 640
BGR_SHAPES = [(1083, 1921), (1079, 1919), (1085, 1930)]
NV12_SHAPES = [(1078, 1918), (1084, 1928), (1082, 1920)]


@pytest.mark.parametrize("nv12", [False, True])
def test_sparse_upload_with_geometry_equals_full_upload(nv12):
    import torch

    N = _N()
    h = _handle()
    try:
        for i, (fh, fw) in enumerate(NV12_SHAPES if nv12 else BGR_SHAPES):
            m, oh, ow = N.letterbox_meta_ultralytics(fh, fw, *IN, True, 32)
            ref_new_h = N.letterbox_meta(fh, fw, *IN).new_h
            if (fh, fw) != (1082, 1920):
                assert m.new_h != ref_new_h
            host = torch.from_numpy(_nv12(500 + i, fh, fw) if nv12 else synth.synth_frame(500 + i, fh, fw)).pin_memory()
            shape = tuple(host.shape)
            full = torch.zeros(shape, dtype=torch.uint8, device="cuda")
            full.copy_(host)
            sparse = torch.zeros(shape, dtype=torch.uint8, device="cuda")
            if nv12:
                src = N.Nv12Frame(host.data_ptr(), host.data_ptr() + fh * fw, fw, fw)
                moved = h.upload_frames_nv12([src], [sparse], geoms=[m])
            else:
                moved = h.upload_frames([(host.data_ptr(), host.stride(0))], [sparse], geoms=[m])
            torch.cuda.synchronize()
            need = _tapped_rows(fh, m.new_h)
            if nv12:
                need_uv = np.zeros(fh // 2, bool)
                need_uv[np.flatnonzero(need) >> 1] = True
                assert moved == (_plane_rows(need) + _plane_rows(need_uv)) * fw, (fh, fw)
            else:
                assert moved == _plane_rows(need) * 3 * fw, (fh, fw)
            assert moved < host.numel()
            for fmt in (N.OUT_F32_RGB_NCHW, N.OUT_U8_BGR_NHWC):
                a = h.preprocess_geom([sparse], [m], (oh, ow), fmt)
                b = h.preprocess_geom([full], [m], (oh, ow), fmt)
                assert _same(a.cpu().numpy(), b.cpu().numpy()), (fh, fw, nv12)
    finally:
        h.close()


def test_reference_geometry_upload_skips_a_row_the_ultralytics_letterbox_reads():
    """1083 x 1921: LetterBox resizes to 361 rows, the reference geometry to 360; row 361 carries weight only in the
    former, so the rows_mode 1 upload for 640 x 640 leaves it out and the Ultralytics letterbox of that frame is wrong."""
    import torch

    N = _N()
    fh, fw = 1083, 1921
    m, oh, ow = N.letterbox_meta_ultralytics(fh, fw, *IN, True, 32)
    ultra, ref = _tapped_rows(fh, m.new_h), _tapped_rows(fh, N.letterbox_meta(fh, fw, *IN).new_h)
    assert ultra[361] and not ref[361]
    h = _handle()
    try:
        host = torch.from_numpy(synth.synth_frame(77, fh, fw)).pin_memory()
        old = torch.zeros((fh, fw, 3), dtype=torch.uint8, device="cuda")
        new = torch.zeros((fh, fw, 3), dtype=torch.uint8, device="cuda")
        h.upload_frames([(host.data_ptr(), host.stride(0))], [old], sparse_for=IN)
        h.upload_frames([(host.data_ptr(), host.stride(0))], [new], geoms=[m])
        torch.cuda.synchronize()
        assert not old[361].any() and torch.equal(new[361].cpu(), host[361])
        full = h.preprocess_geom([_cu(host.numpy())], [m], (oh, ow))
        assert _same(h.preprocess_geom([new], [m], (oh, ow)).cpu().numpy(), full.cpu().numpy())
        assert not _same(h.preprocess_geom([old], [m], (oh, ow)).cpu().numpy(), full.cpu().numpy())
    finally:
        h.close()


# ---- b200va_tick_ultralytics ----------------------------------------------------------------------------------------
TB, THW, TRK, NT = 6, (540, 960), (30, 1, 0.5), 5
CASES = {
    # name: (dense handle, head kwargs, post kwargs, skip mask)
    "sparse": (False, dict(), dict(agnostic=False, max_det=300), None),
    "ties_maxdet_agnostic": (False, dict(ties=True, n_obj=30), dict(agnostic=True, max_det=7), None),
    "dense": (True, dict(n_obj=300, dup=6, nc=10), dict(agnostic=False, max_det=1000), None),
    "skip": (False, dict(), dict(agnostic=False, max_det=300), [0, 1, 0, 0, 1, 0]),
}


def _track_rows(tracks, n=TB):
    out = []
    for s in range(n):
        k = int(tracks["count"][s].item())
        out.append(list(zip(tracks["track_id"][s, :k].cpu().tolist(), tracks["cls"][s, :k].cpu().tolist(),
                            tracks["age"][s, :k].cpu().tolist(), tracks["hits"][s, :k].cpu().tolist(),
                            [tuple(b) for b in tracks["bbox_xyxy"][s, :k].cpu().tolist()])))
    return out


def _det_rows(dets, n=TB):
    out = []
    for s in range(n):
        k = int(dets["count"][s].item())
        out.append((dets["cls"][s, :k].cpu().numpy().copy(), dets["conf"][s, :k].cpu().numpy().copy(),
                    dets["bbox_xyxy"][s, :k].cpu().numpy().copy()))
    return out


def _tick_inputs(case):
    _, hk, _, _ = CASES[case]
    N = _N()
    m, oh, ow = N.letterbox_meta_ultralytics(*THW, *IN, True, 32)
    frames = [[_nv12(900 + 10 * t + s, *THW) for s in range(TB)] for t in range(NT)]
    heads = [np.stack([_head(40 + s, (oh, ow), t=t, **hk) for s in range(TB)]) for t in range(NT)]
    return m, (oh, ow), frames, heads


def _run_ticks(case, schedule, graph, nv12):
    """Network inputs, detections and track rows of every tick of b200va_tick_ultralytics (schedule 4: tables lag one
    call; drained at the end).  Graph mode: one eager call, then one graph per plan, replayed alternately."""
    import torch

    N = _N()
    dense, _, pk, skip = CASES[case]
    m, in_hw, frames, heads = _tick_inputs(case)
    h = _handle(max_batch=8, dense=dense)
    h.tracker_set_next_id(1)
    skip_dev = torch.tensor(skip, dtype=torch.uint8, device="cuda") if skip else None
    if skip_dev is not None:
        h.set_skip_mask(skip_dev)
    net = torch.zeros((TB, 3, *in_hw), dtype=torch.float32, device="cuda")
    shape = (THW[0] * 3 // 2, THW[1]) if nv12 else (*THW, 3)
    dev = [torch.zeros(shape, dtype=torch.uint8, device="cuda") for _ in range(TB)]
    head = torch.zeros((TB, *heads[0].shape[1:]), dtype=torch.float32, device="cuda")
    dets = [h.alloc_dets(TB) for _ in range(2)]
    tracks = [h.alloc_tracks(TB) for _ in range(2)]
    ultra = dict(geoms=[m] * TB, frame_hw=[THW] * TB, in_hw=in_hw, **pk)
    plans = [h.plan_tick(frames=dev, net_out=net, dst_hw=in_hw, head=head, conf_thr=CONF, iou_thr=IOU, filter_conf=CONF,
                         dets=dets[k], slots=list(range(TB)), tracker_cfg=TRK, schedule=schedule, tracks=tracks[k],
                         ultralytics=ultra) for k in range(2)]
    graphs = None
    nets, rows = [], []

    def load(t):
        for s in range(TB):
            dev[s].copy_(torch.from_numpy(frames[t][s] if nv12 else cvr.nv12_to_bgr(frames[t][s])))
        head.copy_(torch.from_numpy(heads[t]))

    def read(k):
        return _det_rows(dets[k]), _track_rows(tracks[k])

    for t in range(NT):
        load(t)
        if graph and graphs is None:
            h.tick(plans[t % 2])
            torch.cuda.synchronize()
            side = torch.cuda.Stream()
            side.wait_stream(torch.cuda.current_stream())
            graphs = []
            with torch.cuda.stream(side):
                for k in range(2):
                    g = torch.cuda.CUDAGraph()
                    with torch.cuda.graph(g, stream=side):
                        h.tick(plans[(t + 1 + k) % 2])
                    graphs.append(g)
            torch.cuda.current_stream().wait_stream(side)
            torch.cuda.synchronize()
        elif graph:
            graphs[(t - 1) % 2].replay()
        else:
            h.tick(plans[t % 2])
        torch.cuda.synchronize()
        nets.append(net.cpu().numpy().copy())
        if schedule != N.SCHEDULE_SOFTWARE_PIPELINED:
            rows.append(read(t % 2))
        elif t > 0:
            rows.append(read((t - 1) % 2))
    if schedule == N.SCHEDULE_SOFTWARE_PIPELINED:
        h.tick(h.plan_tick(schedule=schedule))
        torch.cuda.synchronize()
        rows.append(read((NT - 1) % 2))
    h.set_skip_mask(None)
    h.poll_status()
    h.close()
    return nets, rows


def _run_separate(case, nv12):
    """The same ticks as preprocess_geom* + postprocess_ultralytics + tracker_update, called one after another."""
    import torch

    dense, _, pk, skip = CASES[case]
    m, in_hw, frames, heads = _tick_inputs(case)
    h = _handle(max_batch=8, dense=dense)
    h.tracker_set_next_id(1)
    skip_dev = torch.tensor(skip, dtype=torch.uint8, device="cuda") if skip else None
    h.set_skip_mask(skip_dev)
    net = torch.zeros((TB, 3, *in_hw), dtype=torch.float32, device="cuda")
    nets, rows = [], []
    for t in range(NT):
        dev = [_cu(f if nv12 else cvr.nv12_to_bgr(f)) for f in frames[t]]
        h.preprocess_geom(dev, [m] * TB, in_hw, out=net)
        dets = h.postprocess_ultralytics(_cu(heads[t]), [THW] * TB, in_hw, CONF, IOU, filter_conf=CONF, **pk)
        tracks = h.tracker_update(list(range(TB)), dets, *TRK)
        torch.cuda.synchronize()
        nets.append(net.cpu().numpy().copy())
        rows.append((_det_rows(dets), _track_rows(tracks)))
    h.set_skip_mask(None)
    h.poll_status()
    h.close()
    return nets, rows


def _oracle(case):
    """oracle/ultralytics_restate.py + the tracker oracle, tick by tick."""
    _, _, pk, skip = CASES[case]
    _, in_hw, _, heads = _tick_inputs(case)
    trk = O.IouTracker(max_age=TRK[0], max_iou_distance=TRK[2], min_hits=TRK[1])
    rows = []
    for t in range(NT):
        dets_t, trks_t = [], []
        for s in range(TB):
            want = [] if skip and skip[s] else U.postprocess(heads[t][s], in_hw, THW, CONF, IOU, **pk)
            dets_t.append(want)
            tr = trk.update(f"s{s}", [O.Det(c, f, tuple(b)) for c, f, b in want])
            trks_t.append([(x.track_id, x.class_id, x.age, x.hits, tuple(x.bbox_xyxy)) for x in tr])
        rows.append((dets_t, trks_t))
    return rows


def _rows_equal(a, b):
    (da, ta), (db, tb) = a, b
    return ta == tb and all(all(np.array_equal(x, y) for x, y in zip(p, q)) for p, q in zip(da, db))


_SEPARATE = {}


@pytest.mark.parametrize("nv12", [False, True])
@pytest.mark.parametrize("graph", [False, True])
@pytest.mark.parametrize("schedule", [0, 1, 2, 3, 4, 5, 6])
@pytest.mark.parametrize("case", list(CASES))
def test_tick_ultralytics_matches_separate_calls(case, schedule, graph, nv12):
    key = (case, nv12)
    if key not in _SEPARATE:
        _SEPARATE[key] = _run_separate(case, nv12)
    want_nets, want_rows = _SEPARATE[key]
    got_nets, got_rows = _run_ticks(case, schedule, graph, nv12)
    assert len(got_rows) == len(want_rows) == NT
    for t in range(NT):
        assert _same(got_nets[t], want_nets[t]), (case, schedule, graph, nv12, t)
        assert _rows_equal(got_rows[t], want_rows[t]), (case, schedule, graph, nv12, t)
    assert any(len(r) for _, trk in got_rows for r in trk)


@pytest.mark.parametrize("case", list(CASES))
def test_separate_calls_match_the_oracle(case):
    """Anchors the tick comparison: the separate calls against the NumPy restatement and the tracker oracle."""
    _, rows = _SEPARATE.get((case, False)) or _run_separate(case, False)
    want = _oracle(case)
    _, in_hw, frames, _ = _tick_inputs(case)
    for t in range(NT):
        (dets, trks), (wd, wt) = rows[t], want[t]
        assert trks == wt, (case, t)
        for (cls, conf, box), w in zip(dets, wd):
            assert cls.tolist() == [c for c, _, _ in w]
            assert np.array_equal(conf, np.array([s for _, s, _ in w], dtype=np.float32))
            assert np.array_equal(box.reshape(-1, 4), np.array([b for _, _, b in w], dtype=np.float32).reshape(-1, 4))
    if case == "ties_maxdet_agnostic":
        assert all(len(d[0]) == 7 for d in rows[0][0])
    if case == "dense":
        assert max(len(d[0]) for d in rows[0][0]) > 256
    ref, _ = U.preprocess(cvr.nv12_to_bgr(frames[-1][0]), IN, auto=True, stride=32)
    assert ref.shape[2:] == in_hw


def test_tick_ultralytics_sparse_head_takes_the_fused_kernel():
    """A sparse scene runs NMS + tracker of the Ultralytics post-process as one k_post_track<true> launch, and a dense
    one the dense kernels with the tracker in the resolving CTA."""
    from torch.profiler import ProfilerActivity, profile

    names = {}
    for case in ("sparse", "dense"):
        with profile(activities=[ProfilerActivity.CUDA]) as prof:
            _run_ticks(case, 1, False, False)
        names[case] = " ".join(e.key for e in prof.key_averages())
    assert "k_post_track<true>" in names["sparse"]
    assert "k_dense_resolve_track" in names["dense"] and "k_post_track" not in names["dense"]


# ---- HotPathEngine / TickCollector in Ultralytics mode --------------------------------------------------------------
class _PerFrame:
    """One reference stream worker on the Ultralytics backend: ROI -> downsample -> motion -> adaptive FPS ->
    B200UltralyticsDetector.predict -> filter_detections -> rescale -> B200IouTracker.update."""

    def __init__(self, spec, det, trk, box, idx):
        self.spec, self.det, self.trk, self.box, self.idx = spec, det, trk, box, idx
        self.motion = None
        self.frame_index, self.idle_frames, self.process_every = 0, 0, 1
        s = spec
        self.max_process_every = max(1, int(round((s.target_fps or 30.0) / max(s.min_target_fps, 1.0))))
        self.idle_tolerance = max(int(s.idle_frame_tolerance), 1)

    def _adjust(self, n_det, n_trk):
        if not self.spec.adaptive_fps:
            return
        if n_det > 0 or n_trk > 0:
            self.idle_frames, self.process_every = 0, 1
        else:
            self.idle_frames += 1
            if self.idle_frames >= self.idle_tolerance:
                self.process_every = max(self.max_process_every, 1)

    def process(self, frame, t):
        from realtime_video_analytics_32streams_b200 import FramePacket, filter_detections

        s = self.spec
        self.frame_index += 1
        f = frame
        host_nv12 = isinstance(f, np.ndarray) and f.ndim == 2
        if s.roi_polygons or s.downsample_ratio < 0.999 or s.motion_filter:
            f = cvr.nv12_to_bgr(f) if host_nv12 else f
            if s.roi_polygons:
                f = O.apply_roi(f, s.roi_polygons, backend="cv2")
            if s.downsample_ratio < 0.999:
                f = O.downsample(f, s.downsample_ratio, backend="cv2")
        reason = None
        if s.motion_filter:
            if self.motion is None:
                self.motion = O.MotionFilter(s.motion_threshold, backend="cv2")
            if not self.motion.should_process(f):
                reason = "motion"
        if reason is None and s.adaptive_fps and self.process_every > 1 and (self.frame_index - 1) % self.process_every:
            reason = "adaptive"
        if reason is not None:
            tracks = self.trk.update(s.name, [])
            self._adjust(0, len(tracks))
            return False, reason, [], tracks
        self.box["s"], self.box["t"] = self.idx, t
        dets = filter_detections(self.det.predict(FramePacket(s, f, t)), CONF)
        if s.downsample_ratio < 0.999:
            sc = 1.0 / max(s.downsample_ratio, 1e-6)
            dets = [types.SimpleNamespace(class_id=d.class_id, confidence=d.confidence,
                                          bbox_xyxy=tuple(v * sc for v in d.bbox_xyxy)) for d in dets]
        tracks = self.trk.update(s.name, dets)
        self._adjust(len(dets), len(tracks))
        return True, None, dets, tracks


def _synthetic_infer(box, h):
    """Per-stream synthetic heads: stream s at tick t gets _head(s, in_hw, t) (stream 2 is quiet in ticks 5-11)."""
    import torch

    def infer(tensor, streams=None):
        in_hw = tuple(tensor.shape[2:])
        idx = streams if streams is not None else [box["s"]]
        t = box["t"]
        out = [np.zeros((84, _anchors(in_hw)), np.float32) if (s == 2 and 5 <= t < 12) else _head(70 + s, in_hw, n_obj=6, t=t)
               for s in idx]
        return torch.from_numpy(np.stack(out)).to(h.device)

    return infer


def _streams(specs):
    from realtime_video_analytics_32streams_b200 import StreamConfig

    out = []
    for i, (hw, cfg, _) in enumerate(specs):
        kw = {k: v for k, v in cfg.items() if k != "roi"}
        if cfg.get("roi"):
            kw["roi_polygons"] = synth.synth_polygons(400 + i, *hw)
        out.append(StreamConfig(name=f"cam{i}", **kw))
    return out


def _frame(scenes, specs, i, t):
    """Host BGR, host NV12, CUDA NV12 or a (y, uv) pair of stream i at tick t, and the frame the reference sees."""
    hw, _, how = specs[i]
    bgr = scenes[i].frame(t)
    if how == "bgr":
        return bgr, bgr
    nv = _bgr_to_nv12(bgr)
    if how == "nv12":
        return nv, nv
    if how == "cuda":
        return _cu(nv), nv
    return (_cu(nv[:hw[0]]), _cu(nv[hw[0]:])), nv


def _bgr_to_nv12(bgr):
    import cv2

    h, w = bgr.shape[:2]
    i420 = cv2.cvtColor(bgr, cv2.COLOR_BGR2YUV_I420)
    y, u, v = i420[:h], i420[h:h + h // 4].reshape(h // 2, w // 2), i420[h + h // 4:].reshape(h // 2, w // 2)
    return np.concatenate([y, np.stack([u, v], axis=2).reshape(h // 2, w)])


def _result_tuple(processed, reason, dets, tracks):
    return (processed, reason, [(d.class_id, d.confidence, tuple(d.bbox_xyxy)) for d in dets],
            [(x.track_id, x.class_id, x.confidence, tuple(x.bbox_xyxy), x.age, x.hits) for x in tracks])


def _make_pair(specs, device_gates=False, collector=False):
    from realtime_video_analytics_32streams_b200 import (B200IouTracker, B200UltralyticsDetector, DetectorConfig,
                                                         HotPathEngine, TrackerConfig)

    ha, hb = _handle(), _handle()
    dcfg = DetectorConfig(confidence_threshold=CONF, iou_threshold=IOU, backend="b200_ultralytics")
    tcfg = TrackerConfig(max_age=3, max_iou_distance=0.5, min_hits=1)
    box_e, box_r = {}, {}
    infer_e = _synthetic_infer(box_e, ha)
    det_e = B200UltralyticsDetector(dcfg, input_hw=IN, handle=ha,
                                    infer=lambda tensor: infer_e(tensor, box_e["eng"].active_streams))
    det_r = B200UltralyticsDetector(dcfg, input_hw=IN, handle=hb, infer=_synthetic_infer(box_r, hb))
    streams = _streams(specs)
    if collector:
        from realtime_video_analytics_32streams_b200.collector import default_engine_factory

        eng = default_engine_factory(streams, det_e, types.SimpleNamespace(tracker=tcfg))
    else:
        eng = HotPathEngine(streams, dcfg, tcfg, infer=None, detector=det_e, device_gates=device_gates)
    box_e["eng"] = eng
    trk = B200IouTracker(tcfg, handle=hb)
    workers = [_PerFrame(s, det_r, trk, box_r, i) for i, s in enumerate(streams)]
    return eng, box_e, workers, (ha, hb)


ENGINE_CONFIGS = {
    "one_group": [((1080, 1920), dict(), "bgr")] * 4,
    "interleaved_groups": [((1080, 1920), dict(), "bgr"), ((480, 640), dict(), "bgr"), ((1920, 1080), dict(), "bgr"),
                           ((1080, 1920), dict(), "bgr"), ((480, 640), dict(), "bgr")],
    "mixed_bgr_nv12": [((1080, 1920), dict(), "nv12"), ((480, 640), dict(), "bgr"), ((720, 1280), dict(), "cuda"),
                       ((1080, 1920), dict(), "bgr"), ((480, 640), dict(), "pair")],
    "roi_downsample": [((1080, 1920), dict(roi=True), "bgr"), ((1080, 1920), dict(downsample_ratio=0.5), "bgr"),
                       ((720, 1280), dict(roi=True, downsample_ratio=0.75), "nv12"), ((480, 640), dict(roi=True), "cuda")],
    "motion_adaptive": [((540, 960), dict(motion_filter=True, motion_threshold=0.01), "bgr"),
                        ((480, 640), dict(roi=True, motion_filter=True, motion_threshold=0.004), "nv12"),
                        ((540, 960), dict(adaptive_fps=True, target_fps=25, min_target_fps=5, idle_frame_tolerance=2), "bgr"),
                        ((1080, 1920), dict(), "bgr")],
}


def _scenes(specs):
    """Moving scenes; a stream whose motion threshold is 0.004 (motion_adaptive) sees a static one."""
    return [synth.MotionScene(300 + i, *hw, static=cfg.get("motion_threshold") == 0.004) for i, (hw, cfg, _) in enumerate(specs)]


def _drive(name, T=14, device_gates=False):
    specs = ENGINE_CONFIGS[name]
    eng, box_e, workers, handles = _make_pair(specs, device_gates=device_gates)
    scenes = _scenes(specs)
    seen = {"motion": 0, "adaptive": 0, "processed": 0, "dets": 0}
    host_bytes = 0
    try:
        for t in range(T):
            frames, refs = zip(*[_frame(scenes, specs, i, t) for i in range(len(specs))])
            host_bytes += sum(f.nbytes for f in frames if isinstance(f, np.ndarray))
            box_e["t"] = t
            got = eng.tick(list(frames), [t] * len(specs))
            for i, (g, w) in enumerate(zip(got, workers)):
                want = _result_tuple(*w.process(refs[i], t))
                assert _result_tuple(g.processed, g.skip_reason, g.detections, g.tracks) == want, (name, t, i)
                seen["processed"] += int(g.processed)
                seen["dets"] += len(g.detections)
                if g.skip_reason:
                    seen[g.skip_reason] += 1
        return seen, eng.stager.bytes_moved, host_bytes
    finally:
        for h in handles:
            h.close()


@pytest.mark.parametrize("name", ["one_group", "interleaved_groups", "mixed_bgr_nv12", "roi_downsample"])
def test_engine_ultralytics_matches_the_per_frame_loop(name):
    seen, moved, host_bytes = _drive(name)
    assert seen["processed"] > 0 and seen["dets"] > 0
    if host_bytes:
        assert moved < host_bytes  # only the rows each frame's LetterBox reads cross the bus


@pytest.mark.parametrize("device_gates", [False, True])
def test_engine_ultralytics_motion_and_adaptive_gates(device_gates):
    seen, _, _ = _drive("motion_adaptive", T=18, device_gates=device_gates)
    assert seen["motion"] > 0 and seen["adaptive"] > 0 and seen["dets"] > 0, seen


def test_engine_ultralytics_pipelined_submit_collect():
    specs = ENGINE_CONFIGS["mixed_bgr_nv12"]
    eng, box_e, workers, handles = _make_pair(specs)
    scenes = _scenes(specs)
    try:
        pending, n = None, 0
        for t in range(9):
            frames, refs = zip(*[_frame(scenes, specs, i, t) for i in range(len(specs))])
            box_e["t"] = t
            ctx = eng.submit(list(frames), [t] * len(specs))  # tick t+1 is in flight while tick t is collected
            if pending is not None:
                got = eng.collect(pending[0])
                for i, (g, w) in enumerate(zip(got, workers)):
                    assert _result_tuple(g.processed, g.skip_reason, g.detections, g.tracks) == \
                        _result_tuple(*w.process(pending[1][i], t - 1)), (t - 1, i)
                    n += len(g.detections)
            pending = (ctx, refs)
        got = eng.collect(pending[0])
        for i, (g, w) in enumerate(zip(got, workers)):
            assert _result_tuple(g.processed, g.skip_reason, g.detections, g.tracks) == \
                _result_tuple(*w.process(pending[1][i], 8)), (8, i)
        assert n > 0
    finally:
        for h in handles:
            h.close()


def test_collector_with_ultralytics_detector_runs_ultralytics_semantics():
    """TickCollector over default_engine_factory(B200UltralyticsDetector): the per-frame results of that detector.  (A
    factory that builds a B200Detector returns reference-semantics detections here, which differ.)"""
    from realtime_video_analytics_32streams_b200.collector import TickCollector

    specs = ENGINE_CONFIGS["interleaved_groups"]
    eng, box_e, workers, handles = _make_pair(specs, collector=True)
    assert eng.ultralytics
    scenes = _scenes(specs)
    col = TickCollector(eng, max_wait_s=5.0)
    streams = eng.streams

    async def drive():
        n = 0
        for t in range(6):
            frames, refs = zip(*[_frame(scenes, specs, i, t) for i in range(len(specs))])
            box_e["t"] = t
            pkts = [types.SimpleNamespace(stream=s, frame=f, frame_id=t) for s, f in zip(streams, frames)]
            res = await asyncio.gather(*[col.process(s.name, p) for s, p in zip(streams, pkts)])
            for i, (g, w) in enumerate(zip(res, workers)):
                assert _result_tuple(g.processed, g.skip_reason, g.detections, g.tracks) == \
                    _result_tuple(*w.process(refs[i], t)), (t, i)
                n += len(g.detections)
        await col.close()
        return n

    try:
        assert asyncio.run(drive()) > 0
    finally:
        for h in handles:
            h.close()
