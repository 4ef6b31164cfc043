"""NV12 frames on the hot path: every NV12 entry point must give, byte for byte, what the BGR entry point of the same
name gives on ``cv2.cvtColor(frame, COLOR_YUV2BGR_NV12)`` (restated by ``nv12_restate.nv12_to_bgr``), and what
``oracle.hotpath`` gives on that frame.  Float outputs are compared as bit patterns."""
import ctypes as C

import numpy as np
import pytest

import nv12_restate as cvr
from oracle import hotpath as O
from realtime_video_analytics_32streams_b200 import synth

pytestmark = pytest.mark.gpu

IN_HW = (640, 640)
# (h, w): 1080p (identity taps), 4K / 720p / 1440p (2 x 2 box), 640x360 (scale 1), 320x240 (upscale), 2x2, and
# 1002x750, whose horizontal taps straddle chroma pairs
SIZES = [(1080, 1920), (2160, 3840), (720, 1280), (1440, 2560), (360, 640), (240, 320), (2, 2), (750, 1002)]
FMTS = ["f32", "f16", "u8_nchw", "u8_nhwc"]


def _N():
    from realtime_video_analytics_32streams_b200 import _native

    return _native


def _handle(max_batch=80):
    return _N().Handle(device=0, max_batch=max_batch, max_anchors=8400, max_candidates=2048, max_dets=512, max_streams=8,
                       max_tracks=512)


def _fmt(name):
    N = _N()
    return {"f32": N.OUT_F32_RGB_NCHW, "f16": N.OUT_F16_RGB_NCHW, "u8_nchw": N.OUT_U8_BGR_NCHW, "u8_nhwc": N.OUT_U8_BGR_NHWC}[name]


def _nv12(seed, h, w):
    """Uniform-random NV12 frame [3H/2, W] (every Y, Cb, Cr value; saturates in every channel)."""
    return np.random.default_rng(seed).integers(0, 256, size=(h * 3 // 2, w), dtype=np.uint8)


def _cu(a):
    import torch

    return torch.from_numpy(np.ascontiguousarray(a)).cuda()


def _oracle(bgr, fmt_name, mask_polys=None):
    src = O.apply_roi(bgr, mask_polys, backend="cv2") if mask_polys else bgr
    if fmt_name in ("f32", "f16"):
        return O.preprocess(src, IN_HW, half=fmt_name == "f16", backend="cv2")[0][0]
    return O.preprocess_u8(src, IN_HW, nhwc=fmt_name == "u8_nhwc", backend="cv2")[0][0]


def _same(a, b):
    a, b = np.ascontiguousarray(a), np.ascontiguousarray(b)
    return a.shape == b.shape and np.array_equal(a.view(np.uint8), b.view(np.uint8))


@pytest.mark.parametrize("fmt_name", FMTS)
def test_letterbox_all_formats_and_sizes_in_one_launch(fmt_name):
    """Mixed sizes in one call; then the same call with PADS_VALID into a buffer whose content rows were cleared."""
    import torch

    N = _N()
    h = _handle()
    fmt = _fmt(fmt_name)
    nv = [_nv12(10 + i, *hw) for i, hw in enumerate(SIZES)]
    bgr = [cvr.nv12_to_bgr(f) for f in nv]
    got, metas = h.preprocess([_cu(f) for f in nv], IN_HW, fmt)
    ref, ref_metas = h.preprocess([_cu(f) for f in bgr], IN_HW, fmt)
    torch.cuda.synchronize()
    g, r = got.cpu().numpy(), ref.cpu().numpy()
    for i in range(len(SIZES)):
        assert _same(g[i], r[i]), (SIZES[i], "vs BGR entry point")
        assert _same(g[i], _oracle(bgr[i], fmt_name)), (SIZES[i], "vs oracle")
        assert (metas[i].new_h, metas[i].new_w, metas[i].pad_top) == (ref_metas[i].new_h, ref_metas[i].new_w, ref_metas[i].pad_top)
    # PADS_VALID: the pad rows stay as the first call left them, every other row is written again
    again = got.clone()
    for i, m in enumerate(metas):
        if fmt_name == "u8_nhwc":
            again[i, m.pad_top:m.pad_top + m.new_h] = 0
        else:
            again[i, :, m.pad_top:m.pad_top + m.new_h] = 0
    h.preprocess([_cu(f) for f in nv], IN_HW, fmt | N.OUT_FLAG_PADS_VALID, out=again)
    torch.cuda.synchronize()
    assert _same(again.cpu().numpy(), g)
    h.poll_status()
    h.close()


def test_65_frames_two_launch_groups_and_roi_masks():
    import torch

    h = _handle(max_batch=80)
    hw = (360, 640)
    nv = [_nv12(100 + i, *hw) for i in range(65)]
    polys = [synth.synth_polygons(200 + i, *hw) if i % 3 == 0 else None for i in range(65)]
    masks = [h.roi_rasterize(p, *hw) if p else None for p in polys]
    bgr = [cvr.nv12_to_bgr(f) for f in nv]
    got, _ = h.preprocess([_cu(f) for f in nv], IN_HW, _fmt("f32"), roi_masks=masks)
    ref, _ = h.preprocess([_cu(f) for f in bgr], IN_HW, _fmt("f32"), roi_masks=masks)
    torch.cuda.synchronize()
    g, r = got.cpu().numpy(), ref.cpu().numpy()
    assert _same(g, r)
    for i in (0, 1, 3, 63, 64):
        assert _same(g[i], _oracle(bgr[i], "f32", polys[i])), i
    h.close()


@pytest.mark.parametrize("hw", [(1080, 1920), (2160, 3840), (750, 1002)])
def test_roi_masks_large_frames(hw):
    import torch

    h = _handle()
    nv = _nv12(7, *hw)
    bgr = cvr.nv12_to_bgr(nv)
    polys = synth.synth_polygons(8, *hw)
    mask = h.roi_rasterize(polys, *hw)
    for fmt_name in ("f16", "u8_nhwc"):
        got, _ = h.preprocess([_cu(nv)], IN_HW, _fmt(fmt_name), roi_masks=[mask])
        ref, _ = h.preprocess([_cu(bgr)], IN_HW, _fmt(fmt_name), roi_masks=[mask])
        torch.cuda.synchronize()
        assert _same(got.cpu().numpy(), ref.cpu().numpy())
        assert _same(got.cpu().numpy()[0], _oracle(bgr, fmt_name, polys))
    h.close()


def _layouts(nv, hw):
    """The same NV12 frame as (y, uv) CUDA planes in several memory layouts."""
    import torch

    H, W = hw
    y_np, uv_np = nv[:H], nv[H:]
    out = {}
    # chroma in a separate allocation, uv_pitch != y_pitch (both 16-byte multiples: bulk copies)
    yb = torch.zeros((H, W + 64), dtype=torch.uint8, device="cuda")
    ub = torch.zeros((H // 2, W + 192), dtype=torch.uint8, device="cuda")
    yb[:, :W] = _cu(y_np)
    ub[:, :W] = _cu(uv_np)
    out["separate"] = (yb[:, :W], ub[:, :W])
    # decoder surface: chroma plane at pitch * (H + 8)
    P = (W + 255) // 256 * 256
    surf = torch.zeros((H + 8 + H // 2, P), dtype=torch.uint8, device="cuda")
    surf[:H, :W] = _cu(y_np)
    surf[H + 8:, :W] = _cu(uv_np)
    out["surface"] = (surf[:H, :W], surf[H + 8:, :W])
    # unaligned luma base and odd pitch: the byte loader
    ybad = torch.zeros((H, W + 3), dtype=torch.uint8, device="cuda")
    ybad[:, 1:W + 1] = _cu(y_np)
    out["unaligned"] = (ybad[:, 1:W + 1], ub[:, :W])
    # OpenCV's single [3H/2, W] buffer with a row pitch above W
    one = torch.zeros((H * 3 // 2, W + 32), dtype=torch.uint8, device="cuda")
    one[:, :W] = _cu(nv)
    out["pitched"] = one[:, :W]
    return out


@pytest.mark.parametrize("hw", [(1080, 1920), (720, 1280), (750, 1002)])
def test_plane_layouts(hw):
    import torch

    h = _handle()
    nv = _nv12(31, *hw)
    bgr = cvr.nv12_to_bgr(nv)
    ref, _ = h.preprocess([_cu(bgr)], IN_HW, _fmt("f32"))
    want = ref.cpu().numpy()
    lay = _layouts(nv, hw)
    got, _ = h.preprocess(list(lay.values()), IN_HW, _fmt("f32"))
    torch.cuda.synchronize()
    g = got.cpu().numpy()
    for i, name in enumerate(lay):
        assert _same(g[i], want[0]), name
    outs = h.resize(list(lay.values()), [hw] * len(lay))  # cvtColor itself, from every layout
    for name, o in zip(lay, outs):
        assert np.array_equal(o.cpu().numpy(), bgr), name
    h.close()


def test_saturating_values():
    import torch

    ys, cs = [0, 15, 16, 235, 255], [0, 128, 255]
    H, W = 60, 90  # 30 x 45 blocks of 2 x 2: the first 45 of row 0 hold every (Y, Cb, Cr) of the sets above
    rng = np.random.default_rng(3)
    y = np.array(ys, np.uint8)[rng.integers(0, 5, (H, W))]
    uv = np.array(cs, np.uint8)[rng.integers(0, 3, (H // 2, W))]
    for k in range(45):
        y[0:2, 2 * k:2 * k + 2] = ys[k // 9]
        uv[0, 2 * k], uv[0, 2 * k + 1] = cs[(k // 3) % 3], cs[k % 3]
    nv = np.concatenate([y, uv])
    bgr = cvr.nv12_to_bgr(nv)
    import cv2

    assert np.array_equal(bgr, cv2.cvtColor(nv, cv2.COLOR_YUV2BGR_NV12))
    h = _handle()
    out = h.resize([_cu(nv)], [(H, W)])[0]
    assert np.array_equal(out.cpu().numpy(), bgr)
    for fmt_name in FMTS:
        got, _ = h.preprocess([_cu(nv)], IN_HW, _fmt(fmt_name))
        torch.cuda.synchronize()
        assert _same(got.cpu().numpy()[0], _oracle(bgr, fmt_name)), fmt_name
    h.close()


def test_device_skip_mask():
    import torch

    h = _handle()
    hw = (720, 1280)
    nv = [_nv12(50 + i, *hw) for i in range(4)]
    full, _ = h.preprocess([_cu(f) for f in nv], IN_HW, _fmt("f32"))
    out = torch.full_like(full, 7.0)
    skip = torch.tensor([0, 1, 0, 1], dtype=torch.uint8, device="cuda")
    h.set_skip_mask(skip)
    try:
        h.preprocess([_cu(f) for f in nv], IN_HW, _fmt("f32"), out=out)
    finally:
        h.set_skip_mask(None)
    torch.cuda.synchronize()
    o, f = out.cpu().numpy(), full.cpu().numpy()
    assert _same(o[0], f[0]) and _same(o[2], f[2])
    assert (o[1] == 7.0).all() and (o[3] == 7.0).all()
    h.close()


@pytest.mark.parametrize("ratio", [0.5, 0.33, 0.75, 1.0])
def test_resize_nv12_downsample_ratios(ratio):
    import torch

    h = _handle()
    sizes = [(1080, 1920), (720, 1280), (750, 1002)]
    nv = [_nv12(70 + i, *hw) for i, hw in enumerate(sizes)]
    bgr = [cvr.nv12_to_bgr(f) for f in nv]
    polys = synth.synth_polygons(9, *sizes[1])
    masks = [None, h.roi_rasterize(polys, *sizes[1]), None]
    dst = [(int(hh * ratio), int(ww * ratio)) for hh, ww in sizes]
    got = h.resize([_cu(f) for f in nv], dst, masks)
    ref = h.resize([_cu(f) for f in bgr], dst, masks)
    torch.cuda.synchronize()
    for i in range(3):
        g = got[i].cpu().numpy()
        assert np.array_equal(g, ref[i].cpu().numpy()), sizes[i]
        src = O.apply_roi(bgr[i], polys, backend="cv2") if masks[i] is not None else bgr[i]
        want = src if ratio == 1.0 else O.downsample(src, ratio, backend="cv2")
        assert np.array_equal(g, want), sizes[i]
    h.close()


@pytest.mark.parametrize("hw,full,sparse", [((1080, 1920), 3_110_400, 1_382_400), ((2160, 3840), 12_441_600, 4_147_200),
                                           ((720, 1280), 1_382_400, None)])
def test_upload_nv12_rows_modes(hw, full, sparse):
    import torch

    N = _N()
    h = _handle()
    H, W = hw
    nv = _nv12(90, H, W)
    pinned = torch.from_numpy(nv).pin_memory()
    ptr, pitch = pinned.data_ptr(), pinned.stride(0)
    host = [N.Nv12Frame(ptr, ptr + H * pitch, pitch, pitch)]
    dev_full = torch.zeros((H * 3 // 2, W), dtype=torch.uint8, device="cuda")
    dev_sparse = torch.zeros_like(dev_full)
    assert h.upload_frames_nv12(host, [dev_full]) == full
    moved = h.upload_frames_nv12(host, [dev_sparse], sparse_for=IN_HW)
    torch.cuda.synchronize()
    assert np.array_equal(dev_full.cpu().numpy(), nv)
    if sparse is not None:
        assert moved == sparse
    assert moved <= full
    a, _ = h.preprocess([dev_full], IN_HW, _fmt("f32"))
    b, _ = h.preprocess([dev_sparse], IN_HW, _fmt("f32"))
    torch.cuda.synchronize()
    assert _same(a.cpu().numpy(), b.cpu().numpy())
    # a decoder-surface destination: separate plane pitches
    P = (W + 511) // 512 * 512
    surf = torch.zeros((H + 16 + H // 2, P), dtype=torch.uint8, device="cuda")
    planes = (surf[:H, :W], surf[H + 16:, :W])
    assert h.upload_frames_nv12(host, [planes], sparse_for=IN_HW) == moved
    c, _ = h.preprocess([planes], IN_HW, _fmt("f32"))
    torch.cuda.synchronize()
    assert _same(c.cpu().numpy(), a.cpu().numpy())
    h.close()


def test_invalid_arguments_are_refused():
    import torch

    N = _N()
    h = _handle()
    out = torch.empty((1, 3, *IN_HW), dtype=torch.float32, device="cuda")
    y = torch.zeros((8, 8), dtype=torch.uint8, device="cuda")
    metas = (N.Letterbox * 1)()

    def call(frame, hh, ww):
        return h.lib.b200va_preprocess_nv12(h._h, (N.Nv12Frame * 1)(frame), N._int_array([hh]), N._int_array([ww]), 1, None,
                                            C.c_void_p(out.data_ptr()), IN_HW[0], IN_HW[1], N.OUT_F32_RGB_NCHW, metas,
                                            h._stream())

    p = y.data_ptr()
    assert call(N.Nv12Frame(p, p, 8, 8), 8, 8) == N.OK
    assert call(N.Nv12Frame(p, p, 8, 8), 7, 8) == N.ERR_INVALID
    assert call(N.Nv12Frame(p, p, 8, 8), 8, 7) == N.ERR_INVALID
    assert call(N.Nv12Frame(None, p, 8, 8), 8, 8) == N.ERR_INVALID
    assert call(N.Nv12Frame(p, None, 8, 8), 8, 8) == N.ERR_INVALID
    assert call(N.Nv12Frame(p, p, 6, 8), 8, 8) == N.ERR_INVALID
    dst = N._ptr_array([out.data_ptr()])
    assert h.lib.b200va_resize_linear_u8_nv12(h._h, (N.Nv12Frame * 1)(N.Nv12Frame(p, p, 8, 8)), N._int_array([8]),
                                              N._int_array([7]), 1, None, dst, N._int_array([4]), N._int_array([4]),
                                              h._stream()) == N.ERR_INVALID
    assert h.lib.b200va_upload_frames_nv12(h._h, (N.Nv12Frame * 1)(N.Nv12Frame(p, None, 8, 8)),
                                           (N.Nv12Frame * 1)(N.Nv12Frame(p, p, 8, 8)), N._int_array([8]), N._int_array([8]), 1,
                                           640, 640, 0, None, h._stream()) == N.ERR_INVALID
    with pytest.raises(ValueError):  # odd width
        h.preprocess([torch.zeros((9, 7), dtype=torch.uint8, device="cuda")], IN_HW)
    with pytest.raises(ValueError):  # odd height
        h.preprocess([(torch.zeros((5, 8), dtype=torch.uint8, device="cuda"), torch.zeros((2, 8), dtype=torch.uint8, device="cuda"))],
                     IN_HW)
    torch.cuda.synchronize()
    h.close()


# ---- b200va_tick_nv12 -------------------------------------------------------------------------------------------
TB, THW, CONF, IOU, TRK = 6, (540, 960), 0.35, 0.5, (30, 1, 0.5)


def _tick_inputs(n_ticks):
    frames = [[_nv12(900 + 10 * t + s, *THW) for s in range(TB)] for t in range(n_ticks)]
    heads = [np.stack([synth.synth_head(700 + 10 * t + s, 84, 8400, 14, dup=3) for s in range(TB)]) for t in range(n_ticks)]
    return frames, heads


def _track_rows(tracks):
    out = []
    for s in range(TB):
        n = int(tracks["count"][s].item())
        out.append(list(zip(tracks["track_id"][s, :n].cpu().tolist(), tracks["cls"][s, :n].cpu().tolist(),
                            tracks["hits"][s, :n].cpu().tolist(), [tuple(b) for b in tracks["bbox_xyxy"][s, :n].cpu().tolist()])))
    return out


def _run_ticks(nv12, schedule, graph, n_ticks=5):
    """net inputs and track rows of every tick (schedule 4: tables lag one call; drained at the end).  Graph mode: one
    eager call, then two graphs (one per plan) replayed alternately; an odd tick count ends on the graph captured
    last, which is what the host-side state of schedule 4 expects when the pipeline is drained."""
    import torch

    N = _N()
    frames, heads = _tick_inputs(n_ticks)
    h = _handle(max_batch=8)
    h.tracker_set_next_id(1)
    net = torch.zeros((TB, 3, *IN_HW), dtype=torch.float32, device="cuda")
    metas = [N.letterbox_meta(*THW, *IN_HW) for _ in range(TB)]
    shape = (THW[0] * 3 // 2, THW[1]) if nv12 else (*THW, 3)
    dev = [torch.zeros(shape, dtype=torch.uint8, device="cuda") for _ in range(TB)]
    head = torch.zeros((TB, 84, 8400), dtype=torch.float32, device="cuda")
    tracks = [h.alloc_tracks(TB) for _ in range(2)]
    plans = [h.plan_tick(frames=dev, net_out=net, dst_hw=IN_HW, head=head, metas=metas, conf_thr=CONF, iou_thr=IOU,
                         filter_conf=CONF, slots=list(range(TB)), tracker_cfg=TRK, schedule=schedule, tracks=tracks[k])
             for k in range(2)]
    assert (plans[0].nv12 is not None) == nv12
    graphs = None
    nets, rows = [], []

    def load(t):
        for s in range(TB):
            src = frames[t][s] if nv12 else cvr.nv12_to_bgr(frames[t][s])
            dev[s].copy_(torch.from_numpy(src))
        head.copy_(torch.from_numpy(heads[t]))

    for t in range(n_ticks):
        load(t)
        if graph and graphs is None:
            h.tick(plans[t % 2])  # eager first call, then capture one graph per plan
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
            rows.append(_track_rows(tracks[t % 2]))
        elif t > 0:
            rows.append(_track_rows(tracks[(t - 1) % 2]))
    if schedule == N.SCHEDULE_SOFTWARE_PIPELINED:
        h.tick(h.plan_tick(schedule=schedule))
        torch.cuda.synchronize()
        rows.append(_track_rows(tracks[(n_ticks - 1) % 2]))
    h.poll_status()
    h.close()
    return nets, rows, frames


@pytest.mark.parametrize("graph", [False, True])
@pytest.mark.parametrize("schedule", [1, 3, 4, 5, 6])
def test_tick_nv12_matches_bgr_tick(schedule, graph):
    want_nets, want_rows, frames = _run_ticks(False, schedule, graph)
    got_nets, got_rows, _ = _run_ticks(True, schedule, graph)
    assert len(got_rows) == len(want_rows) and got_rows == want_rows
    assert any(len(r) for tick in got_rows for r in tick)
    for t, (g, w) in enumerate(zip(got_nets, want_nets)):
        assert _same(g, w), t
    for s in (0, TB - 1):  # and the oracle on the last tick's converted frames
        assert _same(got_nets[-1][s], _oracle(cvr.nv12_to_bgr(frames[-1][s]), "f32"))


# ---- HotPathEngine ------------------------------------------------------------------------------------------------
def _bgr_to_nv12(bgr):
    import cv2

    h, w = bgr.shape[:2]
    i420 = cv2.cvtColor(bgr, cv2.COLOR_BGR2YUV_I420)
    y, u, v = i420[:h], i420[h:h + h // 4].reshape(h // 2, w // 2), i420[h + h // 4:].reshape(h // 2, w // 2)
    uv = np.stack([u, v], axis=2).reshape(h // 2, w)
    return np.concatenate([y, uv])


class _Scene:
    """A dark textured background with a bright rectangle that moves (or not): the motion gate sees it."""

    def __init__(self, seed, h, w, static=False):
        rng = np.random.default_rng(seed)
        self.bg = (rng.integers(0, 64, ((h + 7) // 8, (w + 7) // 8, 3), dtype=np.uint8).repeat(8, 0).repeat(8, 1) + 60)[:h, :w]
        self.h, self.w, self.static, self.seed = h, w, static, seed

    def frame(self, t):
        f = self.bg.copy()
        x = 0 if self.static else (37 * t * (1 + self.seed % 3)) % max(self.w // 2, 1)
        y = self.h // 4 if self.static or t % 5 else self.h // 3
        f[y:y + self.h // 3, x:x + self.w // 3] = (255, 250 - self.seed % 5, 245)  # far brighter than the background
        return f


@pytest.mark.parametrize("device_gates", [False, True])
def test_engine_nv12_matches_engine_on_converted_frames(device_gates):
    import torch
    from realtime_video_analytics_32streams_b200 import DetectorConfig, HotPathEngine, StreamConfig, TrackerConfig

    T = 24
    # (size, config, how the NV12 frame is handed over)
    specs = [((1080, 1920), dict(), "host"),
             ((720, 1280), dict(roi=True), "cuda"),
             ((540, 960), dict(motion_filter=True, motion_threshold=0.01, adaptive_fps=True, target_fps=25, min_target_fps=5,
                               idle_frame_tolerance=3), "pair"),
             ((720, 1280), dict(downsample_ratio=0.5), "host"),
             ((720, 1280), dict(roi=True, motion_filter=True, motion_threshold=0.004, downsample_ratio=0.5), "cuda"),
             ((540, 960), dict(roi=True, motion_filter=True, motion_threshold=0.02), "host"),
             ((360, 640), dict(), "bgr")]  # a BGR stream in the same batch
    scenes = [_Scene(300 + i, *hw, static=(i == 5)) for i, (hw, _, _) in enumerate(specs)]

    def streams():
        out = []
        for i, (hw, cfg, _) in enumerate(specs):
            kw = {k: v for k, v in cfg.items() if k != "roi"}
            if cfg.get("roi"):
                kw["roi_polygons"] = synth.synth_polygons(400 + i, *hw)
            out.append(StreamConfig(name=f"cam{i}", **kw))
        return out

    def make(h):
        h.tracker_set_next_id(1)
        box = {}

        def infer(tensor):
            t = box["t"]
            heads = []
            for s in box["eng"].active_streams:
                quiet = s == 2 and 6 <= t < 16  # no detections: the adaptive gate raises process_every
                heads.append(np.zeros((84, 8400), np.float32) if quiet else synth.synth_head(1000 + 37 * t + s, 84, 8400, 6, dup=2))
            return torch.from_numpy(np.stack(heads)).to(h.device)

        eng = HotPathEngine(streams(), DetectorConfig(confidence_threshold=CONF, iou_threshold=IOU),
                            TrackerConfig(max_age=3, max_iou_distance=0.5, min_hits=1), infer=infer, handle=h,
                            input_hw=IN_HW, device_gates=device_gates)
        box["eng"] = eng
        return eng, box

    ha, hb = _handle(max_batch=8), _handle(max_batch=8)
    try:
        eng_nv, box_nv = make(ha)
        eng_bgr, box_bgr = make(hb)
        seen = {"motion": 0, "adaptive": 0, "processed": 0}
        for t in range(T):
            bgr_frames, nv_frames = [], []
            for i, (hw, _, how) in enumerate(specs):
                bgr = scenes[i].frame(t)
                if how == "bgr":
                    bgr_frames.append(bgr)
                    nv_frames.append(bgr)
                    continue
                nv = _bgr_to_nv12(bgr)
                bgr_frames.append(cvr.nv12_to_bgr(nv))
                if how == "host":
                    nv_frames.append(nv)
                elif how == "cuda":
                    nv_frames.append(_cu(nv))
                else:
                    H = hw[0]
                    nv_frames.append((_cu(nv[:H]), _cu(nv[H:])))
            box_nv["t"] = box_bgr["t"] = t
            got, want = eng_nv.tick(nv_frames), eng_bgr.tick(bgr_frames)
            for s, (g, w) in enumerate(zip(got, want)):
                assert (g.processed, g.skip_reason, g.frame_id, g.adaptive_state) == \
                    (w.processed, w.skip_reason, w.frame_id, w.adaptive_state), (t, s)
                assert (g.n_detections, g.n_tracks) == (w.n_detections, w.n_tracks), (t, s)
                for k, v in w.detection_arrays.items():
                    assert _same(g.detection_arrays[k], v), (t, s, k)
                for k, v in w.track_arrays.items():
                    assert _same(g.track_arrays[k], v), (t, s, k)
                seen["processed"] += int(w.processed)
                if w.skip_reason:
                    seen[w.skip_reason] += 1
        assert seen["motion"] > 0 and seen["adaptive"] > 0 and seen["processed"] > T, seen
        assert eng_nv.stager.bytes_moved < eng_bgr.stager.bytes_moved
    finally:
        ha.close()
        hb.close()
