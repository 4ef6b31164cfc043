"""GPU parity tests: the CUDA path, called through the C ABI (ctypes -> libb200va.so), against the
CPU oracle and the committed golden vectors.  Bit-exact everywhere (integer / byte / index work
and un-fused float32 / float64 arithmetic).  Run on the B200 box with ``-m gpu``."""
import numpy as np
import pytest

import golden_util as G
from oracle import hotpath as O
from realtime_video_analytics_32streams_b200 import synth

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def H():
    import torch
    from realtime_video_analytics_32streams_b200 import _native

    assert torch.cuda.is_available()
    h = _native.Handle(device=0, max_batch=64, max_anchors=25200, max_candidates=4096, max_dets=1024,
                       max_streams=64, max_tracks=2048)
    yield h
    h.poll_status()
    h.close()


def cu(a):
    import torch

    return torch.from_numpy(np.ascontiguousarray(a)).cuda()


# ------------------------------------------------------------------------------------------------
# a1 / a2 / a10: letterbox + resize
# ------------------------------------------------------------------------------------------------
def test_preprocess_golden_small(H):
    from realtime_video_analytics_32streams_b200 import _native as N

    z = G.load("preprocess")
    for i in range(int(z["pre_n"][0])):
        seed, h, w, ih, iw, half = z[f"pre{i}_cfg"].tolist()
        out, metas = H.preprocess([cu(z[f"pre{i}_frame"])], (ih, iw), N.OUT_F16_RGB_NCHW if half else N.OUT_F32_RGB_NCHW)
        ref = z[f"pre{i}_tensor"]
        got = out.cpu().numpy()
        assert got.dtype == ref.dtype and got.shape == ref.shape
        assert np.array_equal(got.view(np.uint8), ref.view(np.uint8)), f"case {i}"
        oh, ow, left, top = z[f"pre{i}_meta"].tolist()
        m = metas[0].as_meta()
        assert m["orig_shape"] == (oh, ow) and m["pad"] == (left, top) and m["scale"] == float(z[f"pre{i}_scale"][0])


@pytest.mark.parametrize("key", ["1080p_f32", "4k_f32", "720p_f32", "odd_f32", "demo360_f32", "portrait_f32",
                                 "1080p_f16", "4k_f16", "odd_f16", "720p_f16", "portrait_f16"])
def test_preprocess_full_size_digests(H, key):
    from realtime_video_analytics_32streams_b200 import _native as N

    d = G.meta()["preprocess_digests"][key]
    frame = synth.synth_frame(d["seed"], d["h"], d["w"])
    out, metas = H.preprocess([cu(frame)], (640, 640), N.OUT_F16_RGB_NCHW if d["half"] else N.OUT_F32_RGB_NCHW)
    assert G.sha(out.cpu().numpy()) == d["sha256"]
    assert metas[0].scale == d["scale"] and [metas[0].pad_left, metas[0].pad_top] == d["pad"]


def test_preprocess_rknn_u8_golden(H):
    """a2: the uint8 BGR formats against vectors recorded from ``RKNNDetector._preprocess`` (detector.py:777-839)."""
    from realtime_video_analytics_32streams_b200 import _native as N

    z = G.load("preprocess_rknn")
    for i in range(int(z["rk_n"][0])):
        seed, h, w, ih, iw, nhwc = z[f"rk{i}_cfg"].tolist()
        out, metas = H.preprocess([cu(synth.synth_frame(seed, h, w))], (ih, iw), N.OUT_U8_BGR_NHWC if nhwc else N.OUT_U8_BGR_NCHW)
        got, ref = out.cpu().numpy(), z[f"rk{i}_tensor"]
        assert got.dtype == ref.dtype and got.shape == ref.shape and np.array_equal(got, ref), f"case {i}"
        oh, ow, left, top = z[f"rk{i}_meta"].tolist()
        m = metas[0].as_meta()
        assert m["orig_shape"] == (oh, ow) and m["pad"] == (left, top) and m["scale"] == float(z[f"rk{i}_scale"][0])
    for key, d in G.meta()["preprocess_rknn_digests"].items():
        frame = synth.synth_frame(d["seed"], d["h"], d["w"])
        out, metas = H.preprocess([cu(frame)], (640, 640), N.OUT_U8_BGR_NHWC if d["nhwc"] else N.OUT_U8_BGR_NCHW)
        assert G.sha(out.cpu().numpy()) == d["sha256"], key
        assert metas[0].scale == d["scale"] and [metas[0].pad_left, metas[0].pad_top] == d["pad"]


def test_preprocess_mixed_batch_and_formats(H):
    from realtime_video_analytics_32streams_b200 import _native as N

    shapes = [(1080, 1920), (2160, 3840), (720, 1280), (1083, 1921), (360, 640), (1920, 1080), (37, 100), (1000, 1000),
              (480, 854), (641, 641)]
    frames = [synth.synth_frame(300 + i, h, w) for i, (h, w) in enumerate(shapes)]
    dev = [cu(f) for f in frames]
    for fmt, half in ((N.OUT_F32_RGB_NCHW, False), (N.OUT_F16_RGB_NCHW, True)):
        out, metas = H.preprocess(dev, (640, 640), fmt)
        got = out.cpu().numpy()
        for i, f in enumerate(frames):
            ref, meta = O.preprocess(f, (640, 640), half)
            assert np.array_equal(got[i].view(np.uint8), ref[0].view(np.uint8)), (fmt, shapes[i])
            assert metas[i].as_meta() == meta
    for fmt, nhwc in ((N.OUT_U8_BGR_NHWC, True), (N.OUT_U8_BGR_NCHW, False)):
        out, _ = H.preprocess(dev, (640, 640), fmt)
        got = out.cpu().numpy()
        for i, f in enumerate(frames):
            ref, _ = O.preprocess_u8(f, (640, 640), nhwc)
            assert np.array_equal(got[i], ref[0]), (fmt, shapes[i])
    # non-square / odd network inputs (scalar store path)
    for in_hw in ((320, 416), (97, 131), (64, 64)):
        out, _ = H.preprocess(dev[:5], in_hw, N.OUT_F32_RGB_NCHW)
        got = out.cpu().numpy()
        for i in range(5):
            ref, _ = O.preprocess(frames[i], in_hw, False)
            assert np.array_equal(got[i].view(np.uint8), ref[0].view(np.uint8)), (in_hw, shapes[i])


def test_preprocess_pitched_and_unaligned_views(H):
    from realtime_video_analytics_32streams_b200 import _native as N

    big = synth.synth_frame(77, 400, 700)
    dbig = cu(big)
    views = [(slice(3, 303), slice(5, 485)), (slice(0, 400), slice(16, 656)), (slice(10, 60), slice(1, 700))]
    for ys, xs in views:
        out, _ = H.preprocess([dbig[ys, xs]], (128, 160), N.OUT_F32_RGB_NCHW)
        ref, _ = O.preprocess(np.ascontiguousarray(big[ys, xs]), (128, 160), False)
        assert np.array_equal(out.cpu().numpy().view(np.uint8), ref.view(np.uint8))


def test_preprocess_with_roi_mask_matches_apply_roi_then_preprocess(H):
    from realtime_video_analytics_32streams_b200 import _native as N

    for seed, h, w in ((1000, 1080, 1920), (4000, 2160, 3840), (9, 333, 517)):
        frame = synth.synth_frame(seed, h, w)
        polys = synth.synth_polygons(seed, h, w)
        mask = H.roi_rasterize(polys, h, w)
        out, _ = H.preprocess([cu(frame)], (640, 640), N.OUT_F32_RGB_NCHW, [mask])
        ref, _ = O.preprocess(O.apply_roi(frame, polys), (640, 640), False)
        assert np.array_equal(out.cpu().numpy().view(np.uint8), ref.view(np.uint8))


def test_sparse_row_upload_feeds_the_letterbox_exactly(H):
    """Only the rows with a non-zero vertical weight cross PCIe; everything else in the device
    frame is garbage and must never influence the output."""
    import torch
    from realtime_video_analytics_32streams_b200 import _native as N
    from realtime_video_analytics_32streams_b200.runtime import FrameStager

    shapes = [(1080, 1920), (2160, 3840), (720, 1280), (1083, 1921), (360, 640), (1920, 1080), (540, 960)]
    frames = [synth.synth_frame(900 + i, h, w) for i, (h, w) in enumerate(shapes)]
    st = FrameStager(H)
    for k, f in enumerate(frames):  # poison the persistent buffers
        st.device_buffer(k, f.shape).copy_(torch.randint(0, 256, f.shape, dtype=torch.uint8, device="cuda"))
    before = st.bytes_moved
    pinned = [torch.from_numpy(f).pin_memory() if k % 2 else f for k, f in enumerate(frames)]
    dev = st.upload(pinned, sparse_for=(640, 640))
    moved = st.bytes_moved - before
    assert moved < sum(f.nbytes for f in frames) * 0.6  # 1080p: 1/3 of the rows, 4K: 1/3, 720p: all, ...
    out, _ = H.preprocess(dev, (640, 640), N.OUT_F32_RGB_NCHW)
    got = out.cpu().numpy()
    for i, f in enumerate(frames):
        ref, _ = O.preprocess(f, (640, 640), False)
        assert np.array_equal(got[i].view(np.uint8), ref[0].view(np.uint8)), shapes[i]
    # full upload is byte-identical to the source
    dev = st.upload(frames)
    for d, f in zip(dev, frames):
        assert np.array_equal(d.cpu().numpy(), f)


def test_downsample_matches_golden_and_oracle(H):
    from realtime_video_analytics_32streams_b200 import frame_filter as F

    z = G.load("filters")
    src = z["down_in"]
    assert np.array_equal(F.downsample(src, 0.5, H), z["down_out_05"])
    assert np.array_equal(F.downsample(src, 0.37, H), z["down_out_037"])
    assert F.downsample(src, 0.9995, H) is src
    for seed, h, w, s in ((5, 1080, 1920, 0.75), (6, 2160, 3840, 0.5), (7, 1083, 1921, 0.61), (8, 108, 192, 0.75)):
        f = synth.synth_frame(seed, h, w)
        assert np.array_equal(F.downsample(f, s, H), O.downsample(f, s)), (h, w, s)
    # upscale through the raw entry point
    f = synth.synth_frame(9, 90, 120)
    up = H.resize([cu(f)], [(200, 333)])[0].cpu().numpy()
    from oracle import cv_restate as cvr

    assert np.array_equal(up, cvr.resize_linear_u8(f, 333, 200))


def test_resize_batch_groups_by_destination_size(H):
    """b200va_resize_linear_u8 for a batch: frames sharing a destination size go out in one launch with per-frame
    destination pointers; mixed sizes, one ROI mask in the batch, results per frame = cv2.resize restated."""
    from oracle import cv_restate as cvr

    specs = [(1080, 1920, 540, 960), (1080, 1920, 540, 960), (720, 1280, 540, 960), (1080, 1920, 270, 480),
             (1083, 1921, 540, 960), (360, 640, 270, 480), (1080, 1920, 540, 960)]
    frames = [synth.synth_frame(70 + i, h, w) for i, (h, w, _, _) in enumerate(specs)]
    polys = synth.synth_polygons(77, 1080, 1920)
    masks = [None] * len(specs)
    masks[1] = H.roi_rasterize(polys, 1080, 1920)
    launches0 = H.launch_count
    outs = H.resize([cu(f) for f in frames], [(dh, dw) for _, _, dh, dw in specs], masks)
    assert H.launch_count - launches0 == 3  # {540x960 unmasked, 540x960 masked, 270x480}
    for i, (f, (_, _, dh, dw)) in enumerate(zip(frames, specs)):
        src = O.apply_roi(f, polys) if i == 1 else f
        assert np.array_equal(outs[i].cpu().numpy(), cvr.resize_linear_u8(src, dw, dh)), i


# ------------------------------------------------------------------------------------------------
# a9: ROI
# ------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("name", ["a", "b", "c"])
def test_apply_roi_golden(H, name):
    from realtime_video_analytics_32streams_b200 import frame_filter as F

    z = G.load("filters")
    polys = G.polys_from(z[f"roi_{name}_polys"], z[f"roi_{name}_sizes"])
    assert np.array_equal(F.apply_roi(z["roi_frame"], polys, H), z[f"roi_{name}_out"])


@pytest.mark.parametrize("name", ["1080p", "4k"])
def test_roi_full_size_digests(H, name):
    from realtime_video_analytics_32streams_b200 import frame_filter as F

    d = G.meta()["filters_digests"][name]
    polys = [[tuple(p) for p in poly] for poly in d["polys"]]
    assert G.sha(H.roi_rasterize(polys, d["h"], d["w"]).cpu().numpy()) == d["mask_sha256"]
    frame = synth.synth_frame(d["seed"], d["h"], d["w"])
    assert G.sha(F.apply_roi(frame, polys, H)) == d["roi_sha256"]
    assert F.apply_roi(frame, [], H) is frame


def test_roi_random_polygons_vs_oracle(H):
    rng = np.random.default_rng(17)
    for it in range(60):
        h, w = int(rng.integers(8, 200)), int(rng.integers(8, 260))
        lo, hi = (-40, 60) if it % 2 else (0, 0)
        polys = [[(int(rng.integers(lo, w + hi)), int(rng.integers(lo, h + hi))) for _ in range(int(rng.integers(1, 9)))]
                 for _ in range(int(rng.integers(1, 4)))]
        got = H.roi_rasterize(polys, h, w).cpu().numpy()
        assert np.array_equal(got, O.roi_mask((h, w), polys)), (it, h, w, polys)


# ------------------------------------------------------------------------------------------------
# a11: motion
# ------------------------------------------------------------------------------------------------
def test_motion_golden_sequence(H):
    from realtime_video_analytics_32streams_b200 import MotionFilterConfig
    from realtime_video_analytics_32streams_b200.frame_filter import MotionFilter

    z = G.load("filters")
    mf = MotionFilter(MotionFilterConfig(enable=True, threshold=0.02), handle=H)
    for t, frame in enumerate(z["motion_frames"]):
        assert mf.should_process(frame) == bool(z["motion_decisions"][t])
        assert np.array_equal(mf.previous_gray, z["motion_grays"][t]), t


@pytest.mark.parametrize("name", ["1080p", "4k"])
def test_motion_full_size_digest_and_counts(H, name):
    from realtime_video_analytics_32streams_b200 import MotionFilterConfig
    from realtime_video_analytics_32streams_b200.frame_filter import MotionFilter

    d = G.meta()["filters_digests"][name]
    f0 = synth.synth_frame(d["seed"], d["h"], d["w"])
    mf = MotionFilter(MotionFilterConfig(enable=True), handle=H)
    assert mf.should_process(f0) is True
    assert G.sha(mf.previous_gray) == d["blur_sha256"]
    f1 = f0.copy()
    f1[100:400, 200:900] = 255 - f1[100:400, 200:900]
    omf = O.MotionFilter(0.02)
    omf.should_process(f0)
    want = omf.should_process(f1)
    assert mf.should_process(f1) == want
    assert mf.last_count == omf.last_count
    assert np.array_equal(mf.previous_gray, omf.previous_gray)


def test_motion_odd_sizes_masks_and_batches(H):
    shapes = [(72, 128), (33, 77), (5, 9), (3, 3), (1, 40), (40, 1), (257, 513), (300, 256), (64, 272), (2, 2)]
    rng = np.random.default_rng(5)
    import torch

    frames0 = [synth.synth_frame(800 + i, h, w) for i, (h, w) in enumerate(shapes)]
    frames1 = []
    for f in frames0:
        g = f.copy()
        h, w = g.shape[:2]
        g[: max(h // 2, 1), : max(w // 2, 1)] = rng.integers(0, 256, size=g[: max(h // 2, 1), : max(w // 2, 1)].shape, dtype=np.uint8)
        frames1.append(g)
    polys = [[[(1, 1), (w - 2, 2), (w // 2, h - 1)]] if (h > 4 and w > 4 and i % 2 == 0) else None
             for i, (h, w) in enumerate(shapes)]
    masks = [H.roi_rasterize(p, h, w) if p else None for p, (h, w) in zip(polys, shapes)]
    a = [torch.empty((h, w), dtype=torch.uint8, device="cuda") for h, w in shapes]
    b = [torch.empty((h, w), dtype=torch.uint8, device="cuda") for h, w in shapes]
    c0 = H.motion([cu(f) for f in frames0], [None] * len(shapes), a, masks).cpu().numpy()
    assert (c0 == -1).all()
    c1 = H.motion([cu(f) for f in frames1], a, b, masks).cpu().numpy()
    for i, (f0, f1) in enumerate(zip(frames0, frames1)):
        mf = O.MotionFilter(0.02)
        g0 = O.apply_roi(f0, polys[i]) if polys[i] else f0
        g1 = O.apply_roi(f1, polys[i]) if polys[i] else f1
        mf.should_process(g0)
        assert np.array_equal(a[i].cpu().numpy(), mf.previous_gray), shapes[i]
        mf.should_process(g1)
        assert np.array_equal(b[i].cpu().numpy(), mf.previous_gray), shapes[i]
        assert int(c1[i]) == mf.last_count, shapes[i]


# ------------------------------------------------------------------------------------------------
# a3-a7: post-process
# ------------------------------------------------------------------------------------------------
def _post_one(H, head, meta_hw, in_hw, conf, iou, classes=None, filter_conf=None):
    from realtime_video_analytics_32streams_b200 import _native as N

    lb = N.letterbox_meta(meta_hw[0], meta_hw[1], in_hw[0], in_hw[1])
    out = H.postprocess(cu(head), [lb], conf, iou, classes, filter_conf=filter_conf)
    n = int(out["count"].cpu()[0])
    return (out["cls"][0, :n].cpu().numpy().astype(np.int64), out["conf"][0, :n].cpu().numpy().astype(np.float64),
            out["bbox_xyxy"][0, :n].cpu().numpy().astype(np.float64))


def test_postprocess_golden_cases(H):
    z = G.load("postprocess")
    for name in z["post_names"].tolist():
        conf, iou, oh, ow, ih, iw = z[f"post_{name}_cfg"].tolist()
        classes = z[f"post_{name}_classes"].tolist() or None
        cls, cf, box = _post_one(H, z[f"post_{name}_head"], (int(oh), int(ow)), (int(ih), int(iw)), conf, iou, classes)
        assert np.array_equal(cls, z[f"post_{name}_cls"]), name
        assert np.array_equal(cf, z[f"post_{name}_conf"]), name
        assert np.array_equal(box.reshape(-1, 4), z[f"post_{name}_box"]), name


def test_postprocess_dense_digest(H):
    d = G.meta()["postprocess_digests"]["dense_seed5_t0"]
    cls, cf, box = _post_one(H, synth.DenseScene(5).head(0)[None], (1080, 1920), (640, 640), 0.35, 0.5)
    assert len(cls) == d["n"]
    assert (G.sha(cls), G.sha(cf), G.sha(box)) == (d["cls"], d["conf"], d["box"])


def test_postprocess_batch32_mixed_meta_vs_oracle(H):
    from realtime_video_analytics_32streams_b200 import _native as N

    shapes = [(1080, 1920), (2160, 3840), (720, 1280), (1920, 1080)]
    heads, metas, refs = [], [], []
    for b in range(32):
        n_obj, dup = (300, 6) if b % 8 == 0 else (10 + b, 1 + b % 4)
        head = synth.synth_head(3000 + b, 84, 8400, n_obj, dup=dup, n_obj_classes=10 if b % 2 else None)
        hw = shapes[b % 4]
        heads.append(head)
        metas.append(N.letterbox_meta(hw[0], hw[1], 640, 640))
        refs.append(O.postprocess(head[None], O.letterbox_meta(hw[0], hw[1], 640, 640), 0.35, 0.5))
    out = H.postprocess(cu(np.stack(heads)), metas, 0.35, 0.5)
    counts = out["count"].cpu().numpy()
    for b, ref in enumerate(refs):
        rc, rf, rb = G.dets_arrays(ref)
        n = int(counts[b])
        assert n == len(ref), b
        assert np.array_equal(out["cls"][b, :n].cpu().numpy(), rc)
        assert np.array_equal(out["conf"][b, :n].cpu().numpy().astype(np.float64), rf)
        assert np.array_equal(out["bbox_xyxy"][b, :n].cpu().numpy().astype(np.float64), rb)


def test_postprocess_anchor_major_yolov5_shape(H):
    head = synth.synth_head(55, 85, 25200, 40, dup=3, anchor_major=True)
    ref = O.postprocess(head[None], O.letterbox_meta(1080, 1920, 640, 640), 0.45, 0.45)
    cls, cf, box = _post_one(H, head[None], (1080, 1920), (640, 640), 0.45, 0.45)
    rc, rf, rb = G.dets_arrays(ref)
    assert np.array_equal(cls, rc) and np.array_equal(cf, rf) and np.array_equal(box, rb)


def test_postprocess_ties_follow_documented_rule(H):
    # equal scores: the oracle (and the kernel) order them higher candidate index first
    head = synth.synth_head(56, 84, 600, 0)
    for k in range(12):
        a = 17 + 31 * k
        head[:4, a] = (60 + 45 * k, 320, 40, 40)
        head[4, a] = 1.0
        head[5 + (k % 3), a] = 0.75 if k % 2 else 0.5
    ref = O.postprocess(head[None], O.letterbox_meta(1080, 1920, 640, 640), 0.35, 0.5)
    cls, cf, box = _post_one(H, head[None], (1080, 1920), (640, 640), 0.35, 0.5)
    rc, rf, rb = G.dets_arrays(ref)
    assert len(ref) == 12
    assert np.array_equal(cls, rc) and np.array_equal(cf, rf) and np.array_equal(box, rb)


def test_postprocess_filter_fold_and_edge_shapes(H):
    from realtime_video_analytics_32streams_b200 import _native as N

    # float32(0.45) < 0.45: such a box passes the f32 gate, suppresses, but is not emitted
    head = synth.synth_head(57, 84, 300, 0)
    head[:4, 5] = (100, 300, 50, 50)
    head[4, 5] = 1.0
    head[7, 5] = np.float32(0.45)
    head[:4, 6] = (101, 300, 50, 50)
    head[4, 6] = 1.0
    head[7, 6] = 0.449  # below: never a candidate
    head[:4, 9] = (300, 300, 50, 50)
    head[4, 9] = 1.0
    head[9, 9] = 0.9
    meta = O.letterbox_meta(1080, 1920, 640, 640)
    ref = O.filter_detections(O.postprocess(head[None], meta, 0.45, 0.5), 0.45)
    cls, cf, box = _post_one(H, head[None], (1080, 1920), (640, 640), 0.45, 0.5, filter_conf=0.45)
    rc, rf, rb = G.dets_arrays(ref)
    assert len(ref) == 1
    assert np.array_equal(cls, rc) and np.array_equal(cf, rf) and np.array_equal(box, rb)
    # empty head, C == 5, C < 5
    lb = N.letterbox_meta(1080, 1920, 640, 640)
    out = H.postprocess(cu(np.zeros((2, 84, 64), np.float32)), [lb, lb], 0.35, 0.5)
    assert out["count"].cpu().tolist() == [0, 0]
    out = H.postprocess(cu(np.ones((1, 4, 64), np.float32)), [lb], 0.35, 0.5)
    assert out["count"].cpu().tolist() == [0]


def test_postprocess_additive_modes_class_aware_and_v8_native(H):
    """Not reference behaviour (its NMS is class-agnostic, its scoring uses column 4 as objectness):
    the two additive modes of the ABI against the oracle's statement of them."""
    from realtime_video_analytics_32streams_b200 import _native as N

    lb = N.letterbox_meta(1080, 1920, 640, 640)
    meta = O.letterbox_meta(1080, 1920, 640, 640)
    for seed, n_obj, dup, ncls in ((61, 40, 4, 3), (62, 300, 6, 10), (63, 25, 2, None)):
        head = synth.synth_head(seed, 84, 8400, n_obj, dup=dup, n_obj_classes=ncls, jitter=3.0)
        for v8, aware in ((False, True), (True, False), (True, True)):
            thr = 0.35 if not v8 else 0.5
            ref = O.postprocess(head[None], meta, thr, 0.5, v8_native=v8, class_aware=aware)
            out = H.postprocess(cu(head[None]), [lb], thr, 0.5, score_mode=N.SCORE_V8_NATIVE if v8 else N.SCORE_REF_COMPAT,
                                nms_mode=N.NMS_CLASS_AWARE if aware else N.NMS_AGNOSTIC)
            n = int(out["count"].cpu()[0])
            rc, rf, rb = G.dets_arrays(ref)
            assert n == len(ref) and n > 0, (seed, v8, aware)
            assert np.array_equal(out["cls"][0, :n].cpu().numpy(), rc)
            assert np.array_equal(out["conf"][0, :n].cpu().numpy().astype(np.float64), rf)
            assert np.array_equal(out["bbox_xyxy"][0, :n].cpu().numpy().astype(np.float64), rb)
    # class-aware keeps more boxes than agnostic on overlapping objects of different classes
    head = synth.synth_head(62, 84, 8400, 300, dup=6, n_obj_classes=10, jitter=3.0)
    assert len(O.postprocess(head[None], meta, 0.35, 0.5, class_aware=True)) >= len(O.postprocess(head[None], meta, 0.35, 0.5))


def test_postprocess_capacity_flag(H):
    from realtime_video_analytics_32streams_b200 import _native as N

    H.poll_status()
    head = np.zeros((1, 84, 8400), np.float32)
    head[0, 0] = np.arange(8400) % 640
    head[0, 1] = (np.arange(8400) // 640) * 40
    head[0, 2:4] = 4
    head[0, 4] = 1.0
    head[0, 5] = np.linspace(0.5, 0.99, 8400, dtype=np.float32)
    H.postprocess(cu(head), [N.letterbox_meta(1080, 1920, 640, 640)], 0.35, 0.5)
    with pytest.raises(N.B200VAError) as e:
        H.poll_status()
    assert e.value.status == N.ERR_CAPACITY
    H.poll_status()  # flags cleared


# ------------------------------------------------------------------------------------------------
# a8: tracker
# ------------------------------------------------------------------------------------------------
def test_tracker_golden_sequences_reference_api(H):
    """The reference-shaped API: Python Detection objects in, Track objects out (float64 path)."""
    from realtime_video_analytics_32streams_b200 import B200IouTracker, Detection, TrackerConfig

    z = G.load("tracker")
    for ci in z["trk_cases"].tolist():
        max_age, thr, min_hits = z[f"trk{ci}_cfg"].tolist()
        H.tracker_set_next_id(1)
        trk = B200IouTracker(TrackerConfig(max_age=int(max_age), max_iou_distance=thr, min_hits=int(min_hits)), handle=H)
        for s in range(2):
            H.tracker_reset(s)
        for fi in range(int(z[f"trk{ci}_n"][0])):
            stream = "cam%d" % int(z[f"trk{ci}_{fi}_stream"][0])
            dets = [Detection(stream, fi, int(c), float(s), tuple(b.tolist())) for c, s, b in
                    zip(z[f"trk{ci}_{fi}_dcls"], z[f"trk{ci}_{fi}_dconf"], z[f"trk{ci}_{fi}_dbox"])]
            got = G.tracks_arrays(trk.update(stream, dets))
            for k, v in got.items():
                assert np.array_equal(v, z[f"trk{ci}_{fi}_t{k}"]), (ci, fi, k)


def _moving_dets(rng, n_obj, t, pos, vel, cls, miss=0.15, dup=0.2):
    rows = []
    for o in range(n_obj):
        if rng.random() < miss:
            continue
        cx, cy = pos[o, 0] + vel[o, 0] * t, pos[o, 1] + vel[o, 1] * t
        w, h = pos[o, 2], pos[o, 3]
        for r in range(2 if rng.random() < dup else 1):
            j = rng.normal(0, 1.5, 4) if r else np.zeros(4)
            b = (np.array([cx - w / 2, cy - h / 2, cx + w / 2, cy + h / 2]) + j).astype(np.float32)
            rows.append((int(cls[o]), np.float32(rng.uniform(0.4, 1)), b))
    order = rng.permutation(len(rows))
    return [rows[i] for i in order]


def test_tracker_batched_f32_streams_share_id_counter(H):
    """8 streams per launch, float32 device detections, skips and a rescaled stream; compared with
    ONE oracle tracker updated stream by stream in batch order (tracker.py:47 shared counter)."""
    import torch
    from realtime_video_analytics_32streams_b200 import B200IouTracker, TrackerConfig

    S, n_obj, T = 8, 40, 45
    rng = np.random.default_rng(99)
    H.tracker_set_next_id(1)
    for s in range(S):
        H.tracker_reset(s)
    trk = B200IouTracker(TrackerConfig(max_age=5, max_iou_distance=0.5, min_hits=2), handle=H)
    ora = O.IouTracker(5, 0.5, 2)
    pos = [np.stack([rng.uniform(50, 1800, n_obj), rng.uniform(50, 1000, n_obj), rng.uniform(30, 120, n_obj),
                     rng.uniform(30, 120, n_obj)], 1) for _ in range(S)]
    vel = [rng.uniform(-4, 4, (n_obj, 2)) for _ in range(S)]
    cls = [rng.integers(0, 3, n_obj) for _ in range(S)]
    names = [f"s{i}" for i in range(S)]
    md = 128
    for t in range(T):
        box = np.zeros((S, md, 4), np.float32)
        conf = np.zeros((S, md), np.float32)
        cl = np.zeros((S, md), np.int32)
        cnt = np.zeros((S,), np.int32)
        skip = [1 if (t % 7 == 3 and s % 3 == 0) else 0 for s in range(S)]
        scale = [1.0 / 0.75 if s == 5 else 1.0 for s in range(S)]
        want = []
        for s in range(S):
            rows = _moving_dets(rng, n_obj, t, pos[s], vel[s], cls[s])
            cnt[s] = len(rows)
            for i, (c, f, b) in enumerate(rows):
                box[s, i], conf[s, i], cl[s, i] = b, f, c
            dets = [] if skip[s] else [O.Det(c, float(f), tuple(float(v) * scale[s] if s == 5 else float(v) for v in b))
                                       for c, f, b in rows]
            want.append(G.tracks_arrays(ora.update(names[s], dets)))
        soa = {"bbox_xyxy": cu(box), "conf": cu(conf), "cls": cu(cl), "count": cu(cnt)}
        out = trk.update_batch(names, soa, det_scale=scale, skip=skip)
        host = B200IouTracker.soa_to_host(out)
        for s in range(S):
            got = G.tracks_arrays(B200IouTracker.tracks_from_soa(host, s))
            for k, v in got.items():
                assert np.array_equal(v, want[s][k]), (t, s, k)
    H.poll_status()


@pytest.mark.parametrize("threads", [0, 512])
def test_tracker_dense_long_lived(threads, monkeypatch):
    """Config-5 shape: ~300 detections per frame against ~300+ live tracks (the dense-stream phase A: overlap keys, listed
    pairs); also with the update capped at 512 threads (B200VA_TRK_THREADS: other unit-to-warp assignment, same result)."""
    from realtime_video_analytics_32streams_b200 import B200IouTracker, TrackerConfig, _native as N

    if threads:
        monkeypatch.setenv("B200VA_TRK_THREADS", str(threads))
    H = N.Handle(device=0, max_batch=1, max_anchors=8400, max_candidates=4096, max_dets=1024, max_streams=1, max_tracks=1024)
    monkeypatch.delenv("B200VA_TRK_THREADS", raising=False)
    trk = B200IouTracker(TrackerConfig(max_age=30, max_iou_distance=0.5, min_hits=1), handle=H)
    ora = O.IouTracker(30, 0.5, 1)
    scene = synth.DenseScene(5)
    lb = N.letterbox_meta(1080, 1920, 640, 640)
    meta = O.letterbox_meta(1080, 1920, 640, 640)
    for t in range(6):
        head = scene.head(t)
        dets_o = O.filter_detections(O.postprocess(head[None], meta, 0.35, 0.5), 0.35)
        want = G.tracks_arrays(ora.update("dense", dets_o))
        soa = H.postprocess(cu(head[None]), [lb], 0.35, 0.5, filter_conf=0.35)
        host = B200IouTracker.soa_to_host(trk.update_batch(["dense"], soa))
        got = G.tracks_arrays(B200IouTracker.tracks_from_soa(host, 0))
        for k, v in got.items():
            assert np.array_equal(v, want[k]), (t, k)
        assert len(want["id"]) > 250
    H.poll_status()
    H.close()


# ------------------------------------------------------------------------------------------------
# a12: the per-stream driver, against the reference StreamWorker's recorded behaviour
# ------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("device_gates", [False, True])
def test_engine_replays_reference_stream_worker(H, device_gates):
    """``device_gates``: the motion / adaptive-FPS decisions are taken on the device (b200va_gates_decide / _commit)."""
    from test_oracle_golden import replay_pipeline
    from realtime_video_analytics_32streams_b200 import DetectorConfig, HotPathEngine, StreamConfig, TrackerConfig

    box = {}

    class W:
        def __init__(self, i, spec, cfg):
            if "streams" not in box:
                H.tracker_set_next_id(1)
                box["streams"] = []
                box["cfg"] = cfg
            box["streams"].append(StreamConfig(**{k: v for k, v in spec.items()}))
            self.i = i

        def process(self, frame, head):
            if "eng" not in box:
                cfg = box["cfg"]
                for s in range(4):
                    H.tracker_reset(s)
                box["eng"] = HotPathEngine(
                    box["streams"], DetectorConfig(confidence_threshold=cfg["conf"], iou_threshold=cfg["iou"]),
                    TrackerConfig(max_age=cfg["max_age"], max_iou_distance=cfg["thr"], min_hits=cfg["min_hits"]),
                    infer=lambda tensor: box["head"], handle=H, input_hw=cfg["input_hw"], device_gates=device_gates)
            eng = box["eng"]
            box["head"] = cu(head)
            frames = [None, None]
            frames[self.i] = frame
            res = eng.tick(frames)[0]
            st = eng.state[res.stream_name]
            return res.processed, G.tracks_arrays(res.tracks), st.process_every, st.idle_frames

    replay_pipeline(W)
