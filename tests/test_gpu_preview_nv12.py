"""The preview downscale on NV12 frames (``b200va_resize_area_u8_nv12``, ``Handle.resize_area``, ``PreviewRenderer``):
every result must equal, byte for byte, ``cv2.resize(cv2.cvtColor(frame, COLOR_YUV2BGR_NV12), .., INTER_AREA)``, restated
as ``oracle.egress.resize_area(nv12_restate.nv12_to_bgr(frame))``, and the BGR ``resize_area`` on the frame converted
on the device by ``Handle.resize`` at its own size.  ``B200KafkaSink`` and ``TickCollector`` fed NV12 frames must
publish what they publish for the ``cvtColor`` twins."""
import asyncio
import types

import numpy as np
import pytest

import nv12_restate as cvr
from oracle import egress as E
from realtime_video_analytics_32streams_b200 import synth

pytestmark = pytest.mark.gpu


def _N():
    from realtime_video_analytics_32streams_b200 import _native

    return _native


@pytest.fixture(scope="module")
def H():
    import torch

    assert torch.cuda.is_available()
    h = _N().Handle(device=0, max_batch=80, max_anchors=256, max_candidates=256, max_dets=64, max_streams=8, max_tracks=64)
    yield h
    h.close()


def _cu(a):
    import torch

    return torch.from_numpy(np.ascontiguousarray(a)).cuda()


def _nv12(seed, h, w):
    """Uniform-random NV12 frame [3H/2, W]: every Y, Cb, Cr value, so every channel saturates somewhere."""
    return np.random.default_rng(seed).integers(0, 256, size=(h * 3 // 2, w), dtype=np.uint8)


def _bgr_to_nv12(bgr):
    import cv2

    h, w = bgr.shape[:2]
    i420 = cv2.cvtColor(bgr, cv2.COLOR_BGR2YUV_I420)
    y, u, v = i420[:h], i420[h:h + h // 4].reshape(h // 2, w // 2), i420[h + h // 4:].reshape(h // 2, w // 2)
    uv = np.stack([u, v], axis=2).reshape(h // 2, w)
    return np.concatenate([y, uv])


def _check(H, nv, got, new_hw):
    """``got`` (host uint8 [h, w, 3]) against the three references for the NV12 frame ``nv``."""
    import cv2

    nh, nw = new_hw
    h = nv.shape[0] * 2 // 3
    want = E.resize_area(cvr.nv12_to_bgr(nv), nw, nh)
    assert np.array_equal(got, want), (nv.shape, new_hw, "vs oracle")
    assert np.array_equal(got, cv2.resize(cv2.cvtColor(nv, cv2.COLOR_YUV2BGR_NV12), (nw, nh), interpolation=cv2.INTER_AREA)), \
        (nv.shape, new_hw, "vs cv2")
    full = H.resize([_cu(nv)], [(h, nv.shape[1])])[0]
    assert np.array_equal(got, H.resize_area([full], [new_hw])[0].cpu().numpy()), (nv.shape, new_hw, "vs BGR entry point")


# (src_h, src_w, dst_h, dst_w): vector 2 x 2, 2 x 2 with an odd destination width, 3 x 3, 4 x 4, 1 x 2, the same size
# (cvtColor) twice, fractional ratios
GEOMS = [(216, 384, 108, 192), (64, 130, 32, 65), (216, 384, 72, 128), (216, 384, 54, 96), (216, 384, 108, 384),
         (100, 100, 100, 100), (216, 384, 216, 384), (100, 100, 37, 53), (1100, 2000, 1056, 1920), (90, 150, 30, 50)]


def test_every_path_in_one_call(H):
    frames = [_nv12(10 + i, h, w) for i, (h, w, _, _) in enumerate(GEOMS)]
    outs = H.resize_area([_cu(f) for f in frames], [(nh, nw) for _, _, nh, nw in GEOMS])
    for f, o, (_, _, nh, nw) in zip(frames, outs, GEOMS):
        _check(H, f, o.cpu().numpy(), (nh, nw))


@pytest.mark.parametrize("hw,new", [((2160, 3840), (1080, 1920)), ((1440, 2560), (1080, 1920)), ((1080, 1920), (1080, 1920))])
def test_full_size_scenes(H, hw, new):
    nv = _bgr_to_nv12(synth.MotionScene(700 + hw[0], *hw).frame(3))
    got = H.resize_area([_cu(nv)], [new])[0].cpu().numpy()
    _check(H, nv, got, new)


@pytest.mark.parametrize("geom", [(64, 128, 32, 64), (64, 128, 21, 42), (60, 100, 25, 40)])
def test_two_launch_groups(H, geom):
    """65 frames of one geometry: 64 in the first launch, 1 in the second."""
    h, w, nh, nw = geom
    frames = [_nv12(100 + i, h, w) for i in range(65)]
    outs = H.resize_area([_cu(f) for f in frames], [(nh, nw)] * 65)
    for i in (0, 31, 63, 64):
        _check(H, frames[i], outs[i].cpu().numpy(), (nh, nw))
    bgr = [_cu(cvr.nv12_to_bgr(f)) for f in frames]
    ref = H.resize_area(bgr, [(nh, nw)] * 65)
    for i, (o, r) in enumerate(zip(outs, ref)):
        assert np.array_equal(o.cpu().numpy(), r.cpu().numpy()), i


@pytest.mark.parametrize("new", [(108, 192), (72, 128), (80, 150)])
def test_plane_layouts(H, new):
    """A pitched [3H/2, W] view (aligned and 3 bytes into a row), a (y, uv) pair of separate allocations, and a chroma
    pitch that is not a multiple of 8 (off the vector path); all equal to the contiguous frame's result."""
    import torch

    h, w = 216, 384
    nv = _nv12(7, h, w)
    want = H.resize_area([_cu(nv)], [new])[0].cpu().numpy()
    _check(H, nv, want, new)
    wide = torch.zeros((h * 3 // 2, w + 24), dtype=torch.uint8, device="cuda")
    wide[:, 8:8 + w] = _cu(nv)
    odd = torch.zeros((h * 3 // 2, w + 7), dtype=torch.uint8, device="cuda")
    odd[:, 3:3 + w] = _cu(nv)
    pair = (_cu(nv[:h]), _cu(nv[h:]))
    uv_wide = torch.zeros((h // 2, w + 6), dtype=torch.uint8, device="cuda")
    uv_wide[:, :w] = _cu(nv[h:])
    odd_uv = (_cu(nv[:h]), uv_wide[:, :w])
    assert odd_uv[1].stride(0) % 8 != 0
    layouts = [wide[:, 8:8 + w], odd[:, 3:3 + w], pair, odd_uv]
    outs = H.resize_area(layouts, [new] * len(layouts))
    for k, o in enumerate(outs):
        assert np.array_equal(o.cpu().numpy(), want), k
    # an Nv12Batch is taken as it is
    nb = _N().Nv12Batch(layouts)
    for k, o in enumerate(H.resize_area(nb, [new] * len(layouts))):
        assert np.array_equal(o.cpu().numpy(), want), k


@pytest.mark.parametrize("new", [(108, 192), (72, 128), (54, 96), (37, 53), (216, 384)])
def test_saturating_values(H, new):
    """Y in 0-15 and 235-255 and Cb / Cr at 0 and 255: most converted pixels clip, so a block sum of unclipped values
    would differ from cv2's."""
    rng = np.random.default_rng(5)
    h, w = 216, 384
    y = rng.choice(np.r_[0:16, 235:256].astype(np.uint8), size=(h, w))
    uv = rng.choice(np.array([0, 255], np.uint8), size=(h // 2, w))
    nv = np.concatenate([y, uv])
    got = H.resize_area([_cu(nv)], [new])[0].cpu().numpy()
    _check(H, nv, got, new)


def test_refusals(H):
    N = _N()
    nv = _cu(_nv12(3, 64, 64))
    y, uv = nv[:64], nv[64:]
    out = _cu(np.zeros((32, 32, 3), np.uint8))

    def call(frame, sh, sw, dh, dw):
        return H.lib.b200va_resize_area_u8_nv12(H._h, (N.Nv12Frame * 1)(frame), N._int_array([sh]), N._int_array([sw]), 1,
                                                N._ptr_array([out.data_ptr()]), N._int_array([dh]), N._int_array([dw]),
                                                H._stream())

    good = N.Nv12Frame(y.data_ptr(), uv.data_ptr(), 64, 64)
    assert call(good, 64, 64, 32, 32) == N.OK
    cases = {"odd size": (good, 63, 64, 32, 32), "NULL luma": (N.Nv12Frame(None, uv.data_ptr(), 64, 64), 64, 64, 32, 32),
             "NULL chroma": (N.Nv12Frame(y.data_ptr(), None, 64, 64), 64, 64, 32, 32),
             "pitch": (N.Nv12Frame(y.data_ptr(), uv.data_ptr(), 64, 62), 64, 64, 32, 32), "enlarging": (good, 64, 64, 80, 32)}
    for name, args in cases.items():
        with pytest.raises(N.B200VAError) as e:
            H._check(call(*args))
        assert e.value.status == N.ERR_INVALID, name
    with pytest.raises(N.B200VAError) as e:
        H.resize_area([nv], [(128, 64)])
    assert e.value.status == N.ERR_INVALID and b"shrinking" in H.lib.b200va_last_error(H._h)


class _Producer:
    def __init__(self):
        self.sent = []

    async def send_and_wait(self, topic, body):
        self.sent.append((topic, body))


def _sink_cfg():
    return type("Cfg", (), dict(enabled=True, include_frames=True, frame_quality=75, topic="analytics",
                                bootstrap_servers="x", linger_ms=10, max_batch_size=16384))()


_SCENES = {}


def _scene_nv12(hw):
    if hw not in _SCENES:
        _SCENES[hw] = _bgr_to_nv12(synth.MotionScene(800 + hw[0], *hw).frame(1))
    return _SCENES[hw]


@pytest.mark.parametrize("how", ["host", "cuda", "pair"])
@pytest.mark.parametrize("hw", [(2160, 3840), (720, 1280)])
@pytest.mark.parametrize("overlap", [False, True])
def test_sink_send_tracks(H, monkeypatch, how, hw, overlap):
    """B200KafkaSink.send_tracks with include_frames on an NV12 frame: the pre-encode image and the whole message body
    equal those of the same call on the cvtColor frame, on the GPU drawing path and on the in-order replay."""
    import cv2
    from realtime_video_analytics_32streams_b200 import sinks
    from realtime_video_analytics_32streams_b200.types import Track

    nv = _scene_nv12(hw)
    h, w = hw
    frame = {"host": nv, "cuda": _cu(nv), "pair": (_cu(nv[:h]), _cu(nv[h:]))}[how]
    twin = cv2.cvtColor(nv, cv2.COLOR_YUV2BGR_NV12)
    s = w / 3840
    if overlap:  # the second box's outline runs through the first box's label
        boxes = [(400 * s, 400 * s, 900 * s, 900 * s), (420 * s, 380 * s, 1000 * s, 1000 * s)]
    else:
        boxes = [(100 * s, 200 * s, 600 * s, 700 * s), (2000 * s, 1000 * s, 3000 * s, 1800 * s)]
    tracks = [Track(7 + k, 2 + k, 0.9 - 0.1 * k, tuple(float(v) for v in b), 0, 1) for k, b in enumerate(boxes)]
    sinks_ = [sinks.B200KafkaSink(_sink_cfg(), handle=H, producer=_Producer()) for _ in range(2)]
    captured = []
    real = cv2.imencode
    monkeypatch.setattr(cv2, "imencode", lambda ext, img, params=None: (captured.append((ext, img.copy())), real(ext, img, params))[1])
    for sink, f in zip(sinks_, (frame, twin)):
        asyncio.run(sink.send_tracks("cam-nv12", 42, tracks, frame=f))
    assert len(captured) == 2
    (ext_n, img_n), (ext_b, img_b) = captured
    assert ext_n == ext_b and img_n.shape == img_b.shape and np.array_equal(img_n, img_b)
    assert img_n.shape[:2] == ((1080, 1920) if h > 1080 else hw)
    body_n, body_b = sinks_[0]._producer.sent[0][1], sinks_[1]._producer.sent[0][1]
    assert b'"frame_jpeg": "data:image/' in body_n and body_n == body_b
    assert sinks_[0]._renderer.replayed == sinks_[1]._renderer.replayed == (1 if overlap else 0)


class _Recorder:
    def update_counters(self, **kw):
        pass


class _Health:
    def update_success(self, dt):
        pass

    def update_error(self):
        pass


def test_collector_events_carry_the_preview():
    """TickCollector over a real HotPathEngine fed host NV12 packets: every processed event carries frame_jpeg, and
    every published body equals the run on the cvtColor twins."""
    import cv2
    import torch
    from realtime_video_analytics_32streams_b200 import DetectorConfig, HotPathEngine, StreamConfig, TrackerConfig, sinks
    from realtime_video_analytics_32streams_b200.collector import TickCollector, make_process_packet

    in_hw, n_ticks = (64, 64), 6
    sizes = [(2160, 3840), (720, 1280), (216, 384), (216, 384)]
    scenes = [synth.MotionScene(900 + i, *hw, rect=40, speed=9) for i, hw in enumerate(sizes)]
    nv = [[_bgr_to_nv12(sc.frame(t)) for sc in scenes] for t in range(n_ticks)]
    twins = [[cv2.cvtColor(f, cv2.COLOR_YUV2BGR_NV12) for f in fs] for fs in nv]

    def run(frames_of):
        h = _N().Handle(device=0, max_batch=len(sizes), max_anchors=256, max_candidates=256, max_dets=64,
                        max_streams=len(sizes), max_tracks=128)
        try:
            streams = [StreamConfig(name=f"cam{i}") for i in range(len(sizes))]
            tick = {"t": 0}
            eng = HotPathEngine(streams, DetectorConfig(confidence_threshold=0.35, iou_threshold=0.5),
                                TrackerConfig(max_age=3, max_iou_distance=0.5, min_hits=1),
                                infer=lambda tensor: torch.from_numpy(np.concatenate(
                                    [synth.synth_head(5000 + 10 * tick["t"] + i, 20, 256, 4, dup=2, input_hw=in_hw)[None]
                                     for i in eng.active_streams])).to(h.device),
                                handle=h, input_hw=in_hw)
            prod = _Producer()
            sink = sinks.B200KafkaSink(_sink_cfg(), handle=h, producer=prod)
            sink._frame_send_interval = 0
            col = TickCollector(eng, max_wait_s=5.0)
            proc = make_process_packet(lambda wk: col)
            workers = [types.SimpleNamespace(ctx=types.SimpleNamespace(metrics=_Recorder(), kafka=sink, health=_Health()),
                                             _frame_index=0, _maybe_save_snapshot=lambda *a, **k: None, _process_every=1,
                                             _idle_frames=0) for _ in streams]

            async def drive():
                for t in range(n_ticks):
                    tick["t"] = t
                    await asyncio.gather(*[proc(wk, types.SimpleNamespace(stream=s, frame=frames_of[t][i], frame_id=t))
                                           for i, (s, wk) in enumerate(zip(streams, workers))])
                await col.close()

            asyncio.run(drive())
            h.poll_status()
            return sorted(prod.sent, key=lambda m: m[1])
        finally:
            h.close()

    got, want = run(nv), run(twins)
    assert len(got) == len(sizes) * n_ticks
    assert all(b'"frame_jpeg": "data:image/' in body for _, body in got)
    assert got == want
