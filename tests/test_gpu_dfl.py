"""k_dfl_decode (b200va_dfl_decode) against the float64 decode of oracle/dfl.py, at the shapes and values where a
DFL decode goes wrong.

b200va_dfl_decode picks one of four instantiations: k_dfl_decode<16, 4> and <16, 1> (reg_max 16, bins unrolled) and
<0, 4> and <0, 1> (any other reg_max, bins in a run-time loop); VEC = 4 (a thread owns four consecutive anchors, each
looking up its own level) when A % 4 == 0 and raw and out are 16-byte aligned.  Every call records with
torch.profiler which instantiation ran and asserts it is the intended one; the last test asserts that all four ran.

Exact cases -- uniform bins (d = (R - 1) / 2), one-hot bins (d = k), two equal winners (d = (k + k') / 2), class
logits whose sigmoid is 0, 0.5, 1 or NaN -- are compared bit for bit with the float64 result rounded once to float32.
Everything else is compared element by element with the float64 decode under the bound of tests/dfl_bound.py.
Every `out` lies between sentinel words that must come back untouched."""

import ctypes as C

import numpy as np
import pytest

import dfl_bound as DB
from oracle import dfl as D
from oracle import hotpath as O

pytestmark = pytest.mark.gpu

F32 = np.float32
REG_MAX = (1, 2, 7, 16, 17, 32, 64)
KERNELS = ("k_dfl_decode<16,4>", "k_dfl_decode<16,1>", "k_dfl_decode<0,4>", "k_dfl_decode<0,1>")
SEEN = set()  # instantiations observed by the profiler in this module
GUARD = 16  # sentinel floats before and after every `out`
SENTINEL = 0x7FA5A5A5

# (levels, strides); the strides keep every exact case's products exact
GEOMS = {
    "640": (((80, 80), (40, 40), (20, 20)), (8.0, 16.0, 32.0)),  # 8400
    "1280": (((160, 160), (80, 80), (40, 40)), (8.0, 16.0, 32.0)),  # 33600
    "12x20": (((12, 20), (6, 10)), (8.0, 16.0)),  # 300
    "5x7": (((5, 7), (3, 5)), (8.0, 16.0)),  # 50: A % 4 == 2
    "eight": (((7, 9), (1, 1), (1, 13), (11, 1), (4, 6), (2, 2), (3, 1), (1, 5)),
              (8.0, 16.0, 32.0, 12.0, 0.75, 64.0, 4.0, 24.0)),  # 124: a 1x1 level, a 1xW row, an Hx1 column
    # A % 4 == 0 with level boundaries inside a thread's group of four anchors
    "cut16": (((3, 5), (1, 1)), (8.0, 16.0)),
    "cut8": (((2, 3), (1, 2)), (12.0, 0.75)),
    "cut4": (((1, 1), (1, 3)), (32.0, 8.0)),
    "a29": (((5, 5), (2, 2)), (8.0, 16.0)),  # A % 4 == 1
    "a19": (((3, 5), (2, 2)), (0.75, 12.0)),  # A % 4 == 3
    "a1": (((1, 1),), (32.0,)),
}
# class logits with an exact sigmoid: 0.5, 0.5, 1, 0, NaN, and 1 for x >= 20
CLS_EXACT = np.array([0.0, -0.0, np.inf, -np.inf, np.nan, 20.0, 25.5, 1e4, 3e38], F32)
# class logits whose sigmoid is subnormal or flushed by expf's overflow, and around it
CLS_TINY = np.array([-80.0, -87.3, -87.4, -88.5, -88.8, -95.0, -103.9, -104.0, -1e30], F32)


@pytest.fixture(scope="module")
def H():
    import torch
    from realtime_video_analytics_32streams_b200 import _native

    assert torch.cuda.is_available()
    h = _native.Handle(device=0, max_batch=128, max_anchors=8400, max_candidates=4096, max_dets=1024,
                       max_streams=2, max_tracks=64)
    yield h
    h.poll_status()
    h.close()


def _a(geom):
    return sum(h * w for h, w in GEOMS[geom][0])


def _expect(reg_max, a, raw_ptr, out_ptr):
    vec = a % 4 == 0 and raw_ptr % 16 == 0 and out_ptr % 16 == 0
    return f"k_dfl_decode<{16 if reg_max == 16 else 0},{4 if vec else 1}>"


def run(H, raw, nc, reg_max, geom, raw_off=0, out_off=0, dev=False):
    """H.dfl_decode of host `raw` [B, 4 reg_max + nc, A] with raw and out views raw_off / out_off bytes into larger
    buffers and out between sentinel words.  Asserts the intended instantiation ran and the sentinels survived;
    returns the host result (and the device `out` with dev=True)."""
    import torch
    from torch.profiler import ProfilerActivity, profile

    levels, strides = GEOMS[geom]
    b, cin, a = raw.shape
    assert cin == 4 * reg_max + nc and a == _a(geom)
    rbuf = torch.zeros(raw.size + 4, dtype=torch.float32, device="cuda")
    rv = rbuf[raw_off // 4:raw_off // 4 + raw.size].view(raw.shape)
    rv.copy_(torch.from_numpy(np.ascontiguousarray(raw, F32)))
    n = b * (4 + nc) * a
    obuf = torch.full((n + 2 * GUARD + 4,), SENTINEL, dtype=torch.int32, device="cuda").view(torch.float32)
    o0 = GUARD + out_off // 4
    ov = obuf[o0:o0 + n].view(b, 4 + nc, a)
    assert rv.data_ptr() % 16 == raw_off and ov.data_ptr() % 16 == out_off
    expect = _expect(reg_max, a, rv.data_ptr(), ov.data_ptr())
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        ret = H.dfl_decode(rv, nc, reg_max, levels, strides, out=ov)
        torch.cuda.synchronize()
    assert ret is ov
    names = {e.name.replace(" ", "") for e in prof.events() if "k_dfl_decode" in e.name}
    ran = {k for k in KERNELS if any(k in nm for nm in names)}
    SEEN.update(ran)
    assert ran == {expect}, (expect, sorted(names))
    words = obuf.view(torch.int32).cpu().numpy()
    assert (words[:o0] == SENTINEL).all() and (words[o0 + n:] == SENTINEL).all(), "write outside `out`"
    host = words[o0:o0 + n].view(F32).reshape(b, 4 + nc, a)
    return (host, ov) if dev else host


def ref64(raw, nc, reg_max, geom):
    levels, strides = GEOMS[geom]
    return D.dfl_decode(raw, nc, reg_max, levels, strides, dtype=np.float64)


def same_bits(got, want):
    """Equal as float32 bit patterns (signed zeros distinct), NaN positions equal."""
    got = np.asarray(got, F32)
    want = np.asarray(want, np.float64).astype(F32)
    gn, wn = np.isnan(got), np.isnan(want)
    return np.array_equal(gn, wn) and np.array_equal(got[~gn].view(np.uint32), want[~wn].view(np.uint32))


def assert_within(got, want64, reg_max, geom, what):
    levels, strides = GEOMS[geom]
    r = DB.error_ratio(got, want64, reg_max, levels, strides)
    w, at = DB.worst(r)
    assert w <= 1.0, f"{what}: largest error {w:.3g} x the bound at {at}: got {got[at]!r}, float64 {want64[at]!r}"
    return w


def _cls_exact(rng, b, nc, a):
    return CLS_EXACT[rng.integers(len(CLS_EXACT), size=(b, nc, a))]


# ---- exact cases ------------------------------------------------------------------------------------------------

@pytest.mark.parametrize("geom", list(GEOMS))
def test_uniform_bins_map_every_anchor(H, geom):
    """Equal bins on every side: d = (R - 1) / 2, so cx = ax s, cy = ay s, w = h = (R - 1) s exactly -- a bit-exact
    map of every anchor's point and level."""
    levels, strides = GEOMS[geom]
    a = _a(geom)
    anchors, st = D.make_anchors(levels, strides, np.float64)
    b = 1 if a > 10000 else 2
    for reg_max in (REG_MAX if a < 10000 else (1, 16, 17)):
        rng = np.random.default_rng(reg_max * 131 + a)
        nc = (0, 1, 7, 8, 9)[reg_max % 5]
        side = rng.normal(0, 3, size=(b, 4, 1, a)).astype(F32)
        side[..., ::5] = 3e38
        side[..., 1::5] = -3e38
        side[..., 2::5] = 1000.0
        raw = np.concatenate([np.broadcast_to(side, (b, 4, reg_max, a)).reshape(b, 4 * reg_max, a),
                              _cls_exact(rng, b, nc, a)], 1)
        got = run(H, raw, nc, reg_max, geom)
        want = ref64(raw, nc, reg_max, geom)
        assert same_bits(got, want), (geom, reg_max)
        closed = np.stack([anchors[0] * st, anchors[1] * st, (reg_max - 1) * st, (reg_max - 1) * st])
        assert same_bits(got[:, :4], np.broadcast_to(closed, (b, 4, a))), (geom, reg_max)


def _peaked(seed, b, reg_max, nc, a, pair):
    """One-hot bins: the winner k = (3 anchor + 5 side + 7 frame) mod R holds 0, +1000 or 3e38, the losers -1e4 or
    -3e38 (with 3e38 winning, x - m overflows to -inf).  pair=True: on a third of the sides a second winner k' != k
    holds the same logit.  Returns raw and the exact d [B, 4, A]."""
    rng = np.random.default_rng(seed)
    an = np.arange(a)[None, None, :]
    sd = np.arange(4)[None, :, None]
    fr = np.arange(b)[:, None, None]
    k = (3 * an + 5 * sd + 7 * fr) % reg_max
    win = np.array([0.0, 1000.0, 3e38], F32)[(an + fr) % 3]
    lose = np.array([-1e4, -3e38], F32)[(an // 3 + sd) % 2]
    box = np.broadcast_to(lose[:, :, None, :], (b, 4, reg_max, a)).copy()
    ii = np.indices((b, 4, a))
    box[ii[0], ii[1], k, ii[2]] = np.broadcast_to(win, (b, 4, a))
    d = k.astype(np.float64)
    if pair and reg_max > 1:
        two = np.broadcast_to((an + sd + fr) % 3 == 0, (b, 4, a))
        k2 = (k + 1 + an % (reg_max - 1)) % reg_max
        k2 = np.broadcast_to(k2, (b, 4, a))
        box[ii[0][two], ii[1][two], k2[two], ii[2][two]] = np.broadcast_to(win, (b, 4, a))[two]
        d = np.where(two, (np.broadcast_to(k, (b, 4, a)) + k2) / 2.0, np.broadcast_to(d, (b, 4, a)))
    d = np.broadcast_to(d, (b, 4, a))
    raw = np.concatenate([box.reshape(b, 4 * reg_max, a), _cls_exact(rng, b, nc, a)], 1)
    return raw, d


@pytest.mark.parametrize("reg_max", REG_MAX)
@pytest.mark.parametrize("pair", [False, True], ids=["one_hot", "two_winners"])
def test_peaked_bins_exact(H, reg_max, pair):
    """d = k (or (k + k') / 2) exactly: checks the side order l, t, r, b, the bin weights and the max shift."""
    for geom, b in (("640", 1), ("eight", 3), ("a19", 3)):
        levels, strides = GEOMS[geom]
        a = _a(geom)
        nc = 3
        raw, d = _peaked(reg_max + 17 * b, b, reg_max, nc, a, pair)
        got = run(H, raw, nc, reg_max, geom)
        want = ref64(raw, nc, reg_max, geom)
        anchors, st = D.make_anchors(levels, strides, np.float64)
        x1, y1, x2, y2 = anchors[0] - d[:, 0], anchors[1] - d[:, 1], anchors[0] + d[:, 2], anchors[1] + d[:, 3]
        closed = np.stack([(x1 + x2) / 2 * st, (y1 + y2) / 2 * st, (x2 - x1) * st, (y2 - y1) * st], 1)
        assert np.array_equal(want[:, :4], closed), (geom, reg_max)  # the input holds the d it was built for
        assert same_bits(got, want), (geom, reg_max, pair)


# ---- non-finite bins --------------------------------------------------------------------------------------------

@pytest.mark.parametrize("reg_max", REG_MAX)
def test_nonfinite_bins(H, reg_max):
    """d is NaN iff a bin is NaN or +inf, or all bins are -inf; a NaN side poisons exactly its two outputs; a -inf bin
    among finite ones has weight 0 (bit-identical to -3e38 there)."""
    for geom, b in (("eight", 2), ("5x7", 3)):
        a = _a(geom)
        nc = 9
        rng = np.random.default_rng(reg_max * 7 + a)
        raw = rng.normal(0, 2.5, size=(b, 4 * reg_max + nc, a)).astype(F32)
        raw[:, 4 * reg_max:][rng.random((b, nc, a)) < 0.1] = np.nan
        box = raw[:, :4 * reg_max].reshape(b, 4, reg_max, a)  # a view
        kind = rng.integers(0, 8, size=(b, 4, a))
        if reg_max == 1:
            kind[kind == 7] = 0
        nan_side = np.zeros((b, 4, a), bool)
        neg_inf_only = np.zeros(box.shape, bool)  # -inf bins among finite ones
        for f, s, i in zip(*np.nonzero(kind >= 3)):
            k = int(rng.integers(reg_max))
            if kind[f, s, i] == 3:
                box[f, s, k, i] = np.nan
            elif kind[f, s, i] == 4:
                box[f, s, k, i] = np.inf
            elif kind[f, s, i] == 5:
                box[f, s, :, i] = -np.inf
            elif kind[f, s, i] == 6:
                box[f, s, :, i] = [(np.nan, np.inf, -np.inf)[j % 3] for j in range(reg_max)]
            else:
                ks = rng.permutation(reg_max)[:int(rng.integers(1, reg_max))]
                box[f, s, ks, i] = -np.inf
                neg_inf_only[f, s, ks, i] = True
                continue
            nan_side[f, s, i] = True
        got = run(H, raw, nc, reg_max, geom)
        want = ref64(raw, nc, reg_max, geom)
        lr, tb = nan_side[:, 0] | nan_side[:, 2], nan_side[:, 1] | nan_side[:, 3]
        expect_nan = np.stack([lr, tb, lr, tb], 1)
        assert np.array_equal(np.isnan(want[:, :4]), expect_nan)
        assert np.array_equal(np.isnan(got[:, :4]), expect_nan), (geom, reg_max)
        assert_within(got, want, reg_max, geom, f"non-finite bins, {geom}, reg_max {reg_max}")
        if neg_inf_only.any():
            raw2 = raw.copy()
            raw2[:, :4 * reg_max].reshape(b, 4, reg_max, a)[neg_inf_only] = -3e38
            got2 = run(H, raw2, nc, reg_max, geom)
            assert np.array_equal(got.view(np.uint32), got2.view(np.uint32)), (geom, reg_max)


# ---- random logits ----------------------------------------------------------------------------------------------

@pytest.mark.parametrize("reg_max", REG_MAX)
def test_random_logits_within_bound(H, reg_max):
    worst = []
    for scale in (0.5, 2.5, 20.0):
        for geom, b, nc in (("640", 1, 80), ("a29", 3, 17)):
            rng = np.random.default_rng(int(scale * 10) + reg_max * 1000 + b)
            raw = rng.normal(0, scale, size=(b, 4 * reg_max + nc, _a(geom))).astype(F32)
            got = run(H, raw, nc, reg_max, geom)
            worst.append(assert_within(got, ref64(raw, nc, reg_max, geom), reg_max, geom,
                                       f"normal({scale}) logits, {geom}, reg_max {reg_max}"))
    print(f"reg_max {reg_max}: largest error {max(worst):.3f} x the bound")


@pytest.mark.parametrize("nc", (0, 1, 7, 8, 9, 16, 17, 80, 81, 600))
def test_class_counts(H, nc):
    """Class counts that start or cut an 8-row class block differently, in every instantiation; scores hold the exact
    and the subnormal edges of the sigmoid."""
    for reg_max, geom in ((16, "640"), (16, "5x7"), (7, "eight"), (17, "a29")):
        a = _a(geom)
        rng = np.random.default_rng(nc * 3 + reg_max + a)
        raw = rng.normal(0, 4, size=(2, 4 * reg_max + nc, a)).astype(F32)
        cls = raw[:, 4 * reg_max:]
        pick = rng.random(cls.shape)
        exact = pick < 0.15
        cls[exact] = CLS_EXACT[rng.integers(len(CLS_EXACT), size=int(exact.sum()))]
        tiny = (pick >= 0.15) & (pick < 0.25)
        cls[tiny] = CLS_TINY[rng.integers(len(CLS_TINY), size=int(tiny.sum()))]
        got = run(H, raw, nc, reg_max, geom)
        want = ref64(raw, nc, reg_max, geom)
        assert_within(got, want, reg_max, geom, f"nc {nc}, {geom}, reg_max {reg_max}")
        assert same_bits(got[:, 4:][exact], want[:, 4:][exact]), (nc, geom)


# ---- alignment and batches ----------------------------------------------------------------------------------------

@pytest.mark.parametrize("reg_max", (16, 7))
def test_misaligned_views(H, reg_max):
    """raw and out as views 0, 4, 8, 12 bytes into larger buffers with A % 4 == 0: misalignment alone selects the
    one-anchor instantiation, which computes bit for bit what the four-anchor one does."""
    geom, nc = "eight", 9
    rng = np.random.default_rng(reg_max)
    raw = rng.normal(0, 2.5, size=(3, 4 * reg_max + nc, _a(geom))).astype(F32)
    want = ref64(raw, nc, reg_max, geom)
    aligned = run(H, raw, nc, reg_max, geom)
    assert_within(aligned, want, reg_max, geom, "aligned")
    for ro, oo in ((4, 0), (8, 0), (12, 0), (0, 4), (0, 8), (0, 12), (12, 4)):
        got = run(H, raw, nc, reg_max, geom, raw_off=ro, out_off=oo)
        assert np.array_equal(got.view(np.uint32), aligned.view(np.uint32)), (reg_max, ro, oo)


def test_batch_32_full_frames(H):
    """32 frames of [144, 8400], each different, compared in full."""
    rng = np.random.default_rng(32)
    raw = rng.normal(0, 2.5, size=(32, 144, 8400)).astype(F32)
    raw += rng.normal(0, 1, size=(32, 1, 1)).astype(F32)
    got = run(H, raw, 80, 16, "640")
    assert_within(got, ref64(raw, 80, 16, "640"), 16, "640", "32 frames")


@pytest.mark.parametrize("reg_max,geom", [(7, "cut16"), (16, "5x7"), (16, "cut8"), (17, "a19")])
def test_batch_many_small_frames(H, reg_max, geom):
    """67 small frames, every frame's content different, so a frame mix-up shows."""
    rng = np.random.default_rng(reg_max + _a(geom))
    raw = rng.normal(0, 2.5, size=(67, 4 * reg_max + 5, _a(geom))).astype(F32)
    got = run(H, raw, 5, reg_max, geom)
    assert_within(got, ref64(raw, 5, reg_max, geom), reg_max, geom, f"67 frames, {geom}")


# ---- composition --------------------------------------------------------------------------------------------------

@pytest.mark.parametrize("aware", [False, True], ids=["agnostic", "class_aware"])
def test_composition_with_postprocess(H, aware):
    """The decoded tensor feeds b200va_postprocess (SCORE_V8_NATIVE) unchanged: classes, confidences and boxes equal
    oracle.hotpath.postprocess(v8_native=True) on a host copy of the kernel's own output, bit for bit."""
    import torch
    from realtime_video_analytics_32streams_b200 import _native as N

    for geom, b, nc, mu, src, net in (("12x20", 3, 21, -3.0, (96, 160), (96, 160)),
                                      ("640", 2, 80, -8.0, (1080, 1920), (640, 640))):
        rng = np.random.default_rng(nc)
        raw = rng.normal(0, 2.5, size=(b, 64 + nc, _a(geom))).astype(F32)
        raw[:, 64:] = rng.normal(mu, 2.0, size=(b, nc, _a(geom))).astype(F32)
        host, dev = run(H, raw, nc, 16, geom, dev=True)
        out = H.postprocess(dev, [N.letterbox_meta(*src, *net)] * b, 0.25, 0.5, layout=N.HEAD_CHANNEL_MAJOR,
                            score_mode=N.SCORE_V8_NATIVE, nms_mode=N.NMS_CLASS_AWARE if aware else N.NMS_AGNOSTIC)
        torch.cuda.synchronize()
        for i in range(b):
            ref = O.postprocess(host[i][None], O.letterbox_meta(*src, *net), 0.25, 0.5, v8_native=True,
                                class_aware=aware, layout="cm")
            n = int(out["count"][i].item())
            assert n == len(ref) and n > 0, (geom, i, n, len(ref))
            assert out["cls"][i, :n].cpu().numpy().tolist() == [d.class_id for d in ref], (geom, i)
            assert np.array_equal(out["conf"][i, :n].cpu().numpy().astype(np.float64),
                                  np.array([d.confidence for d in ref], np.float64)), (geom, i)
            assert np.array_equal(out["bbox_xyxy"][i, :n].cpu().numpy().astype(np.float64),
                                  np.array([d.bbox_xyxy for d in ref], np.float64).reshape(-1, 4)), (geom, i)
    H.poll_status()


# ---- refusals -----------------------------------------------------------------------------------------------------
# Every wrong `out` below holds at least B (4 + nc) A float32s, so a call that does not refuse it writes only inside it.

@pytest.mark.parametrize("case", ["float64", "extra_anchors", "non_contiguous", "host"])
def test_wrong_out_refused(H, case):
    import torch

    levels, strides = GEOMS["cut16"]
    b, nc, reg_max, a = 2, 3, 7, 16
    raw = torch.zeros((b, 4 * reg_max + nc, a), dtype=torch.float32, device="cuda")
    out = {"float64": lambda: torch.zeros((b, 4 + nc, a), dtype=torch.float64, device="cuda"),
           "extra_anchors": lambda: torch.zeros((b, 4 + nc, a + 4), dtype=torch.float32, device="cuda"),
           "non_contiguous": lambda: torch.zeros((b, a, 4 + nc), dtype=torch.float32, device="cuda").transpose(1, 2),
           "host": lambda: torch.zeros((b, 4 + nc, a), dtype=torch.float32).pin_memory()}[case]()
    try:
        with pytest.raises(ValueError):
            H.dfl_decode(raw, nc, reg_max, levels, strides, out=out)
    finally:
        torch.cuda.synchronize()


@pytest.mark.parametrize("n_strides", [1, 3])
def test_strides_must_match_levels(H, n_strides):
    import torch

    levels = GEOMS["cut16"][0]
    raw = torch.zeros((1, 4 * 16 + 2, 16), dtype=torch.float32, device="cuda")
    try:
        with pytest.raises(ValueError):
            H.dfl_decode(raw, 2, 16, levels, (8.0, 16.0, 32.0)[:n_strides])
    finally:
        torch.cuda.synchronize()


@pytest.mark.parametrize("case", ["reg_max_0", "reg_max_65", "nine_levels", "empty_level"])
def test_geometry_refused(H, case):
    import torch
    from realtime_video_analytics_32streams_b200 import _native as N

    reg_max, levels = {"reg_max_0": (0, ((2, 2),)), "reg_max_65": (65, ((2, 2),)),
                       "nine_levels": (16, ((1, 1),) * 9), "empty_level": (16, ((2, 2), (0, 3)))}[case]
    a = sum(h * w for h, w in levels)
    raw = torch.zeros((1, 4 * reg_max + 2, a), dtype=torch.float32, device="cuda")
    with pytest.raises(N.B200VAError) as e:
        H.dfl_decode(raw, 2, reg_max, levels, (8.0,) * len(levels))
    assert e.value.status == N.ERR_INVALID


def test_anchor_total_beyond_int_refused(H):
    """One 65536 x 65536 level: 2**32 anchors, which a 32-bit count wraps to exactly 0."""
    import torch
    from realtime_video_analytics_32streams_b200 import _native as N

    raw = torch.zeros(64, dtype=torch.float32, device="cuda")
    out = torch.zeros(64, dtype=torch.float32, device="cuda")
    hw = (C.c_int * 2)(65536, 65536)
    st = (C.c_float * 1)(8.0)
    rc = N.load_library().b200va_dfl_decode(H._h, C.c_void_p(raw.data_ptr()), 1, 0, 1, hw, st, 1,
                                            C.c_void_p(out.data_ptr()), H._stream())
    torch.cuda.synchronize()
    assert rc == N.ERR_INVALID, rc


def test_every_instantiation_ran():
    """The cases above reached all four k_dfl_decode instantiations (recorded with torch.profiler)."""
    assert SEEN == set(KERNELS), sorted(SEEN)
