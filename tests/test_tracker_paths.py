"""CPU checks of the tracker path predictor (tests/tracker_paths.py) and of the oracle's NaN semantics, which the GPU
tracker tests (tests/test_gpu_tracker.py) build on."""
import os
import re

from oracle import hotpath as O

import tracker_paths as P

BODY = os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "realtime_video_analytics_32streams_b200",
                    "csrc", "tracker_body.cuh")
NAN = float("nan")


def test_predictor_constants_match_the_kernel():
    src = open(BODY).read()
    for name, value in (("kDetChunk", P.DET_CHUNK), ("kTrkPairs", P.TRK_PAIRS), ("kTrkThreadsMin", P.THREADS_MIN),
                        ("kTrkSmemRowsMax", P.SMEM_ROWS_MAX), ("kCand", P.CAND)):
        assert re.search(rf"constexpr int {name} = {value};", src), name
    # the choices the predictor restates, as the kernel writes them
    assert "const int G = nblk >= 16 ? 2 : (nblk >= 8 ? 4 : 8);" in src
    assert "if (SMALL || pairs <= min(kTrkPairs, 8 * kTrkThreads)) {" in src
    assert "((T0 > 96 || D > 64) ? wide : kTrkThreadsMin)" in src
    assert "D <= kDetChunk && D * (T0 + D) <= 8 * kTrkThreadsMin" in src
    assert "pre_T0 <= kNmsThreadsSmall" in open(os.path.join(os.path.dirname(BODY), "postprocess.cu")).read()


def test_unit_group_boundaries():
    # G = 8 up to 384 tracks at chunk start, G = 4 from 385 to 896, G = 2 from 897
    for tc, want in ((100, "units-G8"), (384, "units-G8"), (385, "units-G4"), (896, "units-G4"), (897, "units-G2"),
                     (4000, "units-G2")):
        assert P.phase_a(64, tc, 512) == want, tc
    # few pairs: nd * Tc + nd^2 <= min(2048, 8 * width)
    assert P.phase_a(20, 82, 256) == "few" and P.phase_a(20, 83, 256) == "units-G8"
    assert P.phase_a(1, 2047, 256) == "few" and P.phase_a(1, 2048, 256) == "units-G2"
    assert P.phase_a(1, 2048, 1024) == "units-G2"  # the list holds 2048 pairs however wide the launch


def test_small_and_table_choices():
    assert P.predict(40, 20, 512, 256, fused=True) == P.Path("small-staged", "shared", "few", 256)
    assert P.predict(300, 6, 512, 256, fused=True) == P.Path("small", "shared", "few", 256)
    assert P.predict(300, 6, 300, 256, fused=True).kind == "general"  # does not fit the launch's table
    assert P.predict(300, 7, 512, 256, fused=True).kind == "general"  # 7 * 307 > 2048
    assert P.predict(40, 20, 512, 512) == P.Path("general", "shared", "few", 256)  # k_tracker has no small path
    assert P.predict(96, 64, 512, 1024).width == 256 and P.predict(97, 64, 512, 1024).width == 1024
    assert P.predict(0, 65, 512, 512).width == 512
    assert P.predict(3000, 72, 3072, 512).table == "shared" and P.predict(3000, 73, 3072, 512).table == "global"
    assert P.predict(300, 40, 8, 256, fused=True) == P.Path("general", "global", "units-G8", 256)


def test_oracle_iou_takes_the_track_coordinate_for_a_nan_of_the_detection():
    """tracker.py's builtin min / max return the first argument (the track's coordinate) when the second is NaN."""
    t = (0.0, 0.0, 10.0, 10.0)
    assert O.iou_f64(t, (NAN, 0.0, NAN, 5.0)) == 1.0
    assert O.iou_f64(t, (NAN, 0.0, 8.0, 10.0)) == 4.0  # area 0, union 20
    assert O.iou_f64(t, (2.0, 0.0, NAN, 10.0)) == 4.0
    assert O.iou_f64(t, (NAN, 0.0, 10.0, 10.0)) == 0.0  # union 0
    assert O.iou_f64(t, (NAN, NAN, NAN, NAN)) == 0.0
    # a NaN of the track empties the intersection
    for k in range(4):
        b = list(t)
        b[k] = NAN
        assert O.iou_f64(tuple(b), (0.0, 0.0, 8.0, 10.0)) == 0.0


def test_oracle_tracker_matches_a_nan_detection():
    ref = O.IouTracker(30, 0.5, 0)
    ref.update("s", [O.Det(0, 0.9, (0.0, 0.0, 10.0, 10.0))])
    got = ref.update("s", [O.Det(0, 0.8, (NAN, 0.0, NAN, 5.0))])
    assert [(t.track_id, t.hits) for t in got] == [(1, 2)]
    # the track now carries the NaN box: the same detection again starts a new track
    got = ref.update("s", [O.Det(0, 0.8, (0.0, 0.0, 10.0, 10.0))])
    assert [(t.track_id, t.hits) for t in got] == [(1, 2), (2, 1)]


def test_update_refuses_more_than_32768_detections_before_staging():
    """``B200IouTracker.update`` refuses an oversized call before its staging buffer grows (the buffer's row count is
    the max_dets of every later call) and without touching the device; the limit is the kernel's."""
    import types

    import pytest

    from realtime_video_analytics_32streams_b200 import _native as N
    from realtime_video_analytics_32streams_b200.tracker import B200IouTracker

    assert re.search(rf"constexpr int kTrkMaxDets = {N.TRACKER_MAX_DETS};", open(BODY).read())
    trk = B200IouTracker(None, handle=types.SimpleNamespace(torch=None))
    dets = [O.Det(0, 0.5, (0.0, 0.0, 1.0, 1.0))] * (N.TRACKER_MAX_DETS + 1)
    with pytest.raises(N.B200VAError) as e:
        trk.update("s", dets)
    assert e.value.status == N.ERR_INVALID
    assert trk._in is None
