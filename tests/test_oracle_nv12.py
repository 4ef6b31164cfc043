"""NV12 on the CPU: ``nv12_restate.nv12_to_bgr`` against the installed ``cv2.cvtColor(COLOR_YUV2BGR_NV12)`` for
every (Y, Cb, Cr) triple and at full frame sizes, and the ctypes mirror of ``b200va_nv12_frame`` against the header
(no GPU needed)."""
import ctypes as C
import os
import shutil
import subprocess

import numpy as np
import pytest

from nv12_restate import nv12_to_bgr

REPO = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_every_yuv_triple_matches_cv2():
    """A 4096 x 4096 frame whose 2048 x 2048 blocks of 2 x 2 enumerate all 2^24 (Y, Cb, Cr): block k holds the chroma
    pair k >> 6 and the four luma values 4 (k & 63) .. 4 (k & 63) + 3."""
    cv2 = pytest.importorskip("cv2")
    k = np.arange(1 << 22, dtype=np.int64)
    pair, sub = k >> 6, k & 63
    by, bx = k // 2048, k % 2048
    y = np.empty((4096, 4096), np.uint8)
    for q, (dy, dx) in enumerate(((0, 0), (0, 1), (1, 0), (1, 1))):
        y[2 * by + dy, 2 * bx + dx] = (4 * sub + q).astype(np.uint8)
    uv = np.empty((2048, 4096), np.uint8)
    uv[by, 2 * bx] = (pair & 255).astype(np.uint8)
    uv[by, 2 * bx + 1] = (pair >> 8).astype(np.uint8)
    frame = np.concatenate([y, uv])
    assert np.array_equal(nv12_to_bgr(frame), cv2.cvtColor(frame, cv2.COLOR_YUV2BGR_NV12))


@pytest.mark.parametrize("hw", [(1080, 1920), (2160, 3840), (2, 2), (750, 1002)])
def test_frame_sizes_match_cv2(hw):
    cv2 = pytest.importorskip("cv2")
    h, w = hw
    frame = np.random.default_rng(h + w).integers(0, 256, size=(h * 3 // 2, w), dtype=np.uint8)
    want = cv2.cvtColor(frame, cv2.COLOR_YUV2BGR_NV12)
    assert np.array_equal(nv12_to_bgr(frame), want)
    assert np.array_equal(nv12_to_bgr(y=frame[:h], uv=frame[h:]), want)


def test_odd_sizes_are_refused():
    with pytest.raises(ValueError):
        nv12_to_bgr(y=np.zeros((4, 5), np.uint8), uv=np.zeros((2, 5), np.uint8))
    with pytest.raises(ValueError):
        nv12_to_bgr(y=np.zeros((4, 4), np.uint8), uv=np.zeros((3, 4), np.uint8))


@pytest.mark.skipif(shutil.which("gcc") is None, reason="no gcc")
def test_nv12_frame_struct_matches_the_header(tmp_path):
    from realtime_video_analytics_32streams_b200 import _native as N

    fields = [f[0] for f in N.Nv12Frame._fields_]
    lines = ['#include <stddef.h>', '#include <stdio.h>', '#include "b200va.h"', "int main(void) {",
             '  printf("size %zu\\n", sizeof(b200va_nv12_frame));']
    lines += [f'  printf("{f} %zu\\n", offsetof(b200va_nv12_frame, {f}));' for f in fields]
    lines += ["  return 0;", "}"]
    src = tmp_path / "nv12_layout.c"
    src.write_text("\n".join(lines))
    exe = tmp_path / "nv12_layout"
    proc = subprocess.run(["gcc", "-std=c99", "-Wall", "-Werror", f"-I{os.path.join(REPO, 'include')}", str(src), "-o", str(exe)],
                          stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True)
    assert proc.returncode == 0, proc.stdout
    out = subprocess.run([str(exe)], stdout=subprocess.PIPE, text=True, check=True).stdout
    got = {k: int(v) for k, v in (line.split() for line in out.strip().splitlines())}
    want = {"size": C.sizeof(N.Nv12Frame), **{f: getattr(N.Nv12Frame, f).offset for f in fields}}
    assert got == want


def test_nv12_entry_points_are_exported():
    from realtime_video_analytics_32streams_b200 import _native as N

    lib = N.load_library()
    for name in ("b200va_preprocess_nv12", "b200va_resize_linear_u8_nv12", "b200va_upload_frames_nv12", "b200va_tick_nv12"):
        assert name in N.EXPORTS
        getattr(lib, name)


def test_nv12_frame_detection():
    from realtime_video_analytics_32streams_b200 import _native as N

    assert N.is_nv12(np.zeros((6, 4), np.uint8))
    assert N.is_nv12((np.zeros((4, 4), np.uint8), np.zeros((2, 4), np.uint8)))
    assert not N.is_nv12(np.zeros((4, 4, 3), np.uint8))
