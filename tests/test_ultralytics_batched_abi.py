"""CPU checks of the batched Ultralytics ABI: the ctypes mirror of ``b200va_tick_ultra`` against the C struct (the gcc
probe of test_abi_layout.py), the new entry points in the header and in ``EXPORTS``, and the host-side pieces of
``HotPathEngine``'s Ultralytics mode that need no GPU."""
import ctypes as C
import os
import re
import shutil
import subprocess

import pytest

REPO = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
NEW = ("b200va_preprocess_geom_nv12", "b200va_upload_frames_geom", "b200va_upload_frames_nv12_geom",
       "b200va_tick_ultralytics")


@pytest.mark.skipif(shutil.which("gcc") is None, reason="no gcc")
def test_tick_ultra_struct_matches_the_header(tmp_path):
    from realtime_video_analytics_32streams_b200 import _native as N

    fields = [f[0] for f in N.TickUltra._fields_]
    assert fields == ["geom", "src_h", "src_w", "in_h", "in_w", "agnostic", "max_det"]
    lines = ['#include <stddef.h>', '#include <stdio.h>', '#include "b200va.h"', "int main(void) {",
             '  printf("size %zu\\n", sizeof(b200va_tick_ultra));']
    lines += [f'  printf("{f} %zu\\n", offsetof(b200va_tick_ultra, {f}));' for f in fields]
    lines += ["  return 0;", "}"]
    src = tmp_path / "ultra.c"
    src.write_text("\n".join(lines))
    exe = tmp_path / "ultra"
    proc = subprocess.run(["gcc", "-std=c99", "-Wall", "-Werror", f"-I{os.path.join(REPO, 'include')}", str(src), "-o", str(exe)],
                          stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True)
    assert proc.returncode == 0, proc.stdout
    out = subprocess.run([str(exe)], stdout=subprocess.PIPE, text=True, check=True).stdout
    got = {k: int(v) for k, v in (line.split() for line in out.strip().splitlines())}
    want = {"size": C.sizeof(N.TickUltra), **{f: getattr(N.TickUltra, f).offset for f in fields}}
    assert got == want


def test_new_entry_points_are_declared_and_exported():
    from realtime_video_analytics_32streams_b200 import _native as N

    header = open(os.path.join(REPO, "include", "b200va.h")).read()
    for name in NEW:
        assert re.search(rf"B200VA_API int {name}\(", header), name
        assert name in N.EXPORTS, name


def test_engine_groups_frames_by_their_own_rect_shape():
    """The rect shapes HotPathEngine's Ultralytics mode gives each frame are those of a batch-1 predict, so 1080p,
    720p and a 1080p downsampled by 0.5 share one 384 x 640 group, while 640 x 480 and portrait 1080p get their own."""
    from realtime_video_analytics_32streams_b200 import _native as N

    def shape(h, w):
        return N.letterbox_meta_ultralytics(h, w, 640, 640, True, 32)[1:]

    assert shape(1080, 1920) == shape(720, 1280) == shape(540, 960) == (384, 640)
    assert shape(480, 640) == (480, 640)
    assert shape(1920, 1080) == (640, 384)
    m = N.letterbox_meta_ultralytics(1083, 1921, 640, 640, True, 32)[0]
    assert (m.new_h, N.letterbox_meta(1083, 1921, 640, 640).new_h) == (361, 360)
