"""NumPy restatement of ``cv2.cvtColor(frame, cv2.COLOR_YUV2BGR_NV12)`` (OpenCV's
``modules/imgproc/src/color_yuv.simd.hpp``, 8-bit path).

TEST INFRASTRUCTURE ONLY, like ``oracle/``: the NV12 tests compare every NV12 entry point with the BGR entry point
and with ``oracle.hotpath`` on the frame this function returns.  ``tests/test_oracle_nv12.py`` pins it against the
installed ``cv2`` on all 2^24 (Y, Cb, Cr) triples.
"""

from __future__ import annotations

import numpy as np


def nv12_to_bgr(frame: np.ndarray = None, y: np.ndarray = None, uv: np.ndarray = None) -> np.ndarray:
    """``cv2.cvtColor(frame, cv2.COLOR_YUV2BGR_NV12)``: OpenCV's BT.601 limited-range 20-bit fixed point with nearest
    chroma.  ``frame`` is OpenCV's ``[3H/2, W]`` NV12 layout; ``(y [H, W], uv [H/2, W])`` planes may be given instead.
    Each 2 x 2 block shares the Cb, Cr pair ``uv[y >> 1][(x & ~1) + {0, 1}]``."""
    if frame is not None:
        frame = np.asarray(frame)
        h = frame.shape[0] * 2 // 3
        y, uv = frame[:h], frame[h:]
    y = np.asarray(y, dtype=np.uint8)
    uv = np.asarray(uv, dtype=np.uint8)
    h, w = y.shape
    if h % 2 or w % 2 or uv.shape != (h // 2, w):
        raise ValueError("NV12 needs an even size and a [H/2, W] chroma plane")
    cb = np.repeat(np.repeat(uv[:, 0::2], 2, axis=0), 2, axis=1).astype(np.int32) - 128
    cr = np.repeat(np.repeat(uv[:, 1::2], 2, axis=0), 2, axis=1).astype(np.int32) - 128
    yy = np.maximum(y.astype(np.int32) - 16, 0) * 1220542 + (1 << 19)
    out = np.empty((h, w, 3), dtype=np.uint8)
    out[..., 0] = np.clip((yy + 2116026 * cb) >> 20, 0, 255)
    out[..., 1] = np.clip((yy - 852492 * cr - 409993 * cb) >> 20, 0, 255)
    out[..., 2] = np.clip((yy + 1673527 * cr) >> 20, 0, 255)
    return out
