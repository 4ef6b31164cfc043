"""CPU statement of the Ultralytics YOLOv8 ``Detect`` head decode (DFL).  TEST INFRASTRUCTURE ONLY.

**Parity unpinned**: this step is not part of ``/root/reference`` -- the reference only reaches it
through the third-party package ``ultralytics==8.3.209`` (``pylock.toml:1432-1433``; call sites
``detector.py:117,129,147-155``), which is neither vendored nor installed here, and the reference's
tests hold no vectors for it.  The published algorithm (``ultralytics/nn/modules/head.py`` ``Detect``
with ``DFL`` and ``dist2bbox(xywh=True)``, ``make_anchors(offset=0.5)``) is restated below, in float32
or in float64.  The CUDA kernel is compared with the float64 decode of its own float32 inputs under an
error bound derived from the kernel's float32 operation order (``tests/dfl_bound.py``): exp / softmax
are not bit-reproducible.
"""

from __future__ import annotations

import numpy as np


def make_anchors(levels=((80, 80), (40, 40), (20, 20)), strides=(8.0, 16.0, 32.0), dtype=np.float32):
    pts, st = [], []
    for (h, w), s in zip(levels, strides):
        ys, xs = np.meshgrid(np.arange(h, dtype=dtype) + 0.5, np.arange(w, dtype=dtype) + 0.5, indexing="ij")
        pts.append(np.stack([xs.ravel(), ys.ravel()], 0))
        st.append(np.full((h * w,), s, dtype=dtype))
    return np.concatenate(pts, 1), np.concatenate(st)


def dfl_decode(raw: np.ndarray, num_classes: int, reg_max: int = 16, levels=((80, 80), (40, 40), (20, 20)),
               strides=(8.0, 16.0, 32.0), dtype=np.float32) -> np.ndarray:
    """raw [B, 4*reg_max + nc, A] float32 -> [B, 4 + nc, A] in ``dtype`` (cx, cy, w, h in input pixels, sigmoid scores).

    ``dtype=np.float64`` decodes the float32 inputs in float64 throughout.  Non-finite values follow IEEE arithmetic:
    a side holding a NaN or +inf bin, or only -inf bins, decodes to NaN; a -inf bin among finite ones has weight 0."""
    dtype = np.dtype(dtype)
    raw = raw.astype(np.float32, copy=False).astype(dtype, copy=False)
    b, _, a = raw.shape
    box = raw[:, :4 * reg_max].reshape(b, 4, reg_max, a)
    with np.errstate(over="ignore", invalid="ignore"):
        e = np.exp(box - box.max(axis=2, keepdims=True))
        prob = e / e.sum(axis=2, keepdims=True)
        dist = (prob * np.arange(reg_max, dtype=dtype)[None, None, :, None]).sum(axis=2)  # [B, 4, A]
        anchors, st = make_anchors(levels, strides, dtype)
        x1y1 = anchors[None] - dist[:, :2]
        x2y2 = anchors[None] + dist[:, 2:]
        cxy = (x1y1 + x2y2) / dtype.type(2)
        wh = x2y2 - x1y1
        out_box = np.concatenate([cxy, wh], 1) * st[None, None]
        cls = dtype.type(1) / (dtype.type(1) + np.exp(-raw[:, 4 * reg_max:]))
    return np.concatenate([out_box, cls], 1).astype(dtype, copy=False)
