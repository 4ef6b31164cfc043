"""Error bound of the float32 DFL decode (k_dfl_decode) around the float64 decode of the same float32 inputs
(``oracle.dfl.dfl_decode(..., dtype=np.float64)``).

Derived from the kernel's float32 operation order.  Per box side, over the R = reg_max bins x_k:
m = max x_k, e_k = expf(x_k - m), s = sum e_k, e = sum k e_k (two running sums, no FMA), d = e / s.  With
eps = 2**-24 (the unit roundoff of float32):

* side expectation, absolute:       delta_d(R) = (2R + 6) * max(R - 1, 1) * eps
  (the rounding of x_k - m, up to 2 ulp of expf, R - 1 rounded additions in each sum and the division, each
  scaled by a weight of at most R - 1)
* box output o in {cx, cy, w, h} of an anchor with coordinate a (ax for cx and w, ay for cy and h) and stride s:
  |o - o64| <= |s| * (2 delta_d + 4 eps (a + R)) + eps |o64|
  (two sides enter each output; x1 = a - d, x2 = a + d', their sum or difference, and the product with the stride
  are rounded once each)
* class score p = 1 / (1 + expf(-x)), the reciprocal correctly rounded:
  |p - p64| <= 4 eps p64 when p64 >= 2**-126; otherwise 0 <= p <= 2**-126 (below x ~ -88.7, expf(-x) overflows to
  inf and the kernel returns 0 where the exact value is subnormal; the float32 oracle does the same).

A NumPy emulation of this order stays below about 0.83 R (R - 1) eps on each side, so the box bound has roughly
3-10x headroom over a correct float32 decode (the emulation reaches 0.32 of it at R = 2, 0.06 at R = 16), while a
real defect (a bin weight off by one, swapped sides, a wrong anchor offset or level) is off by about one bin times
the stride.  The score bound is tighter: the two roundings take 2 eps, leaving 2 eps for the exp (NumPy's float32
exp reaches 0.88 of the bound).  tests/test_oracle_dfl.py checks both directions.
"""

import numpy as np

from oracle import dfl as D

EPS = 2.0 ** -24
TINY = 2.0 ** -126


def delta_d(reg_max: int) -> float:
    return (2 * reg_max + 6) * max(reg_max - 1, 1) * EPS


def error_ratio(got, ref64, reg_max, levels, strides):
    """|got - ref64| / bound per element of a decode [B, 4 + nc, A] (<= 1 inside the bound).  Elements that are equal,
    NaN in both, or (for scores whose exact value is below 2**-126) in [0, 2**-126] count 0; a NaN in only one of the
    two, or a tiny score outside [0, 2**-126], counts inf."""
    got = np.asarray(got, np.float64)
    ref64 = np.asarray(ref64, np.float64)
    anchors, st = D.make_anchors(levels, strides, np.float64)
    coord = anchors[[0, 1, 0, 1]][None]  # cx, cy, w, h
    box_bound = np.abs(st) * (2 * delta_d(reg_max) + 4 * EPS * (coord + reg_max)) + EPS * np.abs(ref64[:, :4])
    cls_bound = 4 * EPS * ref64[:, 4:]
    bound = np.concatenate([np.broadcast_to(box_bound, ref64[:, :4].shape), cls_bound], 1)
    with np.errstate(invalid="ignore", divide="ignore"):
        err = np.abs(got - ref64)
        r = np.where(bound > 0, err / bound, np.where(err == 0, 0.0, np.inf))
    r[got == ref64] = 0.0
    gn, rn = np.isnan(got), np.isnan(ref64)
    r[gn & rn] = 0.0
    r[gn ^ rn] = np.inf
    tiny = np.zeros(got.shape, bool)
    tiny[:, 4:] = ref64[:, 4:] < TINY
    r[tiny] = np.where((got[tiny] >= 0) & (got[tiny] <= TINY), 0.0, np.inf)
    return r


def worst(ratio):
    """(largest ratio, index of it) -- for assertion messages."""
    i = int(np.argmax(ratio))
    return float(ratio.flat[i]), np.unravel_index(i, ratio.shape)
