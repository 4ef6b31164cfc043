"""CPU checks of the DFL oracle and of the error bound the GPU tests hold k_dfl_decode to (tests/dfl_bound.py).

* The float64 decode agrees with an independent torch float64 softmax decode, and the float32 oracle is inside the
  bound around it.
* A NumPy float32 emulation of the kernel's operation order stays inside the bound for every reg_max the kernel's
  instantiations serve, at logit scales from 0.1 to 200.
* Four mutated emulations -- bin weights k + 1, sides l / r swapped, anchor offset 0 instead of 0.5, the level
  lookup one anchor late -- leave the bound on the same inputs, so the bound is tight enough to catch them."""

import numpy as np
import pytest

import dfl_bound as DB
from oracle import dfl as D

REG_MAX = (1, 2, 7, 16, 17, 32, 64)
# the three geometries of the first DFL test, and one with a level boundary inside every 4-anchor group
GEOMS = ((((80, 80), (40, 40), (20, 20)), (8.0, 16.0, 32.0)),
         (((5, 7), (3, 5)), (8.0, 16.0)),
         (((12, 20), (6, 10)), (8.0, 16.0)),
         (((3, 5), (1, 1), (2, 1), (1, 3)), (12.0, 0.75, 32.0, 8.0)))


def _expf(x):
    """Correctly rounded float32 exp (NumPy's own float32 exp is not, and differs between SIMD paths)."""
    with np.errstate(over="ignore"):
        return np.exp(x.astype(np.float64)).astype(np.float32)


def emulate(raw, nc, reg_max, levels, strides, mutation=None):
    """k_dfl_decode's float32 arithmetic in NumPy, in the kernel's order (fmaxf, expf(x - m), two running sums
    without FMA, one division; the anchor's level found by walking the level offsets)."""
    f = np.float32
    raw = np.asarray(raw, f)
    b, _, a = raw.shape
    box = raw[:, :4 * reg_max].reshape(b, 4, reg_max, a)
    m = np.fmax.reduce(box, axis=2, initial=-np.inf)
    s = np.zeros((b, 4, a), f)
    e = np.zeros((b, 4, a), f)
    for k in range(reg_max):
        ek = _expf(box[:, :, k] - m)
        s = s + ek
        e = e + f(k + 1 if mutation == "weights" else k) * ek
    d = e / s
    if mutation == "swap":
        d = d[:, [2, 1, 0, 3]]
    sizes = np.array([h * w for h, w in levels])
    off = np.concatenate([[0], np.cumsum(sizes)])
    idx = np.arange(a)
    lv = np.searchsorted(off[1:-1], idx, side="left" if mutation == "level" else "right")
    k = idx - off[lv]
    w = np.array([w for _, w in levels])[lv]
    half = f(0.0 if mutation == "offset" else 0.5)
    ax = (k % w).astype(f) + half
    ay = (k // w).astype(f) + half
    st = np.asarray(strides, f)[lv]
    x1, y1, x2, y2 = ax - d[:, 0], ay - d[:, 1], ax + d[:, 2], ay + d[:, 3]
    cx = (x1 + x2) * f(0.5) * st
    cy = (y1 + y2) * f(0.5) * st
    bw = (x2 - x1) * st
    bh = (y2 - y1) * st
    cls = f(1) / (f(1) + _expf(-raw[:, 4 * reg_max:]))
    return np.concatenate([np.stack([cx, cy, bw, bh], 1), cls], 1)


def _raw(seed, b, reg_max, nc, a, scale):
    return (np.random.default_rng(seed).normal(0, scale, size=(b, 4 * reg_max + nc, a))).astype(np.float32)


@pytest.mark.parametrize("gi", range(len(GEOMS)))
def test_float64_reference_matches_torch_softmax(gi):
    torch = pytest.importorskip("torch")
    levels, strides = GEOMS[gi]
    a = sum(h * w for h, w in levels)
    for reg_max, nc in ((16, 80), (7, 3)):
        raw = _raw(71 + gi, 3, reg_max, nc, a, 2.5)
        ref = D.dfl_decode(raw, nc, reg_max, levels, strides, dtype=np.float64)
        assert ref.dtype == np.float64 and ref.shape == (3, 4 + nc, a)
        t = torch.from_numpy(raw).double()
        p = t[:, :4 * reg_max].view(3, 4, reg_max, a).softmax(2)
        dist = (p * torch.arange(reg_max, dtype=torch.float64).view(1, 1, reg_max, 1)).sum(2).numpy()
        anchors, st = D.make_anchors(levels, strides, np.float64)
        lt, rb = anchors[None] - dist[:, :2], anchors[None] + dist[:, 2:]
        want = np.concatenate([(lt + rb) / 2 * st, (rb - lt) * st, torch.sigmoid(t[:, 4 * reg_max:]).numpy()], 1)
        np.testing.assert_allclose(ref, want, rtol=1e-13, atol=1e-12)
        r = DB.error_ratio(D.dfl_decode(raw, nc, reg_max, levels, strides), ref, reg_max, levels, strides)
        assert r[:, :4].max() <= 1.0, ("float32 oracle", reg_max, DB.worst(r[:, :4]))
        # NumPy's float32 exp may be off by more than the 2 eps the score bound leaves it
        assert r[:, 4:].max() <= 2.0, ("float32 oracle", reg_max, DB.worst(r[:, 4:]))


@pytest.mark.parametrize("reg_max", REG_MAX)
def test_kernel_order_within_bound(reg_max):
    worst_box = 0.0
    for gi, (levels, strides) in enumerate(GEOMS[1:]):
        a = sum(h * w for h, w in levels)
        for scale in (0.1, 0.5, 2.5, 20.0, 200.0):
            raw = _raw(1000 * reg_max + gi, 4, reg_max, 9, a, scale)
            ref = D.dfl_decode(raw, 9, reg_max, levels, strides, dtype=np.float64)
            r = DB.error_ratio(emulate(raw, 9, reg_max, levels, strides), ref, reg_max, levels, strides)
            assert r.max() <= 1.0, (reg_max, scale, DB.worst(r))
            worst_box = max(worst_box, float(r[:, :4].max()))
    # the box bound leaves headroom over a correct float32 order (the score bound is tighter: 2 roundings + exp)
    assert worst_box < 0.5, worst_box


def test_class_score_edges_within_bound():
    x = np.array([0.0, -0.0, np.inf, -np.inf, np.nan, 20.0, 1e30, 1e-30, -1e-30, 88.7, -80.0, -87.3, -87.4, -88.7,
                  -88.8, -103.9, -104.0, -200.0, -1e30, 15.9, -15.9], np.float32)
    raw = np.zeros((1, 4 + x.size, 1), np.float32)
    raw[0, 4:, 0] = x
    ref = D.dfl_decode(raw, x.size, 1, ((1, 1),), (8.0,), dtype=np.float64)
    for got, limit in ((emulate(raw, x.size, 1, ((1, 1),), (8.0,)), 1.0),
                       (D.dfl_decode(raw, x.size, 1, ((1, 1),), (8.0,)), 2.0)):  # NumPy's float32 exp, as above
        r = DB.error_ratio(got, ref, 1, ((1, 1),), (8.0,))
        assert r.max() <= limit, DB.worst(r)
        p = got[0, 4:, 0]
        assert p[0] == p[1] == 0.5 and p[2] == 1.0 and p[3] == 0.0 and np.isnan(p[4]) and p[5] == p[6] == 1.0


@pytest.mark.parametrize("mutation", ["weights", "swap", "offset", "level"])
def test_bound_rejects_mutated_kernels(mutation):
    """Each defect leaves the bound on inputs the correct order stays inside."""
    for reg_max in (2, 7, 16, 17):
        for levels, strides in GEOMS[1:]:
            a = sum(h * w for h, w in levels)
            raw = _raw(reg_max, 2, reg_max, 3, a, 2.5)
            ref = D.dfl_decode(raw, 3, reg_max, levels, strides, dtype=np.float64)
            assert DB.error_ratio(emulate(raw, 3, reg_max, levels, strides), ref, reg_max, levels, strides).max() <= 1.0
            r = DB.error_ratio(emulate(raw, 3, reg_max, levels, strides, mutation), ref, reg_max, levels, strides)
            # a mutation of the box decode is at least ~100x the bound somewhere; class scores are untouched
            assert r[:, :4].max() > 100.0, (mutation, reg_max, levels, DB.worst(r))
            assert r[:, 4:].max() <= 1.0
