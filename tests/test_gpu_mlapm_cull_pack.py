"""Packed units of the culled symmetric MLAPM evaluation (piml_b200/csrc/mlapm.cu, mlapm_cull_masks_kernel,
mlapm_sym_tiles_kernel): each list item's live columns (within r_cut of its 128-row tile's box, or non-finite) fill
units of 32 column slots.  Culled against dense on crowds where every column is live, few are, none are padded, and
where NaN velocities or positions must reach the rows they reach in the dense evaluation; two calls give the same
bits.  The number of units against a numpy count of the same rule."""
import ctypes as C
import math
import os
import sys
import warnings

import numpy as np
import pytest

from tests.test_gpu_mlapm_cull import GC_KW, TOL, _advance, _err, _radius


def _uniform(N, seed, side=None):
    rng = np.random.default_rng(seed)
    p = rng.random((N, 2)) * (side if side else math.sqrt(N / 0.5))   # default: the bench's density
    d = p + rng.normal(0, 30, (N, 2))
    v = rng.normal(0, 1, (N, 2))
    ds = 1.34 + 0.3 * rng.random((N, 1))
    return [x.astype(np.float32) for x in (p, v, ds, d)]


def _crowd(kind):
    if kind == "bench":
        sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
        import bench
        return [x.numpy() for x in bench.synthetic_crowd(100000)[:4]]
    if kind in ("n16384", "n16401"):
        return _uniform(int(kind[1:]), 3)
    if kind == "cluster":                                          # 20 m: every column of every unit is live
        return _uniform(20000, 4, side=20.0)
    p, v, ds, d = _uniform(20000, 5, side=150.0)
    if kind == "two_clusters":                                     # 150 m squares 2 km apart
        p[10000:] += 2000.0
        d[10000:] += 2000.0
    elif kind == "nan_velocity":                                   # finite position, NaN velocity
        v[777] = np.nan
    elif kind == "nan_position":
        p[4321] = np.nan
    return p, v, ds, d


@pytest.mark.gpu
@pytest.mark.parametrize("kind", ["bench", "n16384", "n16401", "cluster", "two_clusters", "nan_velocity",
                                  "nan_position"])
def test_packed_culled_matches_dense(kind):
    import piml_b200 as P
    p, v, ds, d = _crowd(kind)
    model = P.MLAPM(**GC_KW)
    cul = _advance(model, p, v, ds, d, 2)
    again = _advance(model, p, v, ds, d, 2)
    den = _advance(model, p, v, ds, d, 3)
    for a, b in zip(cul, again):
        assert np.array_equal(a, b, equal_nan=True)                # deterministic
    assert np.array_equal(cul[2], den[2])
    bad = np.isnan(den[0]).any(axis=-1)
    assert np.array_equal(np.isnan(cul[0]).any(axis=-1), bad)     # NaN reaches exactly the rows it reaches dense
    if kind == "nan_velocity":                                     # the rows whose view gate is open towards it
        assert bad.any() and not bad.all()
    elif kind == "nan_position":                                   # a NaN vr poisons every row, as in fp32
        assert bad.all()
        return
    else:
        assert not bad.any()
    assert _err(cul[0][~bad], den[0][~bad], v[~bad]) < TOL


def _hilbert9(x, y):
    x, y, dd = x.copy(), y.copy(), np.zeros_like(x)
    s = 256
    while s > 0:
        rx, ry = (x & s) > 0, (y & s) > 0
        dd += s * s * ((3 * rx.astype(np.int64)) ^ ry.astype(np.int64))
        flip = ~ry & rx
        x[flip], y[flip] = 511 - x[flip], 511 - y[flip]
        sw = ~ry
        x[sw], y[sw] = y[sw], x[sw].copy()
        s //= 2
    return dd


def _packed_units(p, rc):
    """W of the culled step on finite positions: the order kernel's Hilbert sort, the boxes, the list and the packing."""
    N = len(p)
    f32 = np.float32
    lo = (f32(0.5) * p.min(0)).astype(f32)
    hi = (f32(0.5) * p.max(0)).astype(f32)
    half = f32(max(hi[0] - lo[0], hi[1] - lo[1]))
    t = ((f32(0.5) * p - lo) / half).astype(f32) * f32(512)
    cell = np.minimum(t, f32(511)).astype(np.int64)
    q = p[np.argsort(_hilbert9(cell[:, 0], cell[:, 1]), kind="stable")].astype(np.float64)
    T = (N + 511) // 512
    D, npad = T // 2, T * 512
    xy = np.full((npad, 2), np.nan)
    xy[:N] = q

    def boxes(size):
        b = xy.reshape(-1, size, 2)
        with warnings.catch_warnings():
            warnings.simplefilter("ignore", RuntimeWarning)
            return np.concatenate([np.nanmin(b, 1), np.nanmax(b, 1)], 1)     # NaN rows: empty tiles

    rb, cb, bb = boxes(128), boxes(32), boxes(512)

    def near(a, b):
        gx = np.maximum(np.maximum(b[..., 0] - a[..., 2], a[..., 0] - b[..., 2]), 0)
        gy = np.maximum(np.maximum(b[..., 1] - a[..., 3], a[..., 1] - b[..., 3]), 0)
        return gx * gx + gy * gy <= float(np.float32(rc) * np.float32(rc))

    W = 0
    for R in range(4 * T):
        I, r = divmod(R, 4)
        for dd in range(D + 1):
            if T % 2 == 0 and dd == D and 2 * I >= T:
                continue
            J = (I + dd) % T
            if not near(rb[R], bb[J]):
                continue
            live = 0
            for ct in range(4 * r if dd == 0 else 0, 16):
                if not near(rb[R], cb[J * 16 + ct]):
                    continue
                if dd == 0 and ct // 4 == r:
                    W += 1                                          # own column tile: one unit
                    continue
                c = xy[J * 512 + ct * 32:J * 512 + ct * 32 + 32]
                pts = np.stack([c[:, 0], c[:, 1], c[:, 0], c[:, 1]], -1)
                live += int(near(rb[R][None], pts).sum())
            W += -(-live // 32)
    return W


@pytest.mark.gpu
def test_unit_count_matches_the_packing_rule():
    import piml_b200 as P
    from piml_b200 import _lib as L
    p, v, ds, d = _crowd("n16401")
    model = P.MLAPM(**GC_KW)
    _advance(model, p, v, ds, d, 2)
    units = C.c_int64()
    L.check(L.load().piml_mlapm_cull_items(L.ptr(model._ws), len(p), C.byref(units)), "piml_mlapm_cull_items")
    assert units.value == _packed_units(p, _radius(1, GC_KW['B'], GC_KW['C'], GC_KW['D']))
