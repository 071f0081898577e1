"""The culled symmetric MLAPM evaluation (piml_b200/csrc/mlapm.cu, mlapm_sym_list_kernel): pairs farther apart than
piml_mlapm_cull_radius are skipped because their fp32 weight is exactly 0.  The radius against a numpy evaluation of
the exponent's bound (CPU), the exact-zero premise at the radius itself, and the culled path (algorithm 2) against the
dense symmetric path (algorithm 3) on crowds that stress the spatial sort and the boxes."""
import ctypes as C
import math
import os
import sys

import numpy as np
import pytest
import torch

TOL = 1e-5
GC_KW = dict(version='GC', tau=0.5, A=7.55, B=-3.00, C=0.2, D=-0.3, theta=56)
LOG2E = np.float32(1.4426950408889634)


def _radius(version, B, C_, D, exact=0):
    from piml_b200 import _lib as L
    prm = L.MlapmParams(version, 0.5, 7.55, float(B), float(C_), float(D), 56.0, exact)
    return float(L.load().piml_mlapm_cull_radius(C.byref(prm)))


def _max_arg(version, B, C_, D, r):
    """Largest exponent (log2 units) of a pair at distance r over every relative velocity: the cosine is +-1."""
    Bl, Cl, Dl = (np.float32(np.float64(x) * np.float64(LOG2E)) for x in (B, C_, D))
    Bl, Cl, Dl = float(Bl), float(Cl), float(Dl)
    if version == 0:
        return Bl * r
    return max(Bl * r + cs * (Cl + Dl * r) for cs in (-1.0, 1.0))


@pytest.mark.parametrize("version", [0, 1])
def test_cull_radius_against_the_exponent_bound(version):
    rng = np.random.default_rng(11 + version)
    sets = [(-3.0, 0.2, -0.3), (-1.0, 2.0, 0.5), (-0.5, -1.5, 0.2), (-8.0, 0.0, 0.0), (-0.05, 3.0, -0.01)]
    sets += [tuple(x) for x in np.c_[-rng.uniform(0.05, 6, 20), rng.uniform(-4, 4, 20), rng.uniform(-2, 2, 20)]]
    for B, C_, D in sets:
        if version == 1 and B + abs(D) >= 0:
            continue
        rc = _radius(version, B, C_, D)
        assert math.isfinite(rc) and rc > 0
        # beyond r_cut every pair's exponent is below -127: exp2 underflows to exactly 0 (flushed below -126)
        for r in rc * np.array([1.0, 1.5, 4.0, 100.0]):
            assert _max_arg(version, B, C_, D, r) < -127.0, (B, C_, D, rc, r)
        # the radius is not far from the tight one: the bound (B + |D|) r + |C| is reached up to the 1 % margin
        slope = B if version == 0 else B + abs(D)
        r0 = (127 + (0 if version == 0 else abs(C_) * float(LOG2E))) / -(slope * float(LOG2E))
        assert rc <= r0 * 1.02 + 0.02


def test_cull_radius_is_infinite_without_decay():
    assert math.isinf(_radius(1, -0.3, 0.2, 0.3))          # B + |D| = 0
    assert math.isinf(_radius(1, -0.3, 0.2, -0.5))         # B + |D| > 0
    assert math.isinf(_radius(0, 0.5, 0.0, 0.0))           # raw: B >= 0
    assert math.isinf(_radius(1, -3.0, 0.2, -0.3, exact=1))
    assert math.isfinite(_radius(1, -3.0, 0.2, -0.3))
    assert abs(_radius(1, -3.0, 0.2, -0.3) - 32.7 * 1.01) < 0.1


# ---- GPU -----------------------------------------------------------------------------------------------------------
def _algo(a):
    from piml_b200 import _lib as L
    L.check(L.load().piml_set_mlapm_algorithm(a), "piml_set_mlapm_algorithm")


def _advance(model, p, v, ds, d, algo):
    _algo(algo)
    try:
        out = model.advance(*[torch.as_tensor(x).float().cuda() for x in (p, v, ds, d)], 0.08, 0.3)
    finally:
        _algo(0)
    return [t.cpu().numpy() for t in out]


def _err(got, ref, v):
    num = np.linalg.norm(np.asarray(got, np.float64) - ref, axis=-1)
    den = np.maximum(np.maximum(np.linalg.norm(ref, axis=-1), np.linalg.norm(v, axis=-1)), 1e-6)
    return float((num / den).max())


def _crowd(kind, seed=5):
    rng = np.random.default_rng(seed)
    N = {"cluster": 20000, "two_clusters": 20000, "far": 20000, "nan_inf": 20000, "ragged": 17123}[kind]
    if kind == "cluster":                                         # one cluster smaller than r_cut: nothing culled
        p = rng.random((N, 2)) * 20.0
    elif kind == "two_clusters":                                  # two 100 m clusters 1 km apart
        p = rng.random((N, 2)) * 100.0
        p[N // 2:] += 1000.0
    else:
        p = rng.random((N, 2)) * math.sqrt(N / 0.5)
        if kind == "far":                                         # 1e6 m: the cell coordinates wrap modulo 2^16
            p += 1.0e6
    d = p + rng.normal(0, 30, (N, 2))
    v = rng.normal(0, 1, (N, 2))
    ds = 1.34 + 0.3 * rng.random((N, 1))
    p, v, ds, d = (x.astype(np.float32) for x in (p, v, ds, d))
    if kind == "nan_inf":
        p[123] = np.nan
        p[4567, 0] = np.inf
    return p, v, ds, d


@pytest.mark.gpu
@pytest.mark.parametrize("version", ["GC", "raw"])
def test_weight_is_exactly_zero_at_the_cull_radius(version):
    """Two agents exactly r_cut apart, both view gates open (each walks towards the other), so the relative velocity is
    antiparallel to vr: cos = -1, which maximises the exponent B r + (C + D r) cos for these parameters
    (C + D r < 0).  Each agent's action is bit for bit its action alone."""
    import piml_b200 as P
    kw = dict(GC_KW, version=version)
    rc = _radius(1 if version == "GC" else 0, kw['B'], kw['C'], kw['D'])
    assert kw['C'] + kw['D'] * rc < 0
    p = np.array([[0.0, 0.0], [rc, 0.0]], np.float32)
    v = np.array([[1.0, 0.0], [-1.0, 0.0]], np.float32)
    d = np.array([[5.0, 3.0], [rc - 5.0, -3.0]], np.float32)
    ds = np.full((2, 1), 1.3, np.float32)
    model = P.MLAPM(**kw)
    for algo in (2, 3):
        pair = _advance(model, p, v, ds, d, algo)[0]
        for i in range(2):
            alone = _advance(model, p[i:i + 1], v[i:i + 1], ds[i:i + 1], d[i:i + 1], algo)[0]
            assert np.array_equal(pair[i], alone[0]), (algo, i, pair[i], alone[0])


@pytest.mark.gpu
@pytest.mark.parametrize("kind", ["bench", "cluster", "two_clusters", "far", "nan_inf", "ragged"])
def test_culled_matches_dense(kind):
    import piml_b200 as P
    if kind == "bench":
        sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
        import bench
        p, v, ds, d, _ = [x.numpy() for x in bench.synthetic_crowd(100000)]
    else:
        p, v, ds, d = _crowd(kind)
    model = P.MLAPM(**GC_KW)
    cul = _advance(model, p, v, ds, d, 0 if kind == "bench" else 2)
    again = _advance(model, p, v, ds, d, 2)
    den = _advance(model, p, v, ds, d, 3)
    for a, b in zip(cul, again):
        assert np.array_equal(a, b, equal_nan=True)               # deterministic
    if kind == "nan_inf":
        assert np.isnan(cul[0]).all() and np.isnan(den[0]).all()  # one NaN agent poisons every row, as in fp32
        return
    assert np.isfinite(cul[0]).all()
    assert _err(cul[0], den[0], v) < TOL
    assert np.array_equal(cul[2], den[2])
    # p' = p + action dt: two ulps of the coordinate plus the action gate carried through dt
    scale = np.maximum(np.linalg.norm(den[0], axis=-1), np.linalg.norm(v, axis=-1))[:, None]
    bound = 2 * np.spacing(np.abs(den[1]).astype(np.float32)) + 0.08 * TOL * scale
    assert (np.abs(cul[1] - den[1]) <= bound).all()


@pytest.mark.gpu
@pytest.mark.parametrize("N", [1 << 14, 100000, 1000000, 3000000])
def test_cub_scratch_fits_the_reserved_bound(N):
    """The culled path checks CUB's real scratch size against the bound reserved without a device and fails the call
    if it does not fit: a successful step on algorithm 2 at each size is the check."""
    import piml_b200 as P
    g = torch.Generator().manual_seed(N)
    side = math.sqrt(N / 0.5)
    p = torch.rand(N, 2, generator=g) * side
    v = torch.randn(N, 2, generator=g)
    d = torch.rand(N, 2, generator=g) * side
    ds = torch.full((N, 1), 1.3)
    act = _advance(P.MLAPM(**GC_KW), p, v, ds, d, 2)[0]
    assert np.isfinite(act).all()
