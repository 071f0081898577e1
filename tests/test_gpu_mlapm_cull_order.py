"""The spatial order of the culled symmetric MLAPM step (mlapm_cull_order_kernel: a Hilbert key on a 512 x 512 grid
fitted to the crowd's box, two stable 9-bit LSD passes): crowds whose box degenerates, coordinates whose extent
overflows fp32, and a permutation that depends on the positions alone, not on what the workspace held before."""
import numpy as np
import pytest

from tests.test_gpu_mlapm_cull import GC_KW, TOL, _advance, _err


def _crowd(kind, seed=7):
    rng = np.random.default_rng(seed)
    N = 20000
    if kind == "one_point":                                       # zero extent: every agent in cell (0, 0)
        p = np.full((N, 2), 12.5)
        d = p + rng.normal(0, 30, (N, 2))
    elif kind == "far_clusters":                                  # two 100 m clusters 1e5 m apart: the fitted grid's
        p = rng.random((N, 2)) * 100.0                            # cells are 195 m, one cluster spans one to four
        p[N // 2:, 0] += 1.0e5
        d = p + rng.normal(0, 30, (N, 2))
    elif kind == "huge":                                          # max - min = 6e38 overflows fp32
        p = (rng.random((N, 2)) * 2.0 - 1.0) * 3.0e38
        p[:8] = [[-3.0e38, -3.0e38], [3.0e38, 3.0e38], [-3.0e38, 3.0e38], [3.0e38, -3.0e38],
                 [0.0, 0.0], [-3.0e38, 0.0], [3.0e38, 0.0], [0.0, 3.0e38]]
        d = rng.random((N, 2)) * 100.0
    else:                                                         # bench-like density: 0.5 per m^2
        side = np.sqrt(N / 0.5)
        p = rng.random((N, 2)) * side
        d = rng.random((N, 2)) * side
    v = rng.normal(0, 1, (N, 2))
    ds = 1.34 + 0.3 * rng.random((N, 1))
    return [x.astype(np.float32) for x in (p, v, ds, d)]


@pytest.mark.gpu
@pytest.mark.parametrize("kind", ["one_point", "far_clusters"])
def test_culled_matches_dense_on_degenerate_boxes(kind):
    import piml_b200 as P
    p, v, ds, d = _crowd(kind)
    model = P.MLAPM(**GC_KW)
    cul = _advance(model, p, v, ds, d, 2)
    again = _advance(model, p, v, ds, d, 2)
    den = _advance(model, p, v, ds, d, 3)
    for a, b in zip(cul, again):
        assert np.array_equal(a, b, equal_nan=True)               # deterministic
    assert np.isfinite(cul[0]).all()
    assert _err(cul[0], den[0], v) < TOL
    assert np.array_equal(cul[2], den[2])


@pytest.mark.gpu
def test_extent_beyond_fp32_completes_and_repeats():
    """Coordinates near +-3e38: the box's extent is not an fp32 number, the keys still are.  Pair differences overflow
    too, so there is nothing to compare with the dense path; the step completes and repeats bit for bit.  The keys stay
    spatial: the sorted tiles' boxes are compact, so few (row tile, column tile) units touch.  Keys that collapsed to
    one cell would leave the crowd in index order, every tile's box would span the crowd and every unit would be live."""
    import ctypes as C
    import piml_b200 as P
    from piml_b200 import _lib as L
    p, v, ds, d = _crowd("huge")
    model = P.MLAPM(**GC_KW)
    first = _advance(model, p, v, ds, d, 2)
    units = C.c_int64()
    L.check(L.load().piml_mlapm_cull_items(L.ptr(model._ws), len(p), C.byref(units)), "piml_mlapm_cull_items")
    T = (len(p) + 511) // 512
    assert 0 < units.value < 0.5 * T * (T // 2 + 1) * 4 * 16, units.value
    for a, b in zip(first, _advance(model, p, v, ds, d, 2)):
        assert np.array_equal(a, b, equal_nan=True)


@pytest.mark.gpu
def test_order_does_not_depend_on_the_workspace_history():
    """Crowd A, then crowd B of the same size, then A again on one MLAPM object (one workspace): A's step is bit for bit
    what it was the first time."""
    import piml_b200 as P
    a = _crowd("bench", seed=1)
    b = _crowd("far_clusters", seed=2)
    model = P.MLAPM(**GC_KW)
    first = _advance(model, *a, 2)
    mid = _advance(model, *b, 2)
    assert not np.array_equal(first[0], mid[0])
    for x, y in zip(first, _advance(model, *a, 2)):
        assert np.array_equal(x, y, equal_nan=True)

