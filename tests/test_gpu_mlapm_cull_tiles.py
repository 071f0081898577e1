"""The culled symmetric MLAPM evaluation (mlapm_sym_tiles_kernel) against the dense one on crowd sizes that exercise
the unit schedule's edges: the smallest crowd the automatic choice culls, a last column tile of 1 or 17 agents, and odd
and even block counts T (the d = T/2 rule).  Each culled step is repeated and must be bit-identical."""
import math

import numpy as np
import pytest

from tests.test_gpu_mlapm_cull import GC_KW, TOL, _advance, _err


def _uniform_crowd(N, seed):
    rng = np.random.default_rng(seed)
    p = rng.random((N, 2)) * math.sqrt(N / 0.5)                   # the bench's density: most tile pairs are culled
    d = p + rng.normal(0, 30, (N, 2))
    v = rng.normal(0, 1, (N, 2))
    ds = 1.34 + 0.3 * rng.random((N, 1))
    return [x.astype(np.float32) for x in (p, v, ds, d)]


@pytest.mark.gpu
@pytest.mark.parametrize("N", [16384, 16401, 20001, 25000])      # T = 32, 33, 40, 49; N % 32 = 0, 17, 1, 8
def test_culled_tiles_match_dense(N):
    import piml_b200 as P
    p, v, ds, d = _uniform_crowd(N, N)
    model = P.MLAPM(**GC_KW)
    cul = _advance(model, p, v, ds, d, 2)
    again = _advance(model, p, v, ds, d, 2)
    den = _advance(model, p, v, ds, d, 3)
    for a, b in zip(cul, again):
        assert np.array_equal(a, b)                               # deterministic
    assert np.isfinite(cul[0]).all()
    assert _err(cul[0], den[0], v) < TOL
    assert np.array_equal(cul[2], den[2])
