"""MLAPM.advance_scenes / rollout_scenes (piml_mlapm_scenes_advance_f32): many independent padded scenes in one launch,
each against the CPU oracle on its active agents with its own constants, against MLAPM.advance on the compacted scene,
and against the golden `circle` scene of main_mlapm.py.  Gates as in test_gpu_parity.py."""
import numpy as np
import pytest
import torch

from oracle import oracle as O
from tests.util import golden, group, rel_vec_err

pytestmark = pytest.mark.gpu

TOL = 1e-5
GC_KW = dict(version='GC', tau=0.5, A=7.55, B=-3.00, C=0.2, D=-0.3, theta=56)
GC_ROW = [0.5, 7.55, -3.0, 0.2, -0.3, 56.0]
DT, RADIUS = 0.08, 0.3
MAX_N = 8192                       # PIML_MLAPM_SCENES_MAX_N


def cu(x, dtype=torch.float32):
    return torch.as_tensor(np.asarray(x), dtype=dtype).cuda()


def npy(t):
    return t.detach().cpu().numpy()


def model(ver="GC", exact=False):
    import piml_b200 as P
    return P.MLAPM(**dict(GC_KW, version=ver, exact_math=exact))


def scenes(S, N, seed, inactive=(0.1, 0.3), ds_dim=1, nan_inactive=True):
    """Padded GC-shaped scenes (density 0.5 per m^2 over the scene's slots), 10-30 % of the slots inactive, some
    stationary and some coincident agents, some agents within reach of their destination."""
    rng = np.random.default_rng(seed)
    L = np.sqrt(N / 0.5)
    p = (rng.random((S, N, 2)) * L).astype(np.float32)
    d = (rng.random((S, N, 2)) * L).astype(np.float32)
    near = rng.random((S, N)) < 0.1
    d[near] = p[near] + rng.normal(0, 0.2, (int(near.sum()), 2)).astype(np.float32)
    v = rng.normal(0, 1, (S, N, 2)).astype(np.float32)
    v[rng.random((S, N)) < 0.05] = 0.0                            # stationary: see nobody
    if N >= 4:
        p[:, 3] = p[:, 1]                                         # coincident pair
    ds = (1.34 + 0.3 * rng.normal(0, 1, (S, N, ds_dim))).astype(np.float32)
    frac = rng.uniform(*inactive, (S, 1))
    act = rng.random((S, N)) >= frac
    if nan_inactive:
        p[~act] = np.nan; v[~act] = np.nan; d[~act] = np.nan; ds[~act] = np.nan
    return p, v, ds, d, act


def rand_params(S, seed):
    rng = np.random.default_rng(seed)
    prm = np.tile(np.asarray(GC_ROW, np.float32), (S, 1))
    prm *= rng.uniform(0.7, 1.3, (S, 6)).astype(np.float32)
    return prm


def err(got, ref, v):
    """Operand-scaled gate of test_mlapm_symmetric_evaluation: |got - ref| / max(|ref|, |v|)."""
    num = np.linalg.norm(np.asarray(got, np.float64) - ref, axis=-1)
    den = np.maximum(np.maximum(np.linalg.norm(ref, axis=-1), np.linalg.norm(v, axis=-1)), 1e-6)
    return float((num / den).max()) if num.size else 0.0


def run(m, p, v, ds, d, act, params=None):
    a, q, arr = m.advance_scenes(cu(p), cu(v), cu(ds), cu(d), cu(act, torch.bool), DT, RADIUS,
                                 None if params is None else cu(params))
    return npy(a), npy(q), npy(arr)


def check_scene(a, q, arr, p, v, ds, d, act, ver, prm=GC_ROW, rows=None):
    """One scene's outputs against the oracle step on its active agents (rows: a sub-range of them)."""
    idx = np.nonzero(act)[0]
    inact = ~act
    assert np.isnan(a[inact]).all() and np.isnan(q[inact]).all() and not arr[inact].any()
    if idx.size == 0:
        return
    tau, A, B, C_, D, th = [float(x) for x in prm]
    want = O.mlapm_step(p[idx], v[idx], ds[idx], d[idx], DT, ver, tau=tau, A=A, B=B, C_=C_, D=D, theta=th, rows=rows)
    sel = idx if rows is None else idx[rows[0]:rows[1]]
    assert err(a[sel], want, v[sel]) < TOL
    qw = (p[sel] + want * np.float32(DT)).astype(np.float32)
    assert np.allclose(q[sel], qw, rtol=0, atol=1e-5)
    dist = np.linalg.norm(qw - d[sel], axis=-1)
    clear = np.abs(dist - RADIUS) > 1e-4
    assert np.array_equal(arr[sel][clear], (dist < RADIUS)[clear])


# ---- oracle per scene ------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("exact", [False, True])
@pytest.mark.parametrize("ver", ["GC", "raw"])
@pytest.mark.parametrize("ds_dim", [1, 2])
def test_scenes_vs_oracle_per_scene_constants(ver, exact, ds_dim):
    S, N = 24, 122
    p, v, ds, d, act = scenes(S, N, seed=11 + ds_dim, ds_dim=ds_dim)
    prm = rand_params(S, seed=5)
    a, q, arr = run(model(ver, exact), p, v, ds, d, act, prm)
    for s in range(S):
        check_scene(a[s], q[s], arr[s], p[s], v[s], ds[s], d[s], act[s], ver, prm[s])


def test_desired_speed_without_trailing_axis():
    p, v, ds, d, act = scenes(5, 40, seed=3)
    m = model()
    a1 = run(m, p, v, ds, d, act)
    a2 = run(m, p, v, ds[..., 0], d, act)
    for x, y in zip(a1, a2):
        assert np.array_equal(x, y, equal_nan=True)


# ---- golden circle (main_mlapm.py) inside a batch ------------------------------------------------------------------
def circle_batch(t_pos, t_vel, t_mask, g, S=9, k=4, N=16, seed=0):
    p, v, ds, d, act = scenes(S, N, seed=seed)
    ds = np.repeat(ds, 2, axis=-1)
    n = t_pos.shape[0]
    p[k] = np.nan; v[k] = np.nan; d[k] = np.nan; ds[k] = np.nan; act[k] = False
    p[k, :n], v[k, :n], d[k, :n], ds[k, :n], act[k, :n] = t_pos, t_vel, g["destination"], g["desired_speed"], t_mask
    return p, v, ds, d, act


def test_golden_circle_in_batch():
    from piml_b200.mlapm import rollout_scenes
    g = group(golden("mlapm"), "circle")
    pos, vel, mask = g["position"], g["velocity"], g["mask"]
    n, k = pos.shape[0], 4
    m = model()
    worst = 0.0
    for t in range(pos.shape[1] - 1):
        mt = mask[:, t]
        if not mt.any():
            break
        p, v, ds, d, act = circle_batch(pos[:, t], vel[:, t], mt, g, seed=t)
        a, q, arr = run(m, p, v, ds, d, act)
        worst = max(worst, rel_vec_err(a[k, :n][mt], vel[mt, t + 1]))
        assert np.array_equal(arr[k, :n][mt], ~mask[mt, t + 1])
    assert worst < TOL, worst
    p, v, ds, d, act = circle_batch(pos[:, 0], vel[:, 0], np.ones(n, bool), g, seed=99)
    P_, V_, M_ = rollout_scenes(m, cu(p), cu(v), cu(ds), cu(d), 200, DT, RADIUS, active=cu(act, torch.bool))
    P_, M_ = npy(P_), npy(M_)
    assert np.array_equal(M_[k, :n], mask)
    assert not M_[k, n:].any()
    drift = np.nanmax(np.linalg.norm(P_[k, :n] - pos, axis=-1))
    print(f"free-running drift over 200 steps inside a batch: {drift:.3e} m")
    assert drift < 1e-3


# ---- a scene's result does not depend on the batch -----------------------------------------------------------------
@pytest.mark.parametrize("exact", [False, True])
def test_batch_independence(exact):
    m = model("GC", exact)
    p, v, ds, d, act = scenes(1, 90, seed=21, inactive=(0.0, 0.0))
    alone = run(m, p, v, ds, d, act)
    again = run(m, p, v, ds, d, act)
    for x, y in zip(alone, again):
        assert np.array_equal(x, y, equal_nan=True)
    # the same agents, in the same order, in slots of wider scenes (other batch sizes and packing modes)
    for S, N, k in ((3, 128, 1), (40, 257, 17), (5, 300, 4), (2, 1000, 0)):
        P_, V_, DS, D_, A_ = scenes(S, N, seed=N)
        slots = np.sort(np.random.default_rng(N).choice(N, 90, replace=False))
        A_[k] = False
        P_[k, :] = np.nan
        P_[k, slots], V_[k, slots], DS[k, slots], D_[k, slots], A_[k, slots] = p[0], v[0], ds[0], d[0], True
        out = run(m, P_, V_, DS, D_, A_)
        for x, y in zip(out, alone):
            assert np.array_equal(x[k, slots], y[0], equal_nan=True)


# ---- constants sweep -------------------------------------------------------------------------------------------------
def test_constants_sweep_one_crowd():
    S, N = 32, 200
    p, v, ds, d, act = scenes(1, N, seed=8, inactive=(0.0, 0.0))
    prm = rand_params(S, seed=9)
    rep = [np.repeat(x, S, axis=0) for x in (p, v, ds, d, act)]
    a, q, arr = run(model(), *rep, prm)
    for s in range(S):
        check_scene(a[s], q[s], arr[s], p[0], v[0], ds[0], d[0], act[0], "GC", prm[s])
    # params=None: the constructor's constants
    a0, q0, arr0 = run(model(), *rep)
    for s in (0, S - 1):
        check_scene(a0[s], q0[s], arr0[s], p[0], v[0], ds[0], d[0], act[0], "GC", GC_ROW)


# ---- inactive slots, NaN, empty and single-agent scenes ------------------------------------------------------------
def test_inactive_and_nan():
    S, N = 6, 50
    m = model()
    p, v, ds, d, act = scenes(S, N, seed=4, nan_inactive=False)
    base = run(m, p, v, ds, d, act)
    pn, vn, dsn, dn = p.copy(), v.copy(), ds.copy(), d.copy()
    pn[~act] = np.nan; vn[~act] = np.inf; dsn[~act] = np.nan; dn[~act] = np.nan
    for x, y in zip(run(m, pn, vn, dsn, dn, act), base):
        assert np.array_equal(x, y, equal_nan=True)
    # one NaN in an active agent of scene 2 poisons that scene only (mlapm.py: the pair term is a product)
    j = int(np.nonzero(act[2])[0][5])
    pn = p.copy(); pn[2, j] = np.nan
    out = run(m, pn, v, ds, d, act)
    assert np.isnan(out[0][2]).all()
    for s in (0, 1, 3, 4, 5):
        for x, y in zip(out, base):
            assert np.array_equal(x[s], y[s], equal_nan=True)
    # no agent at all: all NaN; one agent: only the destination term (no pair)
    act2 = act.copy()
    act2[0] = False
    act2[1] = False; act2[1, 7] = True
    a, q, arr = run(m, p, v, ds, d, act2)
    assert np.isnan(a[0]).all() and np.isnan(q[0]).all() and not arr[0].any()
    check_scene(a[1], q[1], arr[1], p[1], v[1], ds[1], d[1], act2[1], "GC")
    dx = (d[1, 7] - p[1, 7]).astype(np.float64)
    ed = dx / np.linalg.norm(dx)
    want = v[1, 7] + ((ds[1, 7, 0] * ed - v[1, 7]) / 0.5) * DT
    assert np.allclose(a[1, 7], want, rtol=1e-6, atol=1e-6)


# ---- shape boundaries ------------------------------------------------------------------------------------------------
# 1..32: one power-of-two lane group per scene (several scenes per warp); 33..256: whole warps per scene, several
# scenes per CTA; from 257: the rows split over CTAs (balanced chunks of whole warps); 8192: the supported maximum.
@pytest.mark.parametrize("N", [1, 2, 7, 8, 9, 31, 32, 33, 64, 127, 128, 129, 255, 256, 257, 511, 513, 2000])
def test_shape_boundaries(N):
    S = 37
    p, v, ds, d, act = scenes(S, N, seed=N)
    a, q, arr = run(model(), p, v, ds, d, act)
    for s in range(S) if N <= 256 else (0, 1, S // 2, S - 1):
        check_scene(a[s], q[s], arr[s], p[s], v[s], ds[s], d[s], act[s], "GC")


@pytest.mark.parametrize("exact", [False, True])
def test_supported_maximum_and_row_split(exact):
    S, N = 8, MAX_N
    p, v, ds, d, act = scenes(S, N, seed=81, inactive=(0.0, 0.1))
    a, q, arr = run(model("GC", exact), p, v, ds, d, act)
    for s in range(S):
        n = int(act[s].sum())
        for r0 in (0, n // 2 - 20, n - 40):                         # rows of the first, a middle and the last chunk
            check_scene(a[s], q[s], arr[s], p[s], v[s], ds[s], d[s], act[s], "GC", rows=(r0, r0 + 40))


def test_above_maximum_is_rejected_before_launch():
    import piml_b200 as P
    p, v, ds, d, act = scenes(1, MAX_N + 1, seed=1)
    before = P._lib.launch_count()
    with pytest.raises(RuntimeError, match="MLAPM.advance"):
        run(model(), p, v, ds, d, act)
    assert P._lib.launch_count() == before


@pytest.mark.parametrize("S,N", [(1, 122), (70001, 7), (70000, 129)])
def test_scene_count(S, N):
    p, v, ds, d, act = scenes(S, N, seed=S)
    a, q, arr = run(model(), p, v, ds, d, act)
    for s in sorted({0, 1, S // 3, S - 2, S - 1} & set(range(S))):
        check_scene(a[s], q[s], arr[s], p[s], v[s], ds[s], d[s], act[s], "GC")


# ---- against MLAPM.advance on each compacted scene -----------------------------------------------------------------
@pytest.mark.parametrize("ver", ["GC", "raw"])
def test_against_advance(ver):
    S, N = 12, 300
    m = model(ver)
    p, v, ds, d, act = scenes(S, N, seed=17)
    a, q, arr = run(m, p, v, ds, d, act)
    for s in range(S):
        idx = np.nonzero(act[s])[0]
        wa, wq, warr = m.advance(cu(p[s, idx]), cu(v[s, idx]), cu(ds[s, idx]), cu(d[s, idx]), DT, RADIUS)
        assert err(a[s, idx], npy(wa).astype(np.float64), v[s, idx]) < TOL
        assert np.allclose(q[s, idx], npy(wq), rtol=0, atol=1e-5)
        assert np.array_equal(arr[s, idx], npy(warr))


# ---- rollout: semantics of mlapm.rollout per scene, no host synchronisation ---------------------------------------
def test_rollout_scenes_matches_rollout_per_scene():
    from piml_b200.mlapm import rollout, rollout_scenes
    S, N, T = 4, 20, 60
    m = model()
    p, v, ds, d, act = scenes(S, N, seed=31, inactive=(0.0, 0.0))
    d = (p + np.random.default_rng(0).normal(0, 2.0, p.shape)).astype(np.float32)   # most agents arrive
    P_, V_, M_ = [npy(x) for x in rollout_scenes(m, cu(p), cu(v), cu(ds), cu(d), T, DT, RADIUS)]
    assert M_[:, :, 0].all() and (~M_[:, :, -1]).any()
    for s in range(S):
        p1, v1, m1 = [npy(x) for x in rollout(m, cu(p[s]), cu(v[s]), cu(ds[s]), cu(d[s]), T, DT, RADIUS)]
        assert np.array_equal(M_[s], m1)
        assert np.array_equal(np.isnan(P_[s]), np.isnan(p1))
        assert np.nanmax(np.abs(P_[s] - p1)) < 1e-3


def test_rollout_step_captures_in_cuda_graph():
    from piml_b200.mlapm import rollout_scenes
    m = model()
    p, v, ds, d, act = [cu(x) if x.dtype != bool else cu(x, torch.bool) for x in scenes(64, 122, seed=2)]
    want = [x.clone() for x in rollout_scenes(m, p, v, ds, d, 1, DT, RADIUS, active=act)]
    side = torch.cuda.Stream()
    side.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(side):                                 # warm-up outside the capture
        rollout_scenes(m, p, v, ds, d, 1, DT, RADIUS, active=act)
    torch.cuda.current_stream().wait_stream(side)
    g = torch.cuda.CUDAGraph()
    with torch.cuda.graph(g):
        out = rollout_scenes(m, p, v, ds, d, 1, DT, RADIUS, active=act)
    g.replay()
    torch.cuda.synchronize()
    for x, y in zip(out, want):
        assert torch.equal(torch.nan_to_num(x.float(), nan=7.0), torch.nan_to_num(y.float(), nan=7.0))
