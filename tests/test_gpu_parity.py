"""Parity of the CUDA path (through the C ABI, via the piml_b200 host adapters) against the golden vectors of the
unmodified reference and against the CPU oracle on seeded synthetic inputs.  Run on the B200 box: pytest -m gpu.

Gates (SURVEY.md 8d): neighbour sets / distances / features bit-exact; forces, MLP outputs within 1e-5 relative
(per-vector 2-norm); positions and velocities of a re-synchronised rollout step bit-exact.
"""
import numpy as np
import pytest
import torch

from oracle import oracle as O
from tests.util import accel_err, golden, group, rel_vec_err, untied_finite, valid_sets

pytestmark = pytest.mark.gpu

TOL = 1e-5


def cu(x, dtype=torch.float32):
    return torch.as_tensor(np.asarray(x), dtype=dtype).cuda()


def npy(t):
    return t.detach().cpu().numpy()


FEATURE_CASES = ["gc", "gc_window", "ucy", "toy", "syn512", "syn300_wide", "channelled"]


@pytest.mark.parametrize("case", FEATURE_CASES)
def test_relative_features_golden(case):
    import piml_b200 as P
    g = group(golden("features"), case)
    kp, ap, tp, ko, ao, to = [int(v) for v in g["params"]]
    vel, acc = cu(g["velocity"]), cu(g["acceleration"])
    ped = P.Pedestrians()
    pf, of, df, (pi, pd, oi, od) = ped.get_relative_features(
        cu(g["position"]), vel, acc, cu(g["destination"]), cu(g["obstacles"]), kp, ap, tp, ko, ao, to,
        return_selection=True)
    assert np.array_equal(npy(df), g["dest_features"])
    # slot order inside the radius is (distance, index) like the reference; compare slot by slot
    assert np.array_equal(npy(pf), g["ped_features"])
    assert np.array_equal(npy(of), g["obs_features"])
    assert np.array_equal(npy(vel), g["velocity_after"]) and np.array_equal(npy(acc), g["acceleration_after"])
    assert valid_sets(npy(pi), npy(pd), tp) == valid_sets(g["ped_idx"], g["ped_dist"], tp)
    assert valid_sets(npy(oi), npy(od), to) == valid_sets(g["obs_idx"], g["obs_dist"], to)


@pytest.mark.parametrize("case", FEATURE_CASES)
def test_heading_and_selection_helpers_golden(case):
    import piml_b200 as P
    g = group(golden("features"), case)
    kp, ap, tp, ko, ao, to = [int(v) for v in g["params"]]
    ped = P.Pedestrians()
    head = ped.get_heading_direction(cu(g["velocity_after"]))
    assert np.array_equal(npy(head), g["heading"])
    pos = cu(g["position"])
    dist, idx = ped.get_nearby_obj_in_sight(pos, pos, head, kp, ap)
    assert np.array_equal(npy(dist), g["ped_dist"])
    fin = untied_finite(g["ped_dist"])
    assert np.array_equal(npy(idx)[fin], g["ped_idx"][fin].astype(np.int64))
    obs = cu(g["obstacles"])
    T = pos.shape[-3]
    obs_t = obs.unsqueeze(-3).repeat(*([1] * (obs.dim() - 2) + [T] + [1, 1]))      # data.py:502-503
    dist, idx = ped.get_nearby_obj_in_sight(pos, obs_t, head, ko, ao)
    assert np.array_equal(npy(dist), g["obs_dist"])
    fin = untied_finite(g["obs_dist"])
    assert np.array_equal(npy(idx)[fin], g["obs_idx"][fin].astype(np.int64))


def _crowd(B, N, M, seed, rho=0.5, nan_frac=0.05):
    rng = np.random.default_rng(seed)
    L = np.sqrt(N / rho)
    p = (rng.random((B, N, 2)) * L).astype(np.float32)
    d = (rng.random((B, N, 2)) * L).astype(np.float32)
    v = rng.normal(0, 1, (B, N, 2)).astype(np.float32)
    a = rng.normal(0, 1, (B, N, 2)).astype(np.float32)
    gone = rng.random((B, N)) < nan_frac
    p[gone] = np.nan
    d[gone] = np.nan
    v[gone] = 0
    v[rng.random((B, N)) < 0.03] = 0                      # stationary agents see nobody at 90 degrees
    obs = (rng.random((M, 2)) * L).astype(np.float32)
    return p, v, a, d, obs


# (B, N, M) chosen to hit the three lane-group variants of the kernel: G=32, G=8, G=1 (see pick_group)
@pytest.mark.parametrize("B,N,M", [(1, 3001, 2000), (8, 1500, 700), (40, 2000, 2000), (3, 7, 3), (2, 129, 0)])
def test_relative_features_vs_oracle(B, N, M):
    import piml_b200 as P
    p, v, a, d, obs = _crowd(B, N, M, seed=B * 1000 + N)
    want = O.relative_features(p, v.copy(), a.copy(), d, obs, 6, 90, 4, 10, 90, 4, return_selection=True)
    ped = P.Pedestrians()
    got = ped.get_relative_features(cu(p), cu(v), cu(a), cu(d), cu(obs).reshape(M, 2), 6, 90, 4, 10, 90, 4,
                                    return_selection=True)
    assert np.array_equal(npy(got[0]), want[0])
    assert np.array_equal(npy(got[2]), want[2])
    if M:
        assert np.array_equal(npy(got[1]), want[1])
    wpi, wpd, woi, wod = want[3]
    gpi, gpd, goi, god = [npy(x) for x in got[3]]
    assert valid_sets(gpi, gpd, 4) == valid_sets(wpi, wpd, 4)
    if M:
        assert valid_sets(goi, god, 4) == valid_sets(woi, wod, 4)


def test_relative_features_large_k_and_angles():
    import piml_b200 as P
    p, v, a, d, obs = _crowd(2, 400, 300, seed=5)
    for kp, ko, ang, thr in ((12, 20, 60, 6), (32, 32, 150, 3), (1, 1, 90, 4)):
        want = O.relative_features(p, v.copy(), a.copy(), d, obs, kp, ang, thr, ko, ang, thr)
        got = P.Pedestrians().get_relative_features(cu(p), cu(v), cu(a), cu(d), cu(obs), kp, ang, thr, ko, ang, thr)
        for w, g_ in zip(want, got):
            assert np.array_equal(npy(g_), w)


def _set_algo(algo):
    from piml_b200 import _lib as L
    L.check(L.load().piml_set_feature_algorithm(algo), "piml_set_feature_algorithm")


def _features_both_ways(args, golden_check=None):
    """Run get_relative_features with the all-pairs kernel and with the cell list; every output must be bit-identical."""
    import piml_b200 as P
    outs = []
    try:
        for algo in (1, 2):
            _set_algo(algo)
            ins = [cu(x) for x in args[:5]]
            r = P.Pedestrians().get_relative_features(*ins, *args[5:], return_selection=True)
            outs.append([npy(x) for x in r[:3]] + [npy(x) for x in r[3]] + [npy(ins[1]), npy(ins[2])])
    finally:
        _set_algo(0)
    for x, y in zip(*outs):
        assert np.array_equal(x, y, equal_nan=True)
    return outs[1]


@pytest.mark.parametrize("B,N,M", [(1, 5003, 2000), (1, 20000, 2000), (3, 4500, 300), (5, 300, 40), (2, 129, 0)])
def test_cell_list_identical_to_all_pairs(B, N, M):
    """The uniform-grid variant (features_cells.cu) returns the same features, indices, distances and side effects as
    the all-pairs kernel, and (where the C oracle finishes in seconds) the same as the oracle."""
    p, v, a, d, obs = _crowd(B, N, M, seed=B * 77 + N)
    v[0, 3] = np.nan; a[0, 4] = np.nan                    # in-place NaN -> 0 side effect on both paths
    got = _features_both_ways((p, v, a, d, obs.reshape(M, 2), 6, 90, 4, 10, 90, 4))
    if B * N * N <= 3e8:
        want = O.relative_features(p, v.copy(), a.copy(), d, obs, 6, 90, 4, 10, 90, 4)
        assert np.array_equal(got[0], want[0]) and np.array_equal(got[2], want[2])
        if M:
            assert np.array_equal(got[1], want[1])


def test_cell_list_awkward_geometry():
    """Negative coordinates, far outliers (the (1e4,1e4) dummy obstacles of data.py:102-103), points beyond the int16
    cell range, dense clumps (many agents per cell), wide angle (self selected), unequal thresholds, per-channel
    obstacles, time axis with heading fill."""
    rng = np.random.default_rng(3)
    Cc, T, N, M = 2, 3, 700, 60
    p = (rng.normal(0, 15, (Cc, T, N, 2))).astype(np.float32)
    p[:, :, :200] = (rng.normal(0, 0.7, (Cc, T, 200, 2)) + 5).astype(np.float32)      # clump
    p[:, :, 200:210] = 1e4
    p[:, :, 210:215] = (rng.random((Cc, T, 5, 2)) * 3 + 2.5e5).astype(np.float32)     # clamped cells
    p[:, :, 215:220] = (-2.5e5 - rng.random((Cc, T, 5, 2)) * 3).astype(np.float32)
    p[0, :, 300] = np.nan
    d = rng.normal(0, 15, (Cc, T, N, 2)).astype(np.float32)
    v = rng.normal(0, 1, (Cc, T, N, 2)).astype(np.float32)
    v[:, 1, ::5] = 0
    a = rng.normal(0, 1, (Cc, T, N, 2)).astype(np.float32)
    obs = rng.normal(0, 15, (Cc, M, 2)).astype(np.float32)
    obs[:, :2] = 1e4
    got = _features_both_ways((p, v, a, d, obs, 8, 100, 3, 12, 120, 5))
    want = O.relative_features(p, v.copy(), a.copy(), d, obs, 8, 100, 3, 12, 120, 5)
    for g_, w in zip(got[:3], want):
        assert np.array_equal(g_, w)


def test_cell_list_rollout_feature_rebuild():
    """piml_state_features_f32 (the per-step rebuild incl. self_features) through the cell list == all pairs."""
    from piml_b200.rollout import state_features
    p, v, a, d, obs = _crowd(1, 6000, 500, seed=9)
    hist = v.copy(); ds = np.full((1, 6000), 1.3, np.float32)
    res = []
    try:
        for algo in (1, 2):
            _set_algo(algo)
            r = state_features(cu(p), cu(v), cu(a), cu(d), cu(obs), cu(hist), cu(ds), 6, 90, 4, 10, 90, 4)
            res.append([npy(x) for x in r])
    finally:
        _set_algo(0)
    for x, y in zip(*res):
        assert np.array_equal(x, y)


def test_collision_label():
    import piml_b200 as P
    g = group(golden("features"), "gc")
    want = O.collision_label(g["ped_features"])
    got = P.Pedestrians.calculate_collision_label(cu(g["ped_features"]))
    assert np.array_equal(npy(got), want)


# ---- MLAPM -------------------------------------------------------------------------------------------------------
GC_KW = dict(version='GC', tau=0.5, A=7.55, B=-3.00, C=0.2, D=-0.3, theta=56)


@pytest.mark.parametrize("exact", [False, True])
@pytest.mark.parametrize("case,ver", [("syn257", "raw"), ("syn257", "GC"), ("syn1000", "raw"), ("syn1000", "GC")])
def test_mlapm_step_golden(case, ver, exact):
    import piml_b200 as P
    g = group(golden("mlapm"), case)
    kw = dict(GC_KW, version=ver, exact_math=exact)
    act = P.MLAPM(**kw).step(cu(g["position"]), cu(g["velocity"]), cu(g["desired_speed"]), cu(g["destination"]),
                             dt=0.08)
    assert rel_vec_err(npy(act), g[ver + "/action"]) < TOL


@pytest.mark.parametrize("exact", [False, True])
def test_mlapm_params_golden(exact):
    import piml_b200 as P
    g = group(golden("mlapm"), "syn300b")
    tau, A, B, C_, D, th, dt = [float(v) for v in g["params"]]
    m = P.MLAPM(version='GC', tau=tau, A=A, B=B, C=C_, D=D, theta=th, exact_math=exact)
    act = m.step(cu(g["position"]), cu(g["velocity"]), cu(g["desired_speed"]), cu(g["destination"]), dt=dt)
    assert rel_vec_err(npy(act), g["GC/action"]) < TOL


def test_mlapm_circle_rollout_golden():
    """main_mlapm.py scene: re-synchronised steps within 1e-5; free-running drift over 200 steps reported."""
    import piml_b200 as P
    from piml_b200.mlapm import rollout
    g = group(golden("mlapm"), "circle")
    pos, vel, mask = g["position"], g["velocity"], g["mask"]
    model = P.MLAPM(**GC_KW)
    worst = 0.0
    for t in range(pos.shape[1] - 1):
        m = mask[:, t]
        if not m.any():
            break
        act, pnew, arrived = model.advance(cu(pos[m, t]), cu(vel[m, t]), cu(g["desired_speed"][m]),
                                           cu(g["destination"][m]), 0.08, 0.3)
        worst = max(worst, rel_vec_err(npy(act), vel[m, t + 1]))
        assert np.array_equal(npy(arrived), ~mask[m, t + 1])
    assert worst < TOL, worst
    p, v, mk = rollout(model, cu(pos[:, 0]), cu(vel[:, 0]), cu(g["desired_speed"]), cu(g["destination"]), 200)
    assert p.shape[1] == pos.shape[1] and np.array_equal(npy(mk), mask)
    drift = np.nanmax(np.linalg.norm(npy(p) - pos, axis=-1))
    print(f"free-running drift over {p.shape[1] - 1} steps: {drift:.3e} m")
    assert drift < 1e-3


@pytest.mark.parametrize("N", [4099, 8192])
def test_mlapm_vs_oracle_and_row_ranges(N):
    import piml_b200 as P
    rng = np.random.default_rng(N)
    L = np.sqrt(N / 0.5)
    p = (rng.random((N, 2)) * L).astype(np.float32)
    d = (rng.random((N, 2)) * L).astype(np.float32)
    v = rng.normal(0, 1, (N, 2)).astype(np.float32)
    ds = (1.34 + 0.3 * rng.normal(0, 1, (N, 1))).astype(np.float32)
    want = O.mlapm_step(p, v, ds, d, 0.08, "GC")
    model = P.MLAPM(**GC_KW)
    full = npy(model.step(cu(p), cu(v), cu(ds), cu(d), 0.08))
    assert rel_vec_err(full, want) < TOL
    exact = npy(P.MLAPM(**dict(GC_KW, exact_math=True)).step(cu(p), cu(v), cu(ds), cu(d), 0.08))
    assert rel_vec_err(exact, want) < TOL
    # agent-sharded row ranges reproduce the full result bit-for-bit (SURVEY A.2b multi-GPU row)
    r0, r1 = N // 3 + 1, 2 * N // 3
    part = npy(model.step(cu(p), cu(v), cu(ds), cu(d), 0.08, rows=(r0, r1)))
    assert rel_vec_err(part, want[r0:r1]) < TOL


def test_mlapm_nan_poisons_like_reference():
    """mlapm.py: view*A*exp(..)*direc is a product, so one NaN position makes every force NaN."""
    import piml_b200 as P
    g = group(golden("mlapm"), "syn257")
    p = g["position"].copy()
    p[17] = np.nan
    act = npy(P.MLAPM(**GC_KW).step(cu(p), cu(g["velocity"]), cu(g["desired_speed"]), cu(g["destination"]), 0.08))
    want = O.mlapm_step(p, g["velocity"], g["desired_speed"], g["destination"], 0.08, "GC")
    assert np.isnan(want).all() and np.isnan(act).all()


def _mlapm_algorithm(algo):
    from piml_b200 import _lib as L
    L.check(L.load().piml_set_mlapm_algorithm(algo), "piml_set_mlapm_algorithm")


@pytest.mark.parametrize("ver", ["GC", "raw"])
@pytest.mark.parametrize("N", [257, 1024, 1500, 2048, 2049, 5000, 8192])
def test_mlapm_symmetric_evaluation(N, ver):
    """The unordered-pair kernel (every pair once, both directions; odd / even / single block schedules, padded block
    tails) against the oracle and against the ordered-pair kernel, incl. stationary agents (view gate false)."""
    import piml_b200 as P
    rng = np.random.default_rng(7 * N + len(ver))
    L = np.sqrt(N / 0.5)
    p = (rng.random((N, 2)) * L).astype(np.float32)
    d = (rng.random((N, 2)) * L).astype(np.float32)
    v = rng.normal(0, 1, (N, 2)).astype(np.float32)
    v[rng.random(N) < 0.05] = 0.0
    ds = (1.34 + 0.3 * rng.normal(0, 1, (N, 1))).astype(np.float32)
    want = O.mlapm_step(p, v, ds, d, 0.08, ver)
    model = P.MLAPM(**dict(GC_KW, version=ver))
    try:
        _mlapm_algorithm(2)
        before = P._lib.launch_count()
        sym, pnew, arrived = model.advance(cu(p), cu(v), cu(ds), cu(d), 0.08, 0.3)
        sym = npy(sym)
        again = npy(model.step(cu(p), cu(v), cu(ds), cu(d), 0.08))
        _mlapm_algorithm(1)
        ordered, pnew_o, arrived_o = model.advance(cu(p), cu(v), cu(ds), cu(d), 0.08, 0.3)
    finally:
        _mlapm_algorithm(0)
    # action = v + F dt: where the two nearly cancel, fp32 rounding is relative to the operand v, not to the small
    # result (the reference's own fp32 result is 2.6e-6 of |action| away from an fp64 evaluation on such an agent,
    # scripts/diag_sym.py), so the scale of the gate is max(|action|, |v|)
    def err(got, ref):
        num = np.linalg.norm(np.asarray(got, np.float64) - ref, axis=-1)
        den = np.maximum(np.maximum(np.linalg.norm(ref, axis=-1), np.linalg.norm(v, axis=-1)), 1e-6)
        return float((num / den).max())
    assert np.isfinite(sym).all()
    assert err(sym, want) < TOL
    assert rel_vec_err(sym, want) < 3 * TOL
    assert np.array_equal(sym, again)                       # deterministic: fixed summation order, no atomics
    assert err(sym, npy(ordered)) < TOL
    assert np.array_equal(npy(arrived), npy(arrived_o))
    assert np.allclose(npy(pnew), npy(pnew_o), rtol=0, atol=1e-5)


def test_mlapm_symmetric_nan_poisons_like_reference():
    import piml_b200 as P
    g = group(golden("mlapm"), "syn1000")
    p = g["position"].copy()
    p[801] = np.nan
    try:
        _mlapm_algorithm(2)
        act = npy(P.MLAPM(**GC_KW).step(cu(p), cu(g["velocity"]), cu(g["desired_speed"]), cu(g["destination"]), 0.08))
    finally:
        _mlapm_algorithm(0)
    assert np.isnan(act).all()


# ---- SFM -----------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("key", ["v0/gc1560", "v0/ucy", "v1/gc2344", "v1/ucy", "v2/gc2344"])
def test_calc_acceleration_golden(key):
    import piml_b200 as P
    z = golden("sfm")
    ver, ds = key.split("/")
    out = npy(P.calc_acceleration(cu(z["ped"]), ver, ds))
    assert rel_vec_err(out, z[key]) < TOL
    assert np.array_equal(out == 0, z[key] == 0)
    outc = npy(P.calc_acceleration(cu(z["ped_c"]), "v2", "gc2344"))
    assert rel_vec_err(outc, z["v2c/gc2344"]) < TOL


# ---- interaction networks ------------------------------------------------------------------------------------------
def _mirror_model(z, kind):
    from tests.golden_args import model_args
    from piml_b200 import models as M
    g = group(z, kind)
    args = model_args(kind, g["cfg"], str(g["dataset_name"]))
    m = M.CLASSES[kind](args)
    m.load_state_dict({k[3:]: torch.from_numpy(v) for k, v in g.items() if k.startswith("sd/")})
    return g, m.cuda().eval()


@pytest.mark.parametrize("kind", ["pinnsf_bm", "pinnsf_m", "pinnsf_bottleneck", "pinnsf"])
def test_pinnsf_forward_golden(kind):
    z = golden("models")
    g, m = _mirror_model(z, kind)
    for suffix in ("", "c"):
        tag = "_c" if suffix else ""
        out = m(cu(z["ped" + tag]), cu(z["obs" + tag]), cu(z["self" + tag]))
        refs = [g[f"out{suffix}{i}"] for i in range(len(out))]
        assert len(out) == len([k for k in g if k.startswith("out" + suffix) and k[len("out" + suffix):].isdigit()])
        for i, (o, ref) in enumerate(zip(out, refs)):
            o = npy(o)
            assert o.shape == ref.shape, (kind, suffix, i, o.shape, ref.shape)
            if o.ndim >= 2 and o.shape[-1] in (2, 128, 32):
                err = rel_vec_err(o, ref, floor=1e-3)
            else:
                err = float(np.abs(o - ref).max())
            assert err < TOL, (kind, suffix, i, err)


@pytest.mark.parametrize("kind", ["pinnsf_bm", "pinnsf_m"])
def test_pinnsf_forward_tensor_cores_golden(kind):
    """The tcgen05 (3xTF32) forward against the reference's own outputs: acceleration within 1e-5 of the operand scale
    (SURVEY.md 8d; accel_err), for (N,.) and channelled (C,N,.) inputs."""
    from piml_b200 import models as M
    z = golden("models")
    g, m = _mirror_model(z, kind)
    ptc = M.pack_device_tc(m.state_dict(), m.spec)
    assert ptc is not None
    packed = M.pack_device(m.state_dict(), m.spec)
    for suffix in ("", "c"):
        tag = "_c" if suffix else ""
        ped, obs, slf = cu(z["ped" + tag]), cu(z["obs" + tag]), cu(z["self" + tag])
        out = M.pinnsf_forward(m.spec, packed, ped, obs, slf, need_msgs=False, packed_tc=ptc)
        ref = g[f"out{suffix}0"]
        if suffix:      # channelled: the destination norm is per channel and component (SURVEY.md B-3), compare directly
            err = rel_vec_err(npy(out[0]), ref, floor=1e-1)
        else:
            err = accel_err(npy(out[0]), ref, z["self"], float(g["tau"]))
        assert err < TOL, (kind, suffix, err)


def test_tensor_core_path_declines_unsupported_nets():
    """Widths that are not multiples of 32 cannot run on the tcgen05 path: pack_device_tc says so (-> FP32 kernel)."""
    from piml_b200 import models as M
    z = golden("models")
    for kind in ("pinnsf_bottleneck", "pinnsf"):
        g, m = _mirror_model(z, kind)
        assert M.pack_device_tc(m.state_dict(), m.spec) is None


@pytest.mark.parametrize("kind,R,kp,ko,chan,has_obs", [
    ("pinnsf_bm", 21, 6, 10, 0, True), ("pinnsf_bm", 3001, 6, 10, 0, True), ("pinnsf_bottleneck", 999, 5, 3, 0, True),
    ("pinnsf_m", 257, 6, 10, 0, True), ("pinnsf", 640, 6, 0, 0, False), ("pinnsf_bm", 640, 6, 2, 5, True),
    ("pinnsf_m", 1200, 4, 7, 6, True)])
def test_pinnsf_forward_tensor_cores_vs_fp32_kernel(kind, R, kp, ko, chan, has_obs):
    """tcgen05 forward vs the FP32-pipe kernel on random inputs: tile tails, both decoder placements, no obstacle
    branch, channelled destination norm, 2-d messages of the per-slot-decoder models."""
    from piml_b200 import models as M
    from .golden_args import base_args
    args = base_args(model=kind, dataset_name="gc1560", obs_feature_dim=6 if has_obs else 0)
    torch.manual_seed(R)
    net = M.CLASSES[kind](args).cuda().eval()
    g = torch.Generator().manual_seed(R + 1)
    lead = (chan, R // chan) if chan else (R,)
    ped = torch.randn(*lead, kp, 6, generator=g).cuda()
    ped[..., -1, :] = 0
    obs = torch.randn(*lead, max(ko, 1), 6, generator=g)[..., :ko, :].cuda()
    slf = torch.randn(*lead, 7, generator=g).cuda()
    packed = M.pack_device(net.state_dict(), net.spec)
    ptc = M.pack_device_tc(net.state_dict(), net.spec)
    need = net.spec.kind == 0 and not net.spec.coll_dims
    ref = M.pinnsf_forward(net.spec, packed, ped, obs, slf, need_msgs=True)
    got = M.pinnsf_forward(net.spec, packed, ped, obs, slf, need_msgs=need, packed_tc=ptc)
    # error relative to the scale of what is summed (messages + destination term), like the FP32 kernel's gate
    err = accel_err(npy(got[0]).reshape(-1, 2), npy(ref[0]).reshape(-1, 2), npy(slf).reshape(-1, 7), net.spec.tau)
    assert err < TOL, err
    if need:
        scale = float(ref[1].abs().max())
        assert float((got[1] - ref[1]).abs().max()) < TOL * scale
        if has_obs:
            assert float((got[2] - ref[2]).abs().max()) < TOL * float(ref[2].abs().max())


@pytest.mark.parametrize("width,kernel", [(128, "pinnsf_tc16_kernel"), (96, "pinnsf_tc_kernel")])
@pytest.mark.parametrize("R,kp,ko", [(700, 1, 1), (401, 1, 7), (333, 2, 1), (130, 3, 1)])
def test_tensor_core_forward_with_one_slot_per_agent(R, kp, ko, width, kernel):
    """topk = 1 packs 128 agents into a dense tile: 256 slot sums for 128 threads (the dense mode of both tensor-core
    kernels wrote only the first 64 agents' sums until round 2; found by scripts/fuzz_parity.py's fused-step family).
    Width 128 runs on the 16-bit kernel; width 96, a multiple of 32 that the 16-bit kernel does not take, on the
    tf32 kernel.  The profiler shows which one ran."""
    from piml_b200 import models as M
    from .golden_args import base_args
    args = base_args(model="pinnsf_bm", dataset_name="gc1560", encoder_hidden_size=width, processor_hidden_size=width)
    net = M.CLASSES["pinnsf_bm"](args).cuda().eval()
    g = torch.Generator().manual_seed(R)
    ped = torch.randn(R, kp, 6, generator=g).cuda()
    obs = torch.randn(R, ko, 6, generator=g).cuda()
    obs[::3] = 0
    slf = torch.randn(R, 7, generator=g).cuda()
    packed = M.pack_device(net.state_dict(), net.spec)
    ptc = M.pack_device_tc(net.state_dict(), net.spec)
    ref = M.pinnsf_forward(net.spec, packed, ped, obs, slf, need_msgs=True)
    with torch.profiler.profile(activities=[torch.profiler.ProfilerActivity.CUDA]) as prof:
        M.pinnsf_forward(net.spec, packed, ped, obs, slf, need_msgs=False, packed_tc=ptc)
        torch.cuda.synchronize()
    names = [e.name for e in prof.events() if e.device_type == torch.autograd.DeviceType.CUDA]
    assert any(kernel + "(" in n or kernel + "<" in n for n in names), names
    for need in (False, True):
        got = M.pinnsf_forward(net.spec, packed, ped, obs, slf, need_msgs=need, packed_tc=ptc)
        err = accel_err(npy(got[0]), npy(ref[0]), npy(slf), net.spec.tau)
        assert err < TOL, (need, err)


@pytest.mark.parametrize("R,kp,ko,pz,chan", [(3001, 6, 10, 0.6, 0), (700, 6, 10, 1.0, 0), (129, 6, 10, 0.0, 0),
                                             (5000, 6, 0, 0.3, 0), (1280, 4, 7, 0.8, 5)])
def test_tensor_core_compact_mode_is_bit_identical(R, kp, ko, pz, chan):
    """Zero-padded slot rows all yield the same message f(0) (model.py:1188-1194 does not mask them), so the tensor-core
    forward only runs the non-zero rows (+ one zero row per branch) when no per-slot output is requested.  A row's
    result does not depend on its place in a tile and the slot sums are formed in the same order, so the acceleration
    must be BIT-identical to the dense evaluation (which the messages request forces)."""
    from piml_b200 import models as M
    from .golden_args import base_args
    has_obs = ko > 0
    args = base_args(model="pinnsf_bottleneck", dataset_name="gc1560", obs_feature_dim=6 if has_obs else 0)
    torch.manual_seed(R)
    net = M.CLASSES["pinnsf_bottleneck"](args).cuda().eval()
    g = torch.Generator().manual_seed(R + 7)
    lead = (chan, R // chan) if chan else (R,)
    ped = torch.randn(*lead, kp, 6, generator=g)
    ped[torch.rand(*lead, kp, generator=g) < pz] = 0
    obs = torch.randn(*lead, max(ko, 1), 6, generator=g)[..., :ko, :]
    if ko:
        obs[torch.rand(*lead, ko, generator=g) < pz] = 0
    ped.view(-1, kp, 6)[:3] = 0                                # whole agents without neighbours
    slf = torch.randn(*lead, 7, generator=g)
    ped, obs, slf = ped.cuda(), obs.cuda(), slf.cuda()
    packed = M.pack_device(net.state_dict(), net.spec)
    ptc = M.pack_device_tc(net.state_dict(), net.spec)
    assert ptc is not None
    dense = M.pinnsf_forward(net.spec, packed, ped, obs, slf, need_msgs=True, packed_tc=ptc)
    compact = M.pinnsf_forward(net.spec, packed, ped, obs, slf, need_msgs=False, packed_tc=ptc)
    assert torch.equal(dense[0], compact[0])
    again = M.pinnsf_forward(net.spec, packed, ped, obs, slf, need_msgs=False, packed_tc=ptc)
    assert torch.equal(again[0], compact[0])                   # independent of the (atomic) row order
    ref = M.pinnsf_forward(net.spec, packed, ped, obs, slf, need_msgs=True)
    err = accel_err(npy(compact[0]).reshape(-1, 2), npy(ref[0]).reshape(-1, 2), npy(slf).reshape(-1, 7), net.spec.tau)
    assert err < TOL, err


@pytest.mark.parametrize("R,kp,ko,pz,chan", [(6000, 6, 10, 0.75, 0), (3100, 6, 0, 0.5, 0), (3300, 6, 0, 0.5, 0),
                                             (5000, 4, 7, 0.9, 5)])
def test_tensor_core_agent_compact_mode_is_bit_identical(R, kp, ko, pz, chan):
    """Summed-embedding networks (pinnsf_m, model.py:1274-1279): an agent whose slots are all zero (an absent agent, or
    one with no obstacle in range) yields the same per-branch output, so only the agents with a non-zero slot (+ one
    all-zero agent per branch) go through the network.  Bit-identical to the dense evaluation, which the library runs
    for the chunks of a batch whose dense tiles fit one wave.  Launch counts show each call's route: the agent-compact
    mode adds tc_compact_agents_kernel, and runs when the whole batch's dense tiles exceed one wave (3100 agents with
    6 slots and no obstacle branch are 148 tiles: dense on a 148-SM B200, compact with 3300)."""
    from piml_b200 import _lib as L, models as M
    from .golden_args import base_args
    from .util import dense_tile_count, tc_forward_in_dense_chunks
    has_obs = ko > 0
    args = base_args(model="pinnsf_m", dataset_name="gc1560", obs_feature_dim=6 if has_obs else 0)
    torch.manual_seed(R)
    net = M.CLASSES["pinnsf_m"](args).cuda().eval()
    g = torch.Generator().manual_seed(R + 3)
    lead = (chan, R // chan) if chan else (R,)
    ped = torch.randn(*lead, kp, 6, generator=g)
    ped[torch.rand(*lead, generator=g) < pz] = 0                   # whole agents without neighbours
    ped[..., -1, :] = 0                                            # and a padded slot on everybody
    obs = torch.randn(*lead, max(ko, 1), 6, generator=g)[..., :ko, :]
    if ko:
        obs[torch.rand(*lead, generator=g) < 0.95] = 0
    slf = torch.randn(*lead, 7, generator=g)
    ped, obs, slf = ped.cuda(), obs.cuda(), slf.cuda()
    packed = M.pack_device(net.state_dict(), net.spec)
    ptc = M.pack_device_tc(net.state_dict(), net.spec)
    assert ptc is not None
    sms = torch.cuda.get_device_properties(0).multi_processor_count
    l0 = L.launch_count()
    full = M.pinnsf_forward(net.spec, packed, ped, obs, slf, need_msgs=False, packed_tc=ptc)[0]
    launches = L.launch_count() - l0
    dense, chunk_launches = tc_forward_in_dense_chunks(net.spec, packed, ptc, ped, obs, slf, sms)
    compact = dense_tile_count(R, kp, ko) > sms
    assert set(chunk_launches) == {launches - compact}, (launches, chunk_launches, compact)
    assert torch.equal(full, dense)
    ref = M.pinnsf_forward(net.spec, packed, ped, obs, slf, need_msgs=True)
    err = accel_err(npy(full).reshape(-1, 2), npy(ref[0]).reshape(-1, 2), npy(slf).reshape(-1, 7), net.spec.tau)
    assert err < TOL, err


# ---- integrator ----------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("name", ["rollout_gc_bm", "rollout_toy5_m", "rollout_ucy_bm"])
def test_integrate_step_golden(name):
    """Re-synchronised steps over the whole reference rollout: p, v, dest bit-exact."""
    from piml_b200.rollout import integrate_step
    z = golden(name)
    i, o = group(z, "in"), group(z, "out")
    T, t0, dt = int(i["num_frames"]), int(i["t_start"]), float(i["time_unit"])
    flag = cu((i["mask_p"] - i["mask_p_pred"]), torch.int64)
    P_, V_, A_ = cu(o["position"]), cu(o["velocity"]), cu(o["acceleration"])
    gt = {k: cu(i[k]) for k in ("position", "velocity", "acceleration", "destination")}
    gt_idx = cu(i["dest_idx"], torch.int64)
    dest = cu(i["destination"][t0]).clone()
    didx = cu(i["dest_idx"][t0], torch.int64).clone()
    dnum = cu(i["dest_num"], torch.int64)
    wp = cu(i["waypoints"])
    for t in range(t0, T - 1):
        p, v, a = P_[t].clone(), V_[t].clone(), A_[t].clone()
        hist = torch.empty_like(v)
        integrate_step(p, v, a, A_[t + 1], dest, didx, dnum, wp, dt, True, flag[t + 1], gt["position"][t + 1],
                       gt["velocity"][t + 1], gt["acceleration"][t + 1], gt["destination"][t + 1], gt_idx[t + 1],
                       hist)
        assert torch.equal(torch.nan_to_num(p, nan=-7.0), torch.nan_to_num(P_[t + 1], nan=-7.0)), (name, t)
        assert torch.equal(v, V_[t + 1]), (name, t)
        assert np.array_equal(npy(dest), o["dest_after_step"][t - t0], equal_nan=True), (name, t)


# ---- whole rollout ---------------------------------------------------------------------------------------------------
def _rollout_inputs(name):
    from tests.golden_args import base_args
    from piml_b200 import models as M
    z = golden(name)
    i, o = group(z, "in"), group(z, "out")
    kind, dsn = str(i["model"]), str(i["dataset_name"])
    args = base_args(model=kind, dataset_name=dsn, time_unit=float(i["time_unit"]))
    m = M.CLASSES[kind](args)
    zm = golden("models")                       # the rollout fixtures use the seed-666 weights stored in models.npz
    sd = {k[3:]: torch.from_numpy(v) for k, v in group(zm, kind).items() if k.startswith("sd/")}
    m.load_state_dict(sd)
    m = m.cuda().eval()
    return z, i, o, args, m


@pytest.mark.parametrize("name", ["rollout_gc_bm", "rollout_toy5_m", "rollout_ucy_bm"])
def test_rollout_resynchronised_steps(name):
    """From the reference's own state at step t: rebuild features, run the network.  The new acceleration must be
    within 1e-5 of the reference's a[t+1] (per agent, relative to the operands' magnitude, tests/util.accel_err)."""
    from piml_b200.rollout import state_features
    from piml_b200 import models as M
    z, i, o, args, m = _rollout_inputs(name)
    T, t0 = int(i["num_frames"]), int(i["t_start"])
    P_, V_, A_ = cu(o["position"]), cu(o["velocity"]), cu(o["acceleration"])
    flag = i["mask_p"] - i["mask_p_pred"]
    ds = cu(i["desired_speed"])[None]
    obs = cu(i["obstacles"])
    spec = m.spec
    packed = M.pack_device(m.state_dict(), spec)
    worst = 0.0
    for t in range(t0 + 1, T - 1, max(1, (T - t0) // 60)):
        p, v, a = P_[t][None].clone(), V_[t][None].clone(), A_[t][None].clone()
        dest = cu(o["dest_after_step"][t - t0 - 1])[None]
        hist = v.clone()                                    # hist_v == v_cur after the update (h = 1)
        ped_f, obs_f, self_f = state_features(p, v, a, dest, obs, hist, ds, 6, 90, 4, 10, 90, 4)
        acc = M.pinnsf_forward(spec, packed, ped_f[0], obs_f[0], self_f[0], need_msgs=False)[0]
        sim = flag[t + 1] == 0                              # entering pedestrians are overwritten from the data
        worst = max(worst, accel_err(npy(acc)[sim], o["acceleration"][t + 1][sim], npy(self_f[0])[sim], spec.tau))
    assert worst < TOL, worst


@pytest.mark.parametrize("name", ["rollout_gc_bm", "rollout_toy5_m", "rollout_ucy_bm"])
def test_rollout_free_running(name):
    """Whole get_multiple_rollouts drop-in: NaN pattern and mask_p identical, drift reported (chaotic dynamics:
    the reference drifts 3e-4..6e-3 m from itself after 725 steps under a 1-ulp perturbation, SURVEY 8d)."""
    from piml_b200.rollout import rollout_scenes
    from piml_b200 import models as M
    z, i, o, args, m = _rollout_inputs(name)
    T, t0 = int(i["num_frames"]), int(i["t_start"])
    scene = {k: cu(i[k])[None] for k in ("position", "velocity", "acceleration", "destination", "waypoints",
                                          "mask_p", "mask_p_pred", "desired_speed")}
    scene["dest_idx"] = cu(i["dest_idx"], torch.int64)[None]
    scene["dest_num"] = cu(i["dest_num"], torch.int64)[None]
    scene["obstacles"] = cu(i["obstacles"])
    for k in ("ped_features0", "obs_features0", "self_features0"):
        scene[k] = cu(i[k])[None]
    packed = M.pack_device(m.state_dict(), m.spec)
    p_res, v_res, a_res, mask = rollout_scenes(m.spec, packed, args, scene, t0, T)
    p_res, mask = npy(p_res[0]), npy(mask[0])
    assert np.array_equal(mask, o["mask_p"])
    drift = np.linalg.norm(p_res - o["position"], axis=-1)
    same_nan = np.array_equal(np.isnan(p_res), np.isnan(o["position"]))
    print(f"{name}: max drift {np.nanmax(drift):.3e} m over {T - t0} steps; NaN pattern identical: {same_nan}")
    first = min(T, t0 + 26)
    assert np.array_equal(np.isnan(p_res[:first]), np.isnan(o["position"][:first]))
    assert np.nanmax(drift[:first]) < 1e-4
    assert np.nanmax(drift) < 0.5


# ---- pure social-force mode (BASELINE config 2) ------------------------------------------------------------------------
def test_sfm_forward_golden_and_oracle():
    """piml_b200.SocialForce against the composed reference module's own outputs and the oracle."""
    import piml_b200 as P
    g = group(golden("rollout_syn_sfm"), "fwd")
    net = P.SocialForce("gc1560")
    acc, pm, om = net(cu(g["ped"]), cu(g["obs"]), cu(g["self"]))
    assert rel_vec_err(npy(pm), g["ped_msgs"], floor=1e-4) < TOL
    assert rel_vec_err(npy(om), g["obs_msgs"], floor=1e-4) < TOL
    assert np.array_equal(npy(pm) == 0, g["ped_msgs"] == 0) and np.array_equal(npy(om) == 0, g["obs_msgs"] == 0)
    assert accel_err(npy(acc), g["acc"], g["self"], 0.5) < TOL
    want = O.sfm_forward(g["ped"], g["obs"], g["self"], "gc1560")
    assert accel_err(npy(acc), want[0], g["self"], 0.5) < TOL
    # host tensors in -> host tensors out, scene-batched leading dimension
    acc2 = net(torch.from_numpy(g["ped"])[None], torch.from_numpy(g["obs"])[None], torch.from_numpy(g["self"])[None])[0]
    assert not acc2.is_cuda and np.array_equal(acc2[0].numpy(), npy(acc))


def _sfm_scene(i):
    scene = {k: cu(i[k])[None] for k in ("position", "velocity", "acceleration", "destination", "waypoints",
                                          "mask_p", "mask_p_pred", "desired_speed")}
    scene["dest_idx"] = cu(i["dest_idx"], torch.int64)[None]
    scene["dest_num"] = cu(i["dest_num"], torch.int64)[None]
    scene["obstacles"] = cu(i["obstacles"])
    for k in ("ped_features0", "obs_features0", "self_features0"):
        scene[k] = cu(i[k])[None]
    return scene


def test_sfm_rollout_resynchronised_steps():
    """From the reference's recorded state at t (composed social-force module rolled out by the unmodified
    get_multiple_rollouts, synthetic GC clip, 725 steps): feature rebuild + SFM forward reproduce a[t+1] within 1e-5
    (the state update itself is covered bit for bit by test_integrate_resynchronised_steps on the other clips and by
    the oracle test of this clip)."""
    import piml_b200 as P
    from piml_b200.rollout import state_features
    z = golden("rollout_syn_sfm")
    i, o = group(z, "in"), group(z, "out")
    T, t0, dt = int(i["num_frames"]), int(i["t_start"]), float(i["time_unit"])
    net = P.SocialForce("gc1560")
    P_, V_, A_ = cu(o["position"]), cu(o["velocity"]), cu(o["acceleration"])
    flag = (i["mask_p"] - i["mask_p_pred"]).astype(np.int64)
    ds, obs = cu(i["desired_speed"])[None], cu(i["obstacles"])
    worst = 0.0
    for t in range(t0 + 1, T - 1, 7):
        p, v, a = P_[t][None].clone(), V_[t][None].clone(), A_[t][None].clone()
        dest = cu(o["dest_after_step"][t - t0 - 1])[None]
        ped_f, obs_f, self_f = state_features(p, v, a, dest, obs, v.clone(), ds, 6, 90, 4, 10, 90, 4)
        acc = net(ped_f[0], obs_f[0], self_f[0])[0]
        sim = flag[t + 1] == 0
        worst = max(worst, accel_err(npy(acc)[sim], o["acceleration"][t + 1][sim], npy(self_f[0])[sim], 0.5))
    assert worst < TOL, worst


def test_sfm_rollout_free_running():
    """BASELINE config 2: the whole 725-step pure social-force rollout in one C call against the reference's run of
    the composed module: arrival / entry pattern (mask_p, NaNs) identical, drift reported."""
    import piml_b200 as P
    from piml_b200.rollout import rollout_scenes
    from tests.golden_args import base_args
    z = golden("rollout_syn_sfm")
    i, o = group(z, "in"), group(z, "out")
    T, t0 = int(i["num_frames"]), int(i["t_start"])
    args = base_args(model="sfm", dataset_name="gc1560", time_unit=float(i["time_unit"]))
    net = P.SocialForce("gc1560")
    before = P._lib.launch_count()
    p_res, v_res, a_res, mask = rollout_scenes(net.spec, None, args, _sfm_scene(i), t0, T)
    assert P._lib.launch_count() - before >= 1
    p_res, v_res, mask = npy(p_res[0]), npy(v_res[0]), npy(mask[0])
    assert np.array_equal(mask, o["mask_p"])
    assert np.array_equal(np.isnan(p_res), np.isnan(o["position"]))
    drift = np.linalg.norm(p_res - o["position"], axis=-1)
    print(f"rollout_syn_sfm: max drift {np.nanmax(drift):.3e} m, mean {np.nanmean(drift):.3e} m over {T - t0} steps")
    assert np.nanmax(drift[:t0 + 26]) < 1e-4
    assert np.nanmax(drift) < 0.05


# ---- agent-sharded NN step: row-range features ---------------------------------------------------------------------
@pytest.mark.parametrize("N,M,rows", [(5000, 300, (1234, 3001)), (4099, 0, (0, 17)), (9000, 2000, (8000, 9000))])
def test_state_features_row_range_matches_full_call(N, M, rows):
    """piml_state_features_rows_f32 (what a rank of an agent-sharded crowd calls for its own rows) returns exactly the
    rows of the unsharded call, and applies the in-place NaN -> 0 of data.py:483-484 to ALL rows so that every rank's
    copy of the state stays the same."""
    from piml_b200 import _lib as L
    from piml_b200.features import cos_threshold
    from piml_b200.rollout import state_features
    rng = np.random.default_rng(N + M)
    side = np.sqrt(N / 0.5)
    p = (rng.random((1, N, 2)) * side).astype(np.float32)
    p[0, rng.random(N) < 0.05] = np.nan                               # absent agents
    v = rng.normal(0, 1, (1, N, 2)).astype(np.float32)
    v[0, rng.random(N) < 0.03] = np.nan
    a = rng.normal(0, 1, (1, N, 2)).astype(np.float32)
    a[0, rng.random(N) < 0.03] = np.nan
    d = (rng.random((1, N, 2)) * side).astype(np.float32)
    obs = (rng.random((M, 2)) * side).astype(np.float32)
    ds = np.full((1, N), 1.3, np.float32)
    L.check(L.load().piml_set_feature_algorithm(2), "piml_set_feature_algorithm")
    try:
        vf, af = cu(v), cu(a)
        pf, of, sf = state_features(cu(p), vf, af, cu(d), cu(obs), vf.clone(), cu(ds), 6, 90, 4, 10, 90, 4)
    finally:
        L.check(L.load().piml_set_feature_algorithm(0), "piml_set_feature_algorithm")
    r0, r1 = rows
    n = r1 - r0
    kp, ko = min(6, N), min(10, M)
    vr, ar = cu(v), cu(a)
    hist = vr.clone()
    ped_f, obs_f = torch.empty(n, kp, 6).cuda(), torch.empty(n, max(ko, 1), 6).cuda()
    self_f, dest_f = torch.empty(n, 7).cuda(), torch.empty(n, 2).cuda()
    pos, dst, ob, dsp = cu(p), cu(d), cu(obs), cu(ds)
    L.check(L.load().piml_state_features_rows_f32(
        L.ptr(pos), L.ptr(vr), L.ptr(ar), L.ptr(dst), L.ptr(ob) if M else None, N, M, r0, r1, 6, cos_threshold(90), 4.0,
        10, cos_threshold(90), 4.0, L.ptr(hist), L.ptr(dsp), L.ptr(ped_f), L.ptr(obs_f) if M else None, L.ptr(self_f),
        L.ptr(dest_f), L.stream_ptr(pos.device)), "piml_state_features_rows_f32")
    assert torch.equal(ped_f, pf[0, r0:r1])
    if M:
        assert torch.equal(obs_f[:, :ko], of[0, r0:r1])
    # self_f holds hist_v, which was captured before the NaN -> 0 (NaN == NaN is False): compare bitwise
    assert torch.equal(self_f.view(torch.int32), sf[0, r0:r1].contiguous().view(torch.int32))
    assert torch.equal(vr.view(torch.int32), vf.view(torch.int32)) and torch.equal(ar.view(torch.int32), af.view(torch.int32))
    assert not torch.isnan(vr).any() and not torch.isnan(ar).any()


@pytest.mark.parametrize("S", [1, 5])
def test_sfm_persistent_rollout_kernel_matches_per_step_path(S):
    """The persistent one-launch rollout kernel (rollout_sfm.cu) against the three-launches-per-step route of
    piml_rollout_f32: every recorded p, v, a and mask bit for bit, for S scenes (the golden clip and jittered copies)."""
    import os
    import piml_b200 as P
    from piml_b200.rollout import rollout_scenes
    from tests.golden_args import base_args
    z = golden("rollout_syn_sfm")
    i, o = group(z, "in"), group(z, "out")
    T, t0 = int(i["num_frames"]), int(i["t_start"])
    T = min(T, t0 + 260)
    args = base_args(model="sfm", dataset_name="gc1560", time_unit=float(i["time_unit"]))
    scene = _sfm_scene(i)
    if S > 1:
        g = torch.Generator().manual_seed(S)
        rep = {}
        for k, v in scene.items():
            if k == "obstacles":
                rep[k] = v
                continue
            v = v.expand(S, *v.shape[1:]).clone()
            if k == "position":
                v = v + 0.05 * torch.randn(v.shape, generator=g).to(v.device)          # NaNs stay NaN
            rep[k] = v
        scene = rep
        from piml_b200.rollout import state_features
        fargs = (args.topk_ped, args.sight_angle_ped, args.dist_threshold_ped, args.topk_obs, args.sight_angle_obs,
                 args.dist_threshold_obs)
        v0 = scene["velocity"][:, t0].contiguous()
        pf, of, sf = state_features(scene["position"][:, t0].contiguous(), v0, scene["acceleration"][:, t0].contiguous(),
                                    scene["destination"][:, t0].contiguous(), scene["obstacles"], v0.clone(),
                                    scene["desired_speed"], *fargs)
        scene["ped_features0"], scene["obs_features0"], scene["self_features0"] = pf, of, sf
    spec = P.SocialForce("gc1560").spec
    outs = {}
    for mode in ("1", "0"):
        os.environ["PIML_SFM_PERSISTENT"] = mode
        try:
            before = P._lib.launch_count()
            outs[mode] = [npy(x) for x in rollout_scenes(spec, None, args, scene, t0, T)]
            launches = P._lib.launch_count() - before
        finally:
            os.environ.pop("PIML_SFM_PERSISTENT", None)
        assert (launches == 1) if mode == "1" else (launches >= 3 * (T - t0))
    for a_, b_ in zip(outs["1"], outs["0"]):
        assert np.array_equal(a_, b_, equal_nan=True)
    if S == 1:
        assert np.array_equal(outs["1"][3][0], o["mask_p"][:T])


def test_predicate_arithmetic_against_torch_primitives_gpu():
    """SURVEY.md A.2b row 1 on the CUDA path: the k smallest gated distances of get_nearby_obj_in_sight on random pairs
    incl. zero / huge / tiny / inf / NaN coordinates equal torch's CPU norm + cosine_similarity bit for bit."""
    import piml_b200 as P
    rng = np.random.default_rng(11)
    N, M, k = 256, 4096, 32
    pos = rng.normal(0, 3, (1, N, 2)).astype(np.float32)
    obj = rng.normal(0, 3, (1, M, 2)).astype(np.float32)
    obj[0, :64] = pos[0, :64]
    obj[0, 64:96] *= 1e18
    obj[0, 96:128] *= 1e-30
    obj[0, 128:140] = np.nan
    obj[0, 140:150, 0] = np.inf
    pos[0, -3:] = np.nan
    head = rng.normal(0, 1, (1, N, 2)).astype(np.float32)
    head[0, :16] = 0.0
    for angle in (90, 100):
        dist, idx = P.Pedestrians().get_nearby_obj_in_sight(cu(pos), cu(obj), cu(head), k, angle)
        p, o, h = torch.from_numpy(pos), torch.from_numpy(obj), torch.from_numpy(head)
        rel = o[:, None, :, :] - p[:, :, None, :]
        rel[torch.isnan(rel)] = float('inf')
        d = torch.norm(rel, p=2, dim=-1)
        cos = torch.cosine_similarity(rel, h[:, :, None, :].expand_as(rel), dim=-1)
        cos[torch.isnan(cos)] = -1
        d[cos < torch.tensor(np.float32(np.cos(3.14 * angle / 180)))] = float('inf')
        want = torch.sort(d, dim=-1)[0][..., :k].numpy()
        assert np.array_equal(npy(dist).view(np.uint32), want.view(np.uint32)), angle


@pytest.mark.parametrize("model", ["sfm", "pinnsf_bm"])
def test_scene_sharded_rollouts_equal_the_unsharded_batch(model):
    """SURVEY.md A.2b multi-GPU row, scene parallelism: rolling S scenes together and rolling two halves of them
    separately (what two ranks do, no communication) give bit-identical trajectories."""
    import os
    import piml_b200 as P
    from piml_b200 import models as M
    from piml_b200.rollout import rollout_scenes, state_features
    from tests.golden_args import base_args
    z = golden("rollout_syn_sfm")
    i = group(z, "in")
    T, t0, S = 60 + int(i["t_start"]), int(i["t_start"]), 6
    args = base_args(model="pinnsf_bm", dataset_name="gc1560", time_unit=float(i["time_unit"]))
    scene = _sfm_scene(i)
    g = torch.Generator().manual_seed(9)
    rep = {}
    for k_, v in scene.items():
        if k_ == "obstacles":
            rep[k_] = v
            continue
        v = v.expand(S, *v.shape[1:]).clone()
        if k_ == "position":
            v = v + 0.05 * torch.randn(v.shape, generator=g).to(v.device)
        rep[k_] = v
    scene = rep
    v0 = scene["velocity"][:, t0].contiguous()
    pf, of, sf = state_features(scene["position"][:, t0].contiguous(), v0, scene["acceleration"][:, t0].contiguous(),
                                scene["destination"][:, t0].contiguous(), scene["obstacles"], v0.clone(),
                                scene["desired_speed"], 6, 90, 4, 10, 90, 4)
    scene["ped_features0"], scene["obs_features0"], scene["self_features0"] = pf, of, sf
    if model == "sfm":
        spec, packed, ptc = P.SocialForce("gc1560").spec, None, None
    else:
        torch.manual_seed(666)
        net = M.CLASSES["pinnsf_bm"](args).cuda().eval()
        spec, packed, ptc = net.spec, M.pack_device(net.state_dict(), net.spec), M.pack_device_tc(net.state_dict(), net.spec)
    full = [npy(x) for x in rollout_scenes(spec, packed, args, scene, t0, T, packed_tc=ptc)]
    for lo, hi in ((0, 3), (3, 6)):
        part_scene = {k_: (v if k_ == "obstacles" else v[lo:hi].contiguous()) for k_, v in scene.items()}
        part = [npy(x) for x in rollout_scenes(spec, packed, args, part_scene, t0, T, packed_tc=ptc)]
        for a_, b_ in zip(full, part):
            assert np.array_equal(a_[lo:hi], b_, equal_nan=True)


# ---- f-4: evaluation metrics -------------------------------------------------------------------------------------------
@pytest.mark.parametrize("name", ["rollout_gc_bm", "rollout_ucy_bm", "rollout_syn_sfm"])
def test_metrics_match_reference_gpu(name):
    """piml_b200.metrics (one launch for all frames) against the reference's own METRIC values on its own rollouts:
    every frame's Sinkhorn OT cost and MMD, the MAE sum and the collision counts."""
    from piml_b200 import metrics as MT
    g = group(golden("metrics"), name)
    p, q, mask = cu(g["p_pred"]), cu(g["labels"]), cu(g["mask"], torch.int64)
    mae = MT.mae_with_time_mask(p, q, mask, reduction='sum')
    assert abs(mae - float(g["mae_sum"])) <= 1e-5 * float(g["mae_sum"])
    ot = np.asarray(MT.ot_with_time_mask(p, q, mask, reduction=None))
    assert ot.shape == g["ot"].shape
    assert np.allclose(ot, g["ot"], rtol=2e-4, atol=1e-6), float(np.abs(ot - g["ot"]).max())
    assert abs(MT.ot_with_time_mask(p, q, mask, reduction='sum') - float(g["ot_sum"])) <= 1e-4 * float(g["ot_sum"])
    mmd = np.asarray(MT.mmd_with_time_mask(p, q, mask, reduction=None))
    assert np.allclose(mmd, g["mmd"], rtol=2e-4, atol=2e-6), float(np.abs(mmd - g["mmd"]).max())
    assert abs(MT.mmd_with_time_mask(p, q, mask, reduction='sum') - float(g["mmd_sum"])) <= 1e-4 * float(g["mmd_sum"]) + 1e-5
    t0 = int(g["t_start"])
    raw = cu(g["p_raw"])
    assert MT.collision_count(raw[t0:], 0.5, reduction='sum') == float(g["collision_count"])
    assert MT.collision_count(raw[t0:], 0.25, reduction='sum') == float(g["hard_collision_count"])
    # host tensors in: staged like every other adapter
    assert abs(MT.mae_with_time_mask(torch.from_numpy(g["p_pred"]), torch.from_numpy(g["labels"]),
                                     torch.from_numpy(g["mask"]), reduction='sum') - mae) < 1e-3


def test_metrics_against_oracle_on_random_frames():
    """Random point sets incl. frames with 0 / 1 / many masked agents, against the numpy restatement."""
    from piml_b200 import metrics as MT
    rng = np.random.default_rng(5)
    T, N = 40, 200
    p = rng.normal(0, 4, (T, N, 2)).astype(np.float32)
    q = (p + rng.normal(0, 0.7, (T, N, 2))).astype(np.float32)
    mask = (rng.random((T, N)) < rng.random((T, 1))).astype(np.int64)
    mask[0] = 0
    mask[1] = 0
    mask[1, 7] = 1
    mask[2] = 1
    fr, want_ot = O.ot_with_time_mask(p, q, mask)
    _, want_mmd = O.mmd_with_time_mask(p, q, mask)
    ot = np.asarray(MT.ot_with_time_mask(cu(p), cu(q), cu(mask, torch.int64), reduction=None))
    mmd = np.asarray(MT.mmd_with_time_mask(cu(p), cu(q), cu(mask, torch.int64), reduction=None))
    assert len(ot) == len(fr) == len(mmd)
    assert np.allclose(ot, want_ot, rtol=2e-4, atol=1e-6), float(np.abs(ot - want_ot).max())
    assert np.allclose(mmd, want_mmd, rtol=2e-4, atol=2e-6), float(np.abs(mmd - want_mmd).max())
    want_mae = O.mae_with_time_mask(p, q, mask)
    assert abs(MT.mae_with_time_mask(cu(p), cu(q), cu(mask, torch.int64), reduction='sum') - want_mae) <= 1e-5 * want_mae


# ---- edge sizes ----------------------------------------------------------------------------------------------------------
def test_edge_sizes_do_not_break_the_adapters():
    """Empty and minimal inputs through every adapter (the reference's own tensors can be this small: toy clips have
    N = 3, M = 2; a frame can have 0 or 1 agents)."""
    import piml_b200 as P
    from piml_b200 import metrics as MT
    ped = P.Pedestrians()
    # one agent, two obstacle points: k' = min(k, N|M)
    p1, v1 = cu([[[1.0, 2.0]]]), cu([[[0.5, 0.0]]])
    a1, d1, ob = cu([[[0.0, 0.0]]]), cu([[[3.0, 2.0]]]), cu([[2.0, 2.0], [9.0, 9.0]])
    pf, of, df = ped.get_relative_features(p1, v1, a1, d1, ob, 6, 90, 4, 10, 90, 4)
    assert pf.shape == (1, 1, 1, 6) and of.shape == (1, 1, 2, 6) and df.shape == (1, 1, 2)
    want = O.relative_features(npy(p1), npy(v1).copy(), npy(a1).copy(), npy(d1), npy(ob))
    for w, g_ in zip(want, (pf, of, df)):
        assert np.array_equal(npy(g_), w)
    # MLAPM with 1 and 2 agents (no pair / one pair), both kernels' entry point
    for N in (1, 2):
        p = cu(np.array([[0.0, 0.0], [1.0, 0.5]][:N], np.float32))
        v = cu(np.array([[1.0, 0.0], [-1.0, 0.0]][:N], np.float32))
        ds, d = cu(np.full((N, 1), 1.3, np.float32)), cu(np.array([[5.0, 0.0], [-5.0, 0.5]][:N], np.float32))
        act = P.MLAPM(**GC_KW).step(p, v, ds, d, 0.08)
        ref = O.mlapm_step(npy(p), npy(v), npy(ds), npy(d), 0.08, "GC")
        assert rel_vec_err(npy(act), ref) < TOL
    # empty batches
    e = torch.empty(0, 2).cuda()
    assert P.MLAPM(**GC_KW).step(e, e, torch.empty(0, 1).cuda(), e, 0.08).shape == (0, 2)
    net = P.SocialForce("gc1560")
    out = net(torch.empty(0, 6, 6).cuda(), torch.empty(0, 10, 6).cuda(), torch.empty(0, 7).cuda())
    assert out[0].shape == (0, 2) and out[1].shape == (0, 6, 2)
    assert P.calc_acceleration(torch.empty(0, 6, 6).cuda()).shape == (0, 6, 2)
    z = torch.zeros(3, 4, 2).cuda()
    m0 = torch.zeros(3, 4, dtype=torch.int64).cuda()
    assert MT.ot_with_time_mask(z, z, m0, reduction=None) == [] and MT.mae_with_time_mask(z, z, m0, reduction='sum') == 0.0


def test_mlapm_symmetric_vs_ordered_at_bench_size():
    """BASELINE config 4 size (N = 100 000, T = 196 blocks): the symmetric kernel the bench times against the ordered-pair
    kernel, two consecutive steps on one workspace.  Both kernels get the SAME inputs at each step (the second step starts
    from the symmetric kernel's state: a free-running comparison would measure how fp32 rounding of step 1 flips
    borderline gates in step 2, not the kernels).  The oracle check at this size is tests/test_gpu_parity_sizes.py."""
    import sys
    import os
    sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
    import bench
    import piml_b200 as P
    N = 100000
    p, v, ds, dest, _ = [x.cuda() for x in bench.synthetic_crowd(N)]
    model = P.MLAPM(**bench.MLAPM_KW)
    pp, vv = p.clone(), v.clone()
    for step in range(2):
        res = {}
        for algo in (2, 1):
            _mlapm_algorithm(algo)
            try:
                act, pn, arr = model.advance(pp, vv, ds, dest, bench.DT, bench.RADIUS)
                res[algo] = (act, pn, arr)
            finally:
                _mlapm_algorithm(0)
        vs, vo = npy(res[2][0]), npy(res[1][0])
        assert np.isfinite(vs).all()
        num = np.linalg.norm(vs.astype(np.float64) - vo, axis=-1)
        den = np.maximum(np.maximum(np.linalg.norm(vo, axis=-1), np.linalg.norm(npy(vv), axis=-1)), 1e-6)
        assert float((num / den).max()) < TOL, (step, float((num / den).max()))
        assert np.abs(npy(res[2][1]) - npy(res[1][1])).max() < 1e-4        # positions up to 450 m: a few fp32 ulps
        assert (npy(res[2][2]) != npy(res[1][2])).sum() <= 2                # arrival test at the radius boundary
        pp, vv = res[2][1], res[2][0]


# ---- round 2: small kernels that replaced the last eager-torch helpers ---------------------------------------------------
@pytest.mark.parametrize("name", ["rollout_gc_bm", "rollout_ucy_bm", "rollout_toy5_m"])
def test_desired_speed_kernel_matches_reference_and_oracle(name):
    """piml_desired_speed_f32 (data.py:797-806) on the clips' velocities: the reference's own make_dataset values."""
    from piml_b200.dataset import desired_speed
    g = golden(name)
    got = npy(desired_speed(cu(g["in/velocity"]), 25))
    assert np.allclose(got, g["in/desired_speed"], rtol=1e-6, atol=0, equal_nan=True)
    assert np.allclose(got, O.desired_speed(g["in/velocity"], 25), rtol=1e-6, atol=0, equal_nan=True)
    v = g["in/velocity"].copy()
    still = min(3, v.shape[1] - 1)
    v[:, still] = 0                                        # a pedestrian that never moves: frames [0, skip)
    assert npy(desired_speed(cu(v), 25))[still] == 0.0
    assert npy(desired_speed(cu(v[:5]), 25)).shape == (v.shape[1],)      # clip shorter than skip_frames


def test_relative_quantity_and_filtered_features_helpers():
    """get_relative_quantity (data.py:398-414) and get_filtered_features (:449-464) as dense kernels for the callers
    outside the hot path: bit-exact against the reference's tensor expressions."""
    import piml_b200 as P
    rng = np.random.default_rng(11)
    A = rng.normal(0, 3, (2, 3, 17, 6)).astype(np.float32)
    B = rng.normal(0, 3, (2, 3, 9, 6)).astype(np.float32)
    A[0, 1, 4] = np.nan
    ped = P.Pedestrians()
    rel = npy(ped.get_relative_quantity(cu(A), cu(B)))
    want = B[:, :, None, :, :] - A[:, :, :, None, :]
    assert rel.shape == (2, 3, 17, 9, 6) and np.array_equal(rel, want, equal_nan=True)
    k = 4
    idx = rng.integers(0, 9, (2, 3, 17, k)).astype(np.int64)
    dist = rng.random((2, 3, 17, k)).astype(np.float32) * 8
    dist[0, 0, 0, 0], dist[0, 0, 0, 1] = np.inf, np.nan
    got = npy(ped.get_filtered_features(cu(want), cu(idx, torch.int64), cu(dist), 4))
    ref = np.take_along_axis(want, idx[..., None].repeat(6, -1), axis=-2)
    ref[dist > 4] = 0                                       # NaN > 4 is False: the slot is kept, as in the reference
    assert np.array_equal(got, ref, equal_nan=True)


def test_metrics_reject_frames_beyond_the_shared_memory_limit():
    """ADVICE r1: more than 1024 masked agents in a frame used to give NaN OT / MMD and a truncated MAE silently."""
    from piml_b200 import metrics as MT
    rng = np.random.default_rng(5)
    T, N = 2, 1500
    p = rng.normal(0, 5, (T, N, 2)).astype(np.float32)
    q = (p + rng.normal(0, 0.3, (T, N, 2))).astype(np.float32)
    mask = np.ones((T, N), np.int64)
    mask[1, 1000:] = 0
    want = O.mae_with_time_mask(p, q, mask)
    got = MT.mae_with_time_mask(cu(p), cu(q), cu(mask, torch.int64), reduction='sum')
    assert abs(got - want) <= 2e-5 * want                  # every masked agent counted, no 1024 cut-off
    with pytest.raises(NotImplementedError):
        MT.ot_with_time_mask(cu(p), cu(q), cu(mask, torch.int64), reduction='sum')
    with pytest.raises(NotImplementedError):
        MT.mmd_with_time_mask(cu(p), cu(q), cu(mask, torch.int64), reduction='sum')
    mask[0, 1024:] = 0                                      # exactly at the limit: supported
    assert np.isfinite(MT.mmd_with_time_mask(cu(p), cu(q), cu(mask, torch.int64), reduction='sum'))
