"""piml_b200.sfm.sweep (piml_sfm_sweep_f32): one clip rolled out by the pure social-force model under many constant
sets in one call, scored on the device.  Each set against rollout_scenes on the clip alone with its constants, on both
routes; the golden clip inside a sweep; the score against a float64 recomputation and across batch shapes; a sweep of
65 536 sets in O(S N) memory; and the edges."""
import os

import numpy as np
import pytest
import torch

from tests.util import golden, group

pytestmark = pytest.mark.gpu

DEFAULT = [8.75, -2.5, 50.0, -5.0, 0.5]          # SocialForce('gc1560'): A_ped, B_ped, A_obs, B_obs, tau
SETS = [[10.67, -3.33, 50.0, -5.0, 0.5], [0.0, -2.5, 50.0, -5.0, 0.5], DEFAULT, [8.75, -2.5, 0.0, -5.0, 0.5],
        [5.0, -1.5, 30.0, -3.0, 0.3], [12.0, -3.0, 80.0, -6.0, 0.8], [8.75, -2.5, 50.0, -5.0, 1.5],
        [2.0, -0.5, 10.0, -1.0, 0.4]]


def cu(x, dtype=torch.float32):
    return torch.as_tensor(np.asarray(x), dtype=dtype).cuda()


def npy(t):
    return t.detach().cpu().numpy()


def clip():
    """The synthetic config-2 clip (N = 110, T = 750, t_start = 25) as the single-scene dict rollout_scenes takes."""
    from tests.golden_args import base_args
    z = golden("rollout_syn_sfm")
    i, o = group(z, "in"), group(z, "out")
    scene = {k: cu(i[k])[None] for k in ("position", "velocity", "acceleration", "destination", "waypoints",
                                          "mask_p", "mask_p_pred", "desired_speed")}
    scene["dest_idx"] = cu(i["dest_idx"], torch.int64)[None]
    scene["dest_num"] = cu(i["dest_num"], torch.int64)[None]
    scene["obstacles"] = cu(i["obstacles"])
    for k in ("ped_features0", "obs_features0", "self_features0"):
        scene[k] = cu(i[k])[None]
    args = base_args(model="sfm", dataset_name="gc1560", time_unit=float(i["time_unit"]))
    return scene, args, int(i["t_start"]), int(i["num_frames"]), i, o


def with_features_at(scene, args, t):
    """The scene with ped / obs / self features of the clip's state at frame t (what a caller starting there passes)."""
    from piml_b200.rollout import state_features
    s = dict(scene)
    v = s["velocity"][:, t].contiguous()
    pf, of, sf = state_features(s["position"][:, t].contiguous(), v, s["acceleration"][:, t].contiguous(),
                                s["destination"][:, t].contiguous(), s["obstacles"], v.clone(), s["desired_speed"],
                                args.topk_ped, args.sight_angle_ped, args.dist_threshold_ped, args.topk_obs,
                                args.sight_angle_obs, args.dist_threshold_obs)
    s["ped_features0"], s["obs_features0"], s["self_features0"] = pf, of, sf
    return s


def alone(scene, args, t0, T, row):
    """rollout_scenes on the clip alone with one set's constants."""
    from piml_b200.rollout import rollout_scenes
    from piml_b200.sfm import EPS, SfmSpec
    A_ped, B_ped, A_obs, B_obs, tau = row
    spec = SfmSpec(A_ped, B_ped, A_obs, B_obs, EPS, tau, has_obs=scene["obstacles"].numel() > 0)
    return [npy(x[0]) for x in rollout_scenes(spec, None, args, scene, t0, T)]


class route(object):
    """PIML_SFM_PERSISTENT for the duration of a block: '2' forces the persistent kernel, '0' the per-step launches."""

    def __init__(self, mode):
        self.mode = mode

    def __enter__(self):
        os.environ["PIML_SFM_PERSISTENT"] = self.mode

    def __exit__(self, *exc):
        os.environ.pop("PIML_SFM_PERSISTENT", None)


def score64(p_rec, mask_rec, position, mask_p, t0):
    """The score recomputed in float64 from recorded trajectories: per slot in time order, then slots in order."""
    S, T, N = mask_rec.shape
    d = p_rec[:, t0:].astype(np.float64) - position[None, t0:T].astype(np.float64)
    term = np.sqrt(d[..., 0] * d[..., 0] + d[..., 1] * d[..., 1])
    use = (mask_rec[:, t0:] == 1) & (mask_p[None, t0:T] == 1)
    term = np.where(use, term, 0.0)
    return term.sum(axis=1).sum(axis=1), use.sum(axis=(1, 2))


_RUNS = {}


def recorded(mode):
    """sweep(SETS, record=True) on the full clip on one route (computed once per route)."""
    if mode not in _RUNS:
        import piml_b200 as P
        from piml_b200 import sfm
        scene, args, t0, T, _, _ = clip()
        with route(mode):
            before = P._lib.launch_count()
            e, c, rec = sfm.sweep(scene, torch.tensor(SETS), args, t0, T, record=True)
            launches = P._lib.launch_count() - before
        _RUNS[mode] = (npy(e), npy(c), [npy(x) for x in rec], launches)
    return _RUNS[mode]


@pytest.mark.parametrize("mode", ["2", "0"])
def test_each_set_equals_its_own_rollout(mode):
    """Set s of a sweep records exactly what rollout_scenes records for the clip alone with SfmSpec(set s): p, v, a and
    mask bit for bit, on the persistent kernel (one launch + the score) and on the per-step route."""
    scene, args, t0, T, _, _ = clip()
    e, c, rec, launches = recorded(mode)
    assert (launches == 2) if mode == "2" else (launches >= 3 * (T - t0))
    with route(mode):
        for s, row in enumerate(SETS):
            want = alone(scene, args, t0, T, row)
            for got, ref in zip(rec, want):
                assert np.array_equal(got[s], ref, equal_nan=True), (s, row)


def test_golden_clip_inside_a_sweep():
    """The default constants placed among other sets meet the gates of the free-running golden rollout."""
    from piml_b200 import sfm
    scene, args, t0, T, _, o = clip()
    rows = [SETS[0], SETS[4], SETS[5], DEFAULT, SETS[7], SETS[1]]
    e, c, (p_res, v_res, a_res, mask) = sfm.sweep(scene, torch.tensor(rows), args, t0, T, record=True)
    p_res, mask = npy(p_res[3]), npy(mask[3])
    assert np.array_equal(mask, o["mask_p"])
    assert np.array_equal(np.isnan(p_res), np.isnan(o["position"]))
    drift = np.linalg.norm(p_res - o["position"], axis=-1)
    assert np.nanmax(drift[:t0 + 26]) < 1e-4
    assert np.nanmax(drift) < 0.05


def test_score_matches_float64_recomputation_on_both_routes():
    """err_sum within 1e-6 relative of a float64 sum over the recorded trajectories, err_count exact, and both routes
    return bit-identical scores."""
    _, _, t0, T, i, _ = clip()
    for mode in ("2", "0"):
        e, c, rec, _ = recorded(mode)
        want_e, want_c = score64(rec[0], rec[3], i["position"], i["mask_p"], t0)
        assert np.array_equal(c, want_c), mode
        assert np.all(np.abs(e - want_e) <= 1e-6 * np.abs(want_e)), (mode, e, want_e)
        assert np.all(c > 0)
    assert np.array_equal(recorded("2")[0], recorded("0")[0]) and np.array_equal(recorded("2")[1], recorded("0")[1])


def test_score_does_not_depend_on_the_batch():
    """A set's score alone, at another position, inside S = 4096 and on a repeated call: the same bits."""
    from piml_b200 import sfm
    scene, args, t0, T, _, _ = clip()
    T = min(T, t0 + 200)
    row = torch.tensor([SETS[4]])
    e1, c1 = sfm.sweep(scene, row, args, t0, T)
    g = torch.Generator().manual_seed(3)
    others = torch.tensor(DEFAULT) * (1 + 0.3 * (torch.rand(4095, 5, generator=g) - 0.5))
    for S, at in ((5, 3), (4096, 1234)):
        prm = torch.cat([others[:at], row, others[at:S - 1]])
        e, c = sfm.sweep(scene, prm, args, t0, T)
        assert e.shape == (S,) and e.dtype == torch.float64 and c.dtype == torch.int64
        assert torch.equal(e[at:at + 1], e1) and torch.equal(c[at:at + 1], c1), S
        if S == 4096:
            e_again, c_again = sfm.sweep(scene, prm, args, t0, T)
            assert torch.equal(e_again, e) and torch.equal(c_again, c)
            e_head, _ = sfm.sweep(scene, prm[:5], args, t0, T)
            assert torch.equal(e_head, e[:5])


def test_sweep_of_65536_sets_fits_in_memory_linear_in_sets_and_slots():
    """S = 65 536 score-only completes on the full clip; peak device memory stays below a bound linear in S N (the
    recorded trajectories alone would take 28 B x S T N = 150 GB); the sets at the ends score as they do alone."""
    from piml_b200 import sfm
    scene, args, t0, T, _, _ = clip()
    N = scene["position"].shape[2]
    S = 65536
    g = torch.Generator().manual_seed(5)
    prm = torch.tensor(DEFAULT) * (1 + 0.4 * (torch.rand(S, 5, generator=g) - 0.5))
    prm[0], prm[-1] = torch.tensor(DEFAULT), torch.tensor(SETS[5])
    torch.cuda.synchronize()
    base = torch.cuda.memory_allocated()
    torch.cuda.reset_peak_memory_stats()
    e, c = sfm.sweep(scene, prm, args, t0, T)
    torch.cuda.synchronize()
    peak = torch.cuda.max_memory_allocated() - base
    assert peak < 1024 * S * N + (64 << 20), peak
    assert torch.isfinite(e).all() and (c > 0).all()
    for k in (0, S - 1):
        e1, c1 = sfm.sweep(scene, prm[k:k + 1], args, t0, T)
        assert torch.equal(e[k:k + 1], e1) and torch.equal(c[k:k + 1], c1)


def test_no_sets():
    from piml_b200 import sfm
    scene, args, t0, T, _, _ = clip()
    e, c = sfm.sweep(scene, torch.zeros(0, 5), args, t0, T)
    assert e.shape == (0,) and c.shape == (0,)
    e, c, rec = sfm.sweep(scene, torch.zeros(0, 5), args, t0, T, record=True)
    assert rec[0].shape == (0, T, scene["position"].shape[2], 2)


@pytest.mark.parametrize("mode", ["2", "0"])
@pytest.mark.parametrize("case", ["last_frame", "no_obstacles"])
def test_edges_equal_their_own_rollouts(mode, case):
    """t_start = T - 1 (one step) and a clip without obstacles (M = 0), on both routes, against rollout_scenes."""
    from piml_b200 import sfm
    scene, args, t0, T, i, _ = clip()
    if case == "last_frame":
        t0 = T - 1
    else:
        T = min(T, t0 + 150)
        scene = dict(scene, obstacles=torch.zeros(0, 2, device="cuda"))
    scene = with_features_at(scene, args, t0)
    rows = [DEFAULT, SETS[1], SETS[6]]
    with route(mode):
        e, c, rec = sfm.sweep(scene, torch.tensor(rows), args, t0, T, record=True)
        for s, row in enumerate(rows):
            for got, ref in zip(rec, alone(scene, args, t0, T, row)):
                assert np.array_equal(npy(got[s]), ref, equal_nan=True), (case, s)
    want_e, want_c = score64(npy(rec[0]), npy(rec[3]), i["position"], i["mask_p"], t0)
    assert np.array_equal(npy(c), want_c)
    assert np.all(np.abs(npy(e) - want_e) <= 1e-6 * np.abs(want_e))
    if case == "last_frame":                     # the state at t_start is the clip's: nothing to miss yet
        assert np.all(npy(e) == 0.0) and np.all(npy(c) == int(i["mask_p"][t0].sum()))
