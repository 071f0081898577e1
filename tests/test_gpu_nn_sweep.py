"""piml_b200.rollout.sweep_networks (piml_nn_sweep_f32) and the tensor-core forward with one network per set
(piml_pinnsf_forward_tc_sets_f32): the per-set forward against the single-network forward bit for bit; every set of a
sweep against rollout_scenes on the clip alone with its network, on the GC and UCY clips and at the edges; the golden
network inside a sweep; the score against a float64 recomputation and across batch shapes; 512 networks in O(S N)
memory; and no networks at all."""
import numpy as np
import pytest
import torch

from tests.util import golden, group

pytestmark = pytest.mark.gpu


def cu(x, dtype=torch.float32):
    return torch.as_tensor(np.asarray(x), dtype=dtype).cuda()


def npy(t):
    return t.detach().cpu().numpy()


def seeded(kind, width, seed, dataset_name="gc1560", has_obs=True):
    """A seeded mirror network with encoder, processor and decoder widths `width` (two processor blocks)."""
    from piml_b200 import models as M
    from tests.golden_args import model_args
    torch.manual_seed(seed)
    return M.CLASSES[kind](model_args(kind, (width, width, width, 2, 2, 2, 1 if has_obs else 0), dataset_name)).eval()


def golden_net(name):
    """The network the golden rollout `name` was produced with, built as the rollout parity tests build it."""
    from piml_b200 import models as M
    from tests.golden_args import base_args
    i = group(golden(name), "in")
    kind, dsn = str(i["model"]), str(i["dataset_name"])
    m = M.CLASSES[kind](base_args(model=kind, dataset_name=dsn, time_unit=float(i["time_unit"])))
    sd = {k[3:]: torch.from_numpy(v) for k, v in group(golden("models"), kind).items() if k.startswith("sd/")}
    m.load_state_dict(sd)
    return m.eval()


def clip(name):
    """A golden rollout clip as the single-scene dict rollout_scenes takes, its args, t_start and T."""
    from tests.golden_args import base_args
    z = golden(name)
    i, o = group(z, "in"), group(z, "out")
    scene = {k: cu(i[k])[None] for k in ("position", "velocity", "acceleration", "destination", "waypoints",
                                          "mask_p", "mask_p_pred", "desired_speed")}
    scene["dest_idx"] = cu(i["dest_idx"], torch.int64)[None]
    scene["dest_num"] = cu(i["dest_num"], torch.int64)[None]
    scene["obstacles"] = cu(i["obstacles"])
    for k in ("ped_features0", "obs_features0", "self_features0"):
        scene[k] = cu(i[k])[None]
    args = base_args(model=str(i["model"]), dataset_name=str(i["dataset_name"]), time_unit=float(i["time_unit"]))
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


def alone(scene, args, t0, T, net):
    """rollout_scenes on the clip alone with one network's tensor-core vector."""
    from piml_b200 import models as M
    from piml_b200.rollout import rollout_scenes
    spec = M.spec_from_module(net)
    ptc = M.pack_device_tc(net.state_dict(), spec)
    return [npy(x[0]) for x in rollout_scenes(spec, None, args, scene, t0, T, packed_tc=ptc)]


def score64(p_rec, mask_rec, position, mask_p, t0):
    """The score recomputed in float64 from recorded trajectories: per slot in time order, then slots in order."""
    S, T, N = mask_rec.shape
    d = p_rec[:, t0:].astype(np.float64) - position[None, t0:T].astype(np.float64)
    term = np.sqrt(d[..., 0] * d[..., 0] + d[..., 1] * d[..., 1])
    use = (mask_rec[:, t0:] == 1) & (mask_p[None, t0:T] == 1)
    term = np.where(use, term, 0.0)
    return term.sum(axis=1).sum(axis=1), use.sum(axis=(1, 2))


# ---- the per-set forward ---------------------------------------------------------------------------------------------
def _perturbed(sd, s):
    g = torch.Generator().manual_seed(1000 + s)
    return {k: v * (1 + 0.25 * (torch.rand(v.shape, generator=g) - 0.5)) for k, v in sd.items()}


FORWARD_CASES = [("pinnsf_bm", 128, True, 1), ("pinnsf_bm", 64, True, 3), ("pinnsf_bottleneck", 32, True, 3),
                 ("pinnsf_bm", 32, True, 200), ("pinnsf_bottleneck", 64, False, 200), ("pinnsf_bm", 128, False, 3)]


@pytest.mark.parametrize("kind,width,has_obs,S", FORWARD_CASES)
def test_forward_per_set_equals_the_single_network_forward(kind, width, has_obs, S):
    """Set s of piml_pinnsf_forward_tc_sets_f32 equals piml_pinnsf_forward_tc_f32 with set s's vector on set s's rows
    alone, bit for bit: N = 50 agents (not a multiple of the 21 / 12 agents a tile holds), kp = 6, ko = 10, a third of
    the slot rows zero and one set all zero; S = 200 with both branches is 400 (set, branch) groups, more than SMs."""
    from piml_b200 import _lib as L, models as M
    net = seeded(kind, width, 7, has_obs=has_obs)
    spec = M.spec_from_module(net)
    desc = spec.desc()
    n = int(L.load().piml_pinnsf_packed_tc_floats(L.C.byref(desc)))
    stride = -(-n // 32) * 32 + 32                 # a stride larger than one vector is allowed
    packed = torch.empty(S, stride, device="cuda")
    sd = net.state_dict()
    for s in range(S):
        M.pack_device_tc(_perturbed(sd, s) if s else sd, spec, out=packed[s])
    N, kp, ko = 50, 6, (10 if has_obs else 0)
    g = torch.Generator().manual_seed(S)
    ped = torch.randn(S, N, kp, 6, generator=g) * 2
    obs = torch.randn(S, N, max(ko, 1), 6, generator=g) * 2
    ped[torch.rand(S, N, kp, generator=g) < 0.33] = 0
    obs[torch.rand(S, N, max(ko, 1), generator=g) < 0.33] = 0
    slf = torch.randn(S, N, 7, generator=g)
    zero = S // 2
    ped[zero], obs[zero] = 0, 0
    ped, obs, slf = ped.cuda(), obs[:, :, :ko].contiguous().cuda(), slf.cuda()
    acc = torch.full((S, N, 2), float("nan"), device="cuda")
    L.check(L.load().piml_pinnsf_forward_tc_sets_f32(
        L.C.byref(desc), L.ptr(packed), stride, S, 1 if has_obs else 0, spec.tau, L.ptr(ped),
        L.ptr(obs) if has_obs else None, L.ptr(slf), N, kp, ko, L.ptr(acc), L.stream_ptr()),
        "piml_pinnsf_forward_tc_sets_f32")
    for s in range(S):
        want = M.pinnsf_forward(spec, None, ped[s], obs[s] if has_obs else None, slf[s], need_msgs=False,
                                packed_tc=packed[s])[0]
        assert torch.equal(acc[s], want), s
    assert torch.isfinite(acc).all()


def test_forward_rejects_networks_the_16_bit_path_does_not_take():
    from piml_b200 import _lib as L, models as M
    net = seeded("pinnsf_m", 64, 3)
    desc = M.spec_from_module(net).desc()
    x = torch.zeros(64, device="cuda")
    rc = L.load().piml_pinnsf_forward_tc_sets_f32(L.C.byref(desc), L.ptr(x), 1 << 20, 1, 1, 0.5, L.ptr(x), L.ptr(x),
                                                   L.ptr(x), 1, 6, 10, L.ptr(x), L.stream_ptr())
    assert rc == 3, L.last_error()                 # PIML_ERR_UNSUPPORTED


# ---- the sweep ---------------------------------------------------------------------------------------------------------
_RUNS = {}


def gc_sweep():
    """sweep_networks on the full GC clip (t_start = 25, 725 steps) with five networks, the first one given twice."""
    if "gc" not in _RUNS:
        from piml_b200 import _lib as L
        from piml_b200.rollout import sweep_networks
        scene, args, t0, T, i, o = clip("rollout_gc_bm")
        gold = golden_net("rollout_gc_bm")
        others = [golden_net("rollout_gc_bm") for _ in range(3)]
        for k, m in enumerate(others):
            m.load_state_dict(_perturbed(gold.state_dict(), k + 1))
        nets = [others[0], gold, others[1], others[0], others[2]]
        before = L.launch_count()
        e, c, rec = sweep_networks(scene, nets, args, t0, T, record=True)
        launches = L.launch_count() - before
        _RUNS["gc"] = (nets, npy(e), npy(c), [npy(x) for x in rec], launches)
    return _RUNS["gc"]


def test_each_set_equals_its_own_rollout_gc():
    """Every set of the GC sweep records exactly what rollout_scenes records with its network alone: p, v, a and mask
    bit for bit (NaN where NaN); the network given twice records the same trajectory twice."""
    scene, args, t0, T, _, _ = clip("rollout_gc_bm")
    nets, e, c, rec, launches = gc_sweep()
    assert launches >= 3 * (T - t0)
    for s, net in enumerate(nets):
        for got, ref in zip(rec, alone(scene, args, t0, T, net)):
            assert np.array_equal(got[s], ref, equal_nan=True), s
    for got in rec:
        assert np.array_equal(got[0], got[3], equal_nan=True)


def test_each_set_equals_its_own_rollout_ucy():
    """The UCY clip: no real obstacles (the two dummy ones), dataset 'ucy', tau = 5/6."""
    from piml_b200 import models as M
    from piml_b200.rollout import sweep_networks
    scene, args, t0, T, _, _ = clip("rollout_ucy_bm")
    gold = golden_net("rollout_ucy_bm")
    assert M.spec_from_module(gold).tau == pytest.approx(5 / 6) and scene["obstacles"].shape == (2, 2)
    other = golden_net("rollout_ucy_bm")
    other.load_state_dict(_perturbed(gold.state_dict(), 9))
    nets = [other, gold, other]
    e, c, rec = sweep_networks(scene, nets, args, t0, T, record=True)
    for s, net in enumerate(nets):
        for got, ref in zip(rec, alone(scene, args, t0, T, net)):
            assert np.array_equal(npy(got[s]), ref, equal_nan=True), s


@pytest.mark.parametrize("case", ["last_frame", "no_obstacles"])
def test_edges_equal_their_own_rollouts(case):
    """t_start = T - 1 (one step), and a clip without obstacles (M = 0) with networks without an obstacle branch."""
    from piml_b200.rollout import sweep_networks
    scene, args, t0, T, i, _ = clip("rollout_gc_bm")
    if case == "last_frame":
        t0 = T - 1
        nets = [seeded("pinnsf_bm", 64, s) for s in (1, 2)]
    else:
        T = min(T, t0 + 150)
        scene = dict(scene, obstacles=torch.zeros(0, 2, device="cuda"))
        nets = [seeded("pinnsf_bottleneck", 32, s, has_obs=False) for s in (1, 2, 3)]
    scene = with_features_at(scene, args, t0)
    e, c, rec = sweep_networks(scene, nets, args, t0, T, record=True)
    for s, net in enumerate(nets):
        for got, ref in zip(rec, alone(scene, args, t0, T, net)):
            assert np.array_equal(npy(got[s]), ref, equal_nan=True), (case, s)
    want_e, want_c = score64(npy(rec[0]), npy(rec[3]), i["position"], i["mask_p"], t0)
    assert np.array_equal(npy(c), want_c)
    assert np.all(np.abs(npy(e) - want_e) <= 1e-6 * np.abs(want_e))
    if case == "last_frame":                     # the state at t_start is the clip's: nothing to miss yet
        assert np.all(npy(e) == 0.0) and np.all(npy(c) == int(i["mask_p"][t0].sum()))


def test_golden_network_inside_a_sweep():
    """The network of the golden GC rollout at position 2 of 4 passes the gate of the free-running GC rollout test."""
    from piml_b200.rollout import sweep_networks
    scene, args, t0, T, _, o = clip("rollout_gc_bm")
    gold = golden_net("rollout_gc_bm")
    nets = [golden_net("rollout_gc_bm") for _ in range(4)]
    for k in (0, 1, 3):
        nets[k].load_state_dict(_perturbed(gold.state_dict(), 20 + k))
    nets[2] = gold
    e, c, (p_res, v_res, a_res, mask) = sweep_networks(scene, nets, args, t0, T, record=True)
    p_res, mask = npy(p_res[2]), npy(mask[2])
    assert np.array_equal(mask, o["mask_p"])
    drift = np.linalg.norm(p_res - o["position"], axis=-1)
    first = min(T, t0 + 26)
    assert np.array_equal(np.isnan(p_res[:first]), np.isnan(o["position"][:first]))
    assert np.nanmax(drift[:first]) < 1e-4
    assert np.nanmax(drift) < 0.5


def test_score_matches_float64_recomputation():
    """err_sum within 1e-6 relative of a float64 sum over the recorded trajectories, err_count exact; the network given
    twice scores the same bits."""
    _, _, t0, T, i, _ = clip("rollout_gc_bm")
    nets, e, c, rec, _ = gc_sweep()
    want_e, want_c = score64(rec[0], rec[3], i["position"], i["mask_p"], t0)
    assert np.array_equal(c, want_c)
    assert np.all(np.abs(e - want_e) <= 1e-6 * np.abs(want_e)), (e, want_e)
    assert np.all(c > 0)
    assert e[0] == e[3] and c[0] == c[3]


def test_score_does_not_depend_on_the_batch():
    """A set's score alone, at other positions of a permuted list, without record and on a repeated call: the same
    bits."""
    from piml_b200.rollout import sweep_networks
    scene, args, t0, T, _, _ = clip("rollout_gc_bm")
    nets, e5, c5, _, _ = gc_sweep()
    for s in (1, 4):
        e1, c1 = sweep_networks(scene, [nets[s]], args, t0, T)
        assert npy(e1)[0] == e5[s] and npy(c1)[0] == c5[s], s
    perm = [4, 2, 0, 1, 3]
    e, c = sweep_networks(scene, [nets[k] for k in perm], args, t0, T)
    assert np.array_equal(npy(e), e5[perm]) and np.array_equal(npy(c), c5[perm])
    e_again, c_again = sweep_networks(scene, [nets[k] for k in perm], args, t0, T)
    assert torch.equal(e_again, e) and torch.equal(c_again, c)


def test_sweep_of_512_networks_fits_in_memory_linear_in_sets_and_slots():
    """S = 512 score-only on the full GC clip: peak device memory below the packed networks plus a bound linear in
    S N; three sampled sets score as they do alone, and as a float64 recomputation from their own rollouts."""
    from piml_b200 import _lib as L, models as M
    from piml_b200.rollout import sweep_networks
    scene, args, t0, T, i, _ = clip("rollout_gc_bm")
    N = scene["position"].shape[2]
    S = 512
    nets = [seeded("pinnsf_bm", 32, s) for s in range(S)]
    desc = M.spec_from_module(nets[0]).desc()
    packed_bytes = S * 4 * (-(-int(L.load().piml_pinnsf_packed_tc_floats(L.C.byref(desc))) // 32) * 32)
    torch.cuda.synchronize()
    base = torch.cuda.memory_allocated()
    torch.cuda.reset_peak_memory_stats()
    e, c = sweep_networks(scene, nets, args, t0, T)
    torch.cuda.synchronize()
    peak = torch.cuda.max_memory_allocated() - base
    assert peak < packed_bytes + 1024 * S * N + (64 << 20), peak
    assert (c > 0).all()
    for k in (0, 301, S - 1):
        e1, c1 = sweep_networks(scene, [nets[k]], args, t0, T)
        assert torch.equal(e[k:k + 1], e1) and torch.equal(c[k:k + 1], c1), k
        p_own, _, _, mask_own = alone(scene, args, t0, T, nets[k])
        want_e, want_c = score64(p_own[None], mask_own[None], i["position"], i["mask_p"], t0)
        assert int(npy(c)[k]) == int(want_c[0]) and abs(float(npy(e)[k]) - want_e[0]) <= 1e-6 * abs(want_e[0]), k


def test_no_networks():
    """S = 0: empty results, no library launch."""
    from piml_b200 import _lib as L
    from piml_b200.rollout import sweep_networks
    scene, args, t0, T, _, _ = clip("rollout_gc_bm")
    before = L.launch_count()
    e, c = sweep_networks(scene, [], args, t0, T)
    assert e.shape == (0,) and c.shape == (0,) and e.dtype == torch.float64 and c.dtype == torch.int64
    e, c, rec = sweep_networks(scene, [], args, t0, T, record=True)
    assert rec[0].shape == (0, T, scene["position"].shape[2], 2)
    assert L.launch_count() == before
