"""CPU checks of piml_b200.rollout.sweep_networks: malformed clips and network lists are rejected before any device
work, networks the 16-bit tensor-core forward cannot run raise NotImplementedError, and the ctypes argument block,
signatures and workspace query match include/piml_b200.h."""
import pytest
import torch

from piml_b200 import _lib as L
from piml_b200 import models as M
from piml_b200.rollout import sweep_networks
from tests.golden_args import model_args
from tests.test_sfm_sweep_args import _header_struct, scene, D, M as MO, N, T


class _HostQueryOnly(object):
    """Stands in for the library: answers the host-only capability query, refuses everything else."""

    @staticmethod
    def piml_nn_step_supported(desc):
        return 1

    def __getattr__(self, name):
        raise AssertionError(f"the library was called: {name}")


@pytest.fixture
def no_library(monkeypatch):
    """No library work apart from asking whether the 16-bit forward takes the network."""
    monkeypatch.setattr(L, "load", lambda: _HostQueryOnly())


def net(kind="pinnsf_bm", width=32, dataset_name="gc1560", has_obs=True, seed=0):
    torch.manual_seed(seed)
    return M.CLASSES[kind](model_args(kind, (width, width, width, 2, 2, 2, 1 if has_obs else 0), dataset_name))


def args():
    return model_args("pinnsf_bm", (32, 32, 32, 2, 2, 2, 1), "gc1560")


CLIP_CASES = ["two_scenes", "position_3d", "velocity_shape", "dest_idx_shape", "mask_shape", "waypoints_shape",
              "dest_num_shape", "desired_speed_shape", "obstacles_per_scene", "ped_features_topk", "obs_features_topk",
              "self_features_shape", "missing_key", "t_start_negative", "t_start_past_num_frames", "t_start_float",
              "time_unit_zero"]


@pytest.mark.parametrize("empty", [False, True])
@pytest.mark.parametrize("case", CLIP_CASES)
def test_sweep_rejects_malformed_clips(no_library, case, empty):
    """The clip checks sfm.sweep applies, with a network list and with an empty one."""
    sc, a, t0, nf = scene(), args(), 2, None
    if case == "two_scenes":
        for k in ("position", "velocity", "acceleration", "destination"):
            sc[k] = torch.zeros(2, T, N, 2)
    elif case == "position_3d":
        sc["position"] = sc["position"][0]
    elif case == "velocity_shape":
        sc["velocity"] = torch.zeros(1, T, N + 1, 2)
    elif case == "dest_idx_shape":
        sc["dest_idx"] = torch.zeros(1, T, N + 1, dtype=torch.int64)
    elif case == "mask_shape":
        sc["mask_p"] = torch.ones(1, T - 1, N)
    elif case == "waypoints_shape":
        sc["waypoints"] = torch.zeros(1, D, N, 3)
    elif case == "dest_num_shape":
        sc["dest_num"] = torch.ones(N, dtype=torch.int64)
    elif case == "desired_speed_shape":
        sc["desired_speed"] = torch.ones(1, N + 2)
    elif case == "obstacles_per_scene":
        sc["obstacles"] = torch.zeros(2, MO, 2)
    elif case == "ped_features_topk":
        sc["ped_features0"] = torch.zeros(1, N, 3, 6)
    elif case == "obs_features_topk":
        sc["obs_features0"] = torch.zeros(1, N, MO + 1, 6)
    elif case == "self_features_shape":
        sc["self_features0"] = torch.zeros(1, N, 6)
    elif case == "missing_key":
        del sc["mask_p_pred"]
    elif case == "t_start_negative":
        t0 = -1
    elif case == "t_start_past_num_frames":
        t0, nf = 6, 6
    elif case == "t_start_float":
        t0 = 2.0
    elif case == "time_unit_zero":
        a.time_unit = 0.0
    models = [] if empty else [net(), net(seed=1)]
    with pytest.raises(ValueError, match="sweep_networks"):
        sweep_networks(sc, models, a, t0, nf)


@pytest.mark.parametrize("case", ["other_class", "other_width", "other_tau", "obs_branch_differs", "not_a_list"])
def test_sweep_rejects_mixed_networks(no_library, case):
    """One sweep takes one architecture and one tau: checked before the library or the device is touched."""
    models = [net(), net(seed=1)]
    if case == "other_class":
        models.append(net("pinnsf_bottleneck"))
    elif case == "other_width":
        models.append(net(width=64))
    elif case == "other_tau":
        models.append(net(dataset_name="ucy"))          # pinnsf_bm: tau 5/6 on ucy, 2 elsewhere
    elif case == "obs_branch_differs":
        models.append(net(has_obs=False))
    else:
        models = models[0]
    with pytest.raises(ValueError, match="sweep_networks"):
        sweep_networks(scene(), models, args(), 2)


@pytest.mark.parametrize("kind", ["pinnsf_m", "pinnsf"])
def test_networks_without_the_16_bit_path_raise_not_implemented(kind):
    """Kind-1 networks (summed embeddings) run on the tf32 / FP32 paths only: NotImplementedError, and before any
    device work (on a machine without a GPU the device would raise RuntimeError)."""
    with pytest.raises(NotImplementedError):
        sweep_networks(scene(), [net(kind), net(kind, seed=1)], model_args(kind, (32, 32, 32, 2, 2, 2, 1), "gc1560"),
                       2)


def test_network_widths_the_16_bit_path_does_not_take_raise_not_implemented():
    with pytest.raises(NotImplementedError):
        sweep_networks(scene(), [net(width=96)], args(), 2)


def test_empty_network_list_passes_validation_up_to_the_device(no_library):
    """No networks: a valid clip is accepted (the result is empty); the refusal here is the missing device."""
    if torch.cuda.is_available():
        pytest.skip("on a GPU machine the call would run")
    with pytest.raises(RuntimeError, match="no CPU fallback"):
        sweep_networks(scene(), [], args(), 2)


def test_ctypes_argument_block_matches_the_header():
    want = _header_struct("piml_nn_sweep_args")
    got = L.NnSweepArgs._fields_
    assert [f[0] for f in want] == [f[0] for f in got]
    kinds = {"int": L.i32, "float": L.f32, "int64_t": L.i64}
    for (name, ctype, is_ptr), (gname, gtype) in zip(want, got):
        if name == "desc":
            assert gtype is L.C.POINTER(L.NetDesc)
        else:
            assert gtype is (L.vp if is_ptr else kinds[ctype]), name


def test_signatures():
    assert L.SIGNATURES["piml_nn_sweep_f32"] == (L.i32, [L.C.POINTER(L.NnSweepArgs), L.vp])
    assert L.SIGNATURES["piml_nn_sweep_workspace_bytes"] == (L.i64, [L.C.POINTER(L.NnSweepArgs)])
    lib = L.load()
    for name in ("piml_nn_sweep_f32", "piml_nn_sweep_workspace_bytes", "piml_pinnsf_forward_tc_sets_f32"):
        assert hasattr(lib, name)


def test_workspace_is_linear_in_sets_and_slots():
    """The workspace query needs no device: O(S N) bytes, none of them per frame."""
    r = L.NnSweepArgs()
    r.M, r.D, r.kp, r.ko, r.thr_p, r.thr_o = 100, 1, 6, 10, 4.0, 4.0
    sizes = {}
    for S, N, Tn in ((1024, 110, 750), (2048, 110, 750), (2048, 110, 10), (1024, 220, 750)):
        r.S, r.N, r.T = S, N, Tn
        sizes[(S, N, Tn)] = L.load().piml_nn_sweep_workspace_bytes(L.C.byref(r))
    assert sizes[(2048, 110, 750)] == sizes[(2048, 110, 10)]
    assert 2 * sizes[(1024, 110, 750)] - 4096 <= sizes[(2048, 110, 750)] <= 2 * sizes[(1024, 110, 750)]
    assert 2 * sizes[(1024, 110, 750)] - 4096 <= sizes[(1024, 220, 750)] <= 2 * sizes[(1024, 110, 750)]
    assert sizes[(2048, 110, 750)] < 1024 * 2048 * 110
    r.S = -1
    assert L.load().piml_nn_sweep_workspace_bytes(L.C.byref(r)) < 0
