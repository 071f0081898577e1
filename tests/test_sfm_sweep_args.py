"""CPU checks of piml_b200.sfm.sweep: malformed arguments are rejected before the library is touched, and the ctypes
argument block and signature match include/piml_b200.h."""
import os
import re

import pytest
import torch

from piml_b200 import _lib as L
from piml_b200 import sfm
from tests.golden_args import base_args

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
T, N, M, D = 12, 5, 4, 2


@pytest.fixture
def no_library(monkeypatch):
    def refuse():
        raise AssertionError("the library was called")
    monkeypatch.setattr(L, "load", refuse)


def scene():
    z2 = torch.zeros(1, T, N, 2)
    return {"position": z2, "velocity": z2.clone(), "acceleration": z2.clone(), "destination": z2.clone(),
            "dest_idx": torch.zeros(1, T, N, dtype=torch.int64), "waypoints": torch.zeros(1, D, N, 2),
            "dest_num": torch.ones(1, N, dtype=torch.int64), "obstacles": torch.zeros(M, 2),
            "mask_p": torch.ones(1, T, N), "mask_p_pred": torch.ones(1, T, N), "desired_speed": torch.ones(1, N),
            "ped_features0": torch.zeros(1, N, min(6, N), 6), "obs_features0": torch.zeros(1, N, min(10, M), 6),
            "self_features0": torch.zeros(1, N, 7)}


def params(S=3):
    return torch.tensor([[8.75, -2.5, 50.0, -5.0, 0.5]] * S)


CASES = ["two_scenes", "position_3d", "velocity_shape", "dest_idx_shape", "mask_shape", "waypoints_shape",
         "dest_num_shape", "desired_speed_shape", "obstacles_per_scene", "ped_features_topk", "obs_features_topk",
         "self_features_shape", "missing_key", "params_width", "params_list", "params_int", "params_nan",
         "params_inf_in_f32", "tau_zero", "tau_negative", "t_start_negative", "t_start_past_num_frames",
         "t_start_float", "time_unit_zero"]


@pytest.mark.parametrize("case", CASES)
def test_sweep_rejects_malformed_arguments(no_library, case):
    sc, prm, args, t0, nf = scene(), params(), base_args(model="sfm", dataset_name="gc1560"), 2, None
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
        sc["obstacles"] = torch.zeros(2, M, 2)
    elif case == "ped_features_topk":
        sc["ped_features0"] = torch.zeros(1, N, 3, 6)
    elif case == "obs_features_topk":
        sc["obs_features0"] = torch.zeros(1, N, M + 1, 6)
    elif case == "self_features_shape":
        sc["self_features0"] = torch.zeros(1, N, 6)
    elif case == "missing_key":
        del sc["mask_p_pred"]
    elif case == "params_width":
        prm = torch.zeros(3, 6)
    elif case == "params_list":
        prm = params().tolist()
    elif case == "params_int":
        prm = params().long()
    elif case == "params_nan":
        prm[1, 2] = float("nan")
    elif case == "params_inf_in_f32":
        prm = params().double()
        prm[0, 0] = 1e39
    elif case == "tau_zero":
        prm[2, 4] = 0.0
    elif case == "tau_negative":
        prm[0, 4] = -0.5
    elif case == "t_start_negative":
        t0 = -1
    elif case == "t_start_past_num_frames":
        t0, nf = 6, 6
    elif case == "t_start_float":
        t0 = 2.0
    elif case == "time_unit_zero":
        args.time_unit = 0.0
    with pytest.raises(ValueError):
        sfm.sweep(sc, prm, args, t0, nf)


def test_sweep_accepts_a_clip_without_obstacles_up_to_the_library(no_library):
    """M = 0 (obstacles (0, 2), obs_features0 of any shape) passes validation: the refusal is the library's."""
    if torch.cuda.is_available():
        pytest.skip("on a GPU machine the call would run")
    sc = scene()
    sc["obstacles"], sc["obs_features0"] = torch.zeros(0, 2), torch.zeros(1, N, 0, 6)
    with pytest.raises(RuntimeError, match="no CPU fallback"):
        sfm.sweep(sc, params(), base_args(model="sfm", dataset_name="gc1560"), 0)


def _header_struct(name):
    src = open(os.path.join(ROOT, "include", "piml_b200.h")).read()
    src = re.sub(r"/\*.*?\*/", "", src, flags=re.S)
    body = re.search(r"typedef struct \{([^}]*)\}\s*" + name + ";", src).group(1)
    fields = []
    for decl in body.split(";"):
        decl = decl.strip()
        if not decl:
            continue
        names = decl.split(None, 2)
        ctype = names[1] if names[0] == "const" else names[0]
        rest = decl[decl.index(ctype) + len(ctype):]
        for n in rest.split(","):
            fields.append((n.strip().lstrip("*"), ctype, "*" in n))
    return fields


def test_ctypes_argument_block_matches_the_header():
    want = _header_struct("piml_sfm_sweep_args")
    got = L.SfmSweepArgs._fields_
    assert [f[0] for f in want] == [f[0] for f in got]
    kinds = {"int": L.i32, "float": L.f32, "int64_t": L.i64}
    for (name, ctype, is_ptr), (gname, gtype) in zip(want, got):
        assert gtype is (L.vp if is_ptr else kinds[ctype]), name


def test_signatures():
    assert L.SIGNATURES["piml_sfm_sweep_f32"] == (L.i32, [L.C.POINTER(L.SfmSweepArgs), L.vp])
    assert L.SIGNATURES["piml_sfm_sweep_workspace_bytes"] == (L.i64, [L.C.POINTER(L.SfmSweepArgs)])
    lib = L.load()
    assert hasattr(lib, "piml_sfm_sweep_f32") and hasattr(lib, "piml_sfm_sweep_workspace_bytes")


def test_workspace_is_linear_in_sets_and_slots():
    """The workspace query needs no device: O(S N) bytes, none of them per frame."""
    r = L.SfmSweepArgs()
    r.N, r.M, r.D, r.kp, r.ko, r.thr_p, r.thr_o = 110, 100, 1, 6, 10, 4.0, 4.0
    os.environ["PIML_SFM_PERSISTENT"] = "0"
    try:
        sizes = {}
        for S, T in ((1024, 750), (2048, 750), (2048, 10)):
            r.S, r.T = S, T
            sizes[(S, T)] = L.load().piml_sfm_sweep_workspace_bytes(L.C.byref(r))
    finally:
        os.environ.pop("PIML_SFM_PERSISTENT", None)
    assert sizes[(2048, 750)] == sizes[(2048, 10)]
    assert 2 * sizes[(1024, 750)] - 4096 <= sizes[(2048, 750)] <= 2 * sizes[(1024, 750)]
    assert sizes[(2048, 750)] < 1024 * 2048 * 110
    r.S = -1
    assert L.load().piml_sfm_sweep_workspace_bytes(L.C.byref(r)) < 0
