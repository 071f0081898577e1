"""CPU checks of MLAPM.advance_scenes: malformed arguments are rejected before the library is touched."""
import pytest
import torch

from piml_b200 import _lib as L
from piml_b200.mlapm import MLAPM

KW = dict(version='GC', tau=0.5, A=7.55, B=-3.0, C=0.2, D=-0.3, theta=56)


@pytest.fixture
def no_library(monkeypatch):
    def refuse():
        raise AssertionError("the library was called")
    monkeypatch.setattr(L, "load", refuse)


def args(S=3, N=5):
    x = torch.zeros(S, N, 2)
    return [x, x.clone(), torch.ones(S, N, 1), x.clone(), torch.ones(S, N, dtype=torch.bool)]


@pytest.mark.parametrize("case", ["pos2d", "vel_shape", "dest_shape", "last_axis", "ds_shape", "ds_dim3",
                                  "active_dtype", "active_shape", "params_shape", "params_list"])
def test_advance_scenes_rejects_malformed_arguments(no_library, case):
    p, v, ds, d, act = args()
    params = None
    if case == "pos2d":
        p = p[0]
    elif case == "vel_shape":
        v = torch.zeros(3, 4, 2)
    elif case == "dest_shape":
        d = torch.zeros(2, 5, 2)
    elif case == "last_axis":
        p, v, d = torch.zeros(3, 5, 3), torch.zeros(3, 5, 3), torch.zeros(3, 5, 3)
    elif case == "ds_shape":
        ds = torch.ones(3, 4)
    elif case == "ds_dim3":
        ds = torch.ones(3, 5, 3)
    elif case == "active_dtype":
        act = act.to(torch.uint8)
    elif case == "active_shape":
        act = torch.ones(3, 6, dtype=torch.bool)
    elif case == "params_shape":
        params = torch.zeros(3, 5)
    elif case == "params_list":
        params = [[0.5, 7.55, -3.0, 0.2, -0.3, 56.0]] * 3
    with pytest.raises(ValueError):
        MLAPM(**KW).advance_scenes(p, v, ds, d, act, 0.08, params=params)


def test_advance_scenes_rejects_ucy_before_library(no_library):
    with pytest.raises(NotImplementedError):
        MLAPM(**dict(KW, version='UCY')).advance_scenes(*args(), 0.08)
