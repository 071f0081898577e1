"""The opt-in switch: piml_b200.patch swaps the five reference signatures and restores them (CPU, no compute)."""
import sys
import types

import pytest

from tests.util import reference_available


def _fake_reference():
    DATA = types.ModuleType("data.data")

    class Pedestrians(object):
        @staticmethod
        def get_heading_direction(velocity):
            return "ref"

        def get_nearby_obj_in_sight(self, position, objects, heading_direction, k, angle_threshold):
            return "ref"

        def get_relative_features(self, *a):
            return "ref"

        @staticmethod
        def calculate_collision_label(ped_features):
            return "ref"

        @staticmethod
        def collision_detection(position, threshold, real_position=None):
            return "ref"

    class RawData(object):
        pass
    DATA.Pedestrians, DATA.RawData = Pedestrians, RawData
    DATA.TimeIndexedPedData = type("TimeIndexedPedData", (Pedestrians,), {"make_dataset": lambda self, a, r: "ref"})
    MODEL = types.ModuleType("models.model")
    for c in ("PINNSF", "PINNSF_bottleneck", "PINNSF_bottleneck_multitask", "PINNSF_multitask"):
        setattr(MODEL, c, type(c, (), {"forward": lambda self, p, o, s: "ref"}))
    ML = types.ModuleType("models.mlapm")
    ML.MLAPM = type("MLAPM", (), {"__init__": lambda self, **a: setattr(self, "args", a),
                                  "step": lambda self, *a, **k: "ref"})
    UT = types.ModuleType("utils.utils")
    UT.calc_acceleration = lambda *a, **k: "ref"
    SIM = types.ModuleType("models.simulators")
    SIM.DATA = DATA
    SIM.BaseSimulator = type("BaseSimulator", (Pedestrians,), {"get_multiple_rollouts": lambda self, d, t_start=0,
                                                               load_model=True: "ref",
                                                               "test_multiple_rollouts_for_training":
                                                               lambda self, d, t_start=0: "ref"})
    return DATA, ML, MODEL, SIM, UT


def test_install_swaps_and_uninstall_restores(monkeypatch):
    import piml_b200.patch as patch
    DATA, ML, MODEL, SIM, UT = _fake_reference()
    monkeypatch.delenv("PIML_B200", raising=False)
    assert patch.install_from_env(DATA=DATA, MLAPM_MOD=ML, MODEL=MODEL, SIM=SIM, UTILS=UT) == []
    assert UT.calc_acceleration() == "ref"
    monkeypatch.setenv("PIML_B200", "1")
    names = patch.install_from_env(DATA=DATA, MLAPM_MOD=ML, MODEL=MODEL, SIM=SIM, UTILS=UT)
    assert len(names) == 6 + 1 + 4 + 1 + 1 + 2
    import piml_b200 as P
    assert UT.calc_acceleration is P.calc_acceleration
    assert DATA.Pedestrians.__dict__["get_relative_features"] is P.Pedestrians.__dict__["get_relative_features"]
    # BaseSimulator inherits Pedestrians in the reference (simulators.py:25): the patched method is what it sees
    assert SIM.BaseSimulator.get_relative_features is DATA.Pedestrians.get_relative_features
    assert ML.MLAPM(version="GC").step.__func__.__name__ == "step"
    patch.uninstall()
    assert UT.calc_acceleration() == "ref"
    assert DATA.Pedestrians().get_relative_features() == "ref"
    assert MODEL.PINNSF().forward(0, 0, 0) == "ref"
    assert ML.MLAPM().step() == "ref" and SIM.BaseSimulator().get_multiple_rollouts(None) == "ref"
    assert SIM.BaseSimulator().test_multiple_rollouts_for_training(None) == "ref"
    assert DATA.Pedestrians.collision_detection(0, 0) == "ref"
    assert DATA.TimeIndexedPedData().make_dataset(None, None) == "ref"
    assert not hasattr(DATA.Pedestrians, "_relative_features_raw")       # helper added by install is removed again


@pytest.mark.skipif(not reference_available(), reason="reference tree not present")
def test_install_on_the_real_reference_modules():
    """In the build container: the real reference modules expose exactly the attributes the patch replaces."""
    import os
    sys.path.insert(0, os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden"))
    import _refharness as H
    DATA, MODEL, MLAPM, SIM, UTILS = H.import_reference()
    import piml_b200.patch as patch
    orig = DATA.Pedestrians.get_relative_features
    import functions.metrics as METRIC
    orig_ot = METRIC.ot_with_time_mask
    names = patch.install(DATA=DATA, MLAPM_MOD=MLAPM, MODEL=MODEL, SIM=SIM, UTILS=UTILS, METRIC=METRIC)
    try:
        assert len(names) == 15 + 4
        assert SIM.BaseSimulator.get_relative_features is not orig
        import piml_b200.metrics as MT
        assert METRIC.ot_with_time_mask is MT.ot_with_time_mask and METRIC.collision_count is MT.collision_count
        # simulators.py calls METRIC.<name>(...) through the module object, so it sees the replacements
        assert SIM.METRIC.mmd_with_time_mask is MT.mmd_with_time_mask
    finally:
        patch.uninstall()
    assert DATA.Pedestrians.get_relative_features is orig and METRIC.ot_with_time_mask is orig_ot


def test_social_force_mirror_constants_and_errors():
    """piml_b200.SocialForce: the ped constants are calc_acceleration's v0 constants per dataset (utils.py:47-52), the
    obstacle constants socialforce.yaml's intensity / radius; unknown datasets are rejected (no GPU needed)."""
    import piml_b200 as P
    gc, ucy = P.SocialForce("gc1560").spec, P.SocialForce("ucy").spec
    assert (gc.A_ped, gc.B_ped) == (8.75, -2.5) and (ucy.A_ped, ucy.B_ped) == (10.67, -3.33)
    assert (gc.A_obs, gc.B_obs, gc.tau, gc.eps) == (50.0, -5.0, 0.5, 1e-6)
    assert len(list(P.SocialForce("gc2344").parameters())) == 0
    with pytest.raises(ValueError):
        P.SocialForce("nope")
