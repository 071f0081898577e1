"""Runs where the upstream source tree is available (tests.util.reference_available, skipped elsewhere): the oracle
against the UNMODIFIED reference imported live, on EVERY frame of the reference's own clips (SURVEY.md A.2b: toy,
GC 1000-1060, synthetic 1560-1620, UCY 0-54) -- the committed golden vectors hold a subset of these frames."""
import os
import sys

import numpy as np
import pytest
import torch

from oracle import oracle as O
from tests.util import reference_available, valid_sets

HAVE_REF = reference_available()
pytestmark = pytest.mark.skipif(not HAVE_REF, reason="reference tree not present")


def _harness():
    sys.path.insert(0, os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden"))
    import _refharness as H
    return H


@pytest.mark.parametrize("clip,step", [("TOY_CLIP", 1), ("GC_CLIP", 3), ("SYN_CLIP", 3), ("UCY_CLIP", 4)])
def test_oracle_features_equal_live_reference_on_whole_clips(clip, step):
    """get_relative_features (data.py:466-512) frame by frame (T = 1 calls, as the rollout makes them) over the clip."""
    H = _harness()
    DATA, *_ = H.import_reference()
    torch.set_num_threads(1)
    raw = H.load_raw(getattr(H, clip))
    ped = DATA.Pedestrians()
    T = raw.position.shape[0]
    n = 0
    for t in range(0, T, step):
        p, d = raw.position[t:t + 1].clone(), raw.destination[t:t + 1].clone()
        v, a = raw.velocity[t:t + 1].clone(), raw.acceleration[t:t + 1].clone()
        if not bool((~torch.isnan(p[..., 0])).any()):
            continue
        with H.quiet():
            pf, of, df = ped.get_relative_features(p, v, a, d, raw.obstacles.clone(), 6, 90, 4, 10, 90, 4)
        v2, a2 = raw.velocity[t:t + 1].numpy().copy(), raw.acceleration[t:t + 1].numpy().copy()
        want = O.relative_features(raw.position[t:t + 1].numpy(), v2, a2, raw.destination[t:t + 1].numpy(),
                                   raw.obstacles.numpy())
        assert np.array_equal(want[0], pf.numpy()), (clip, t)
        assert np.array_equal(want[1], of.numpy()), (clip, t)
        assert np.array_equal(want[2], df.numpy()), (clip, t)
        assert np.array_equal(v2, v.numpy()) and np.array_equal(a2, a.numpy())      # in-place NaN -> 0 side effect
        n += 1
    assert n >= 40


def test_oracle_selection_equals_live_reference_on_gc_frames():
    """get_nearby_obj_in_sight (data.py:416-447): valid sets {idx: dist <= thr} and distances, angles 90 and 100."""
    H = _harness()
    DATA, *_ = H.import_reference()
    raw = H.load_raw(H.GC_CLIP)
    ped = DATA.Pedestrians()
    for t in range(30, raw.position.shape[0], 45):
        p, v = raw.position[t:t + 1].clone(), raw.velocity[t:t + 1].clone()
        v[torch.isnan(v)] = 0
        head = ped.get_heading_direction(v)
        for angle in (90, 100):
            dist, idx = ped.get_nearby_obj_in_sight(p.clone(), p.clone(), head, 6, angle)
            od, oi = O.select(p.numpy(), p.numpy(), head.numpy(), 6, angle)
            assert np.array_equal(od, dist.numpy()), (t, angle)
            assert valid_sets(oi, od, 4) == valid_sets(idx.numpy(), dist.numpy(), 4), (t, angle)


@pytest.mark.parametrize("N,ver,seed", [(5, "GC", 1), (333, "GC", 2), (1500, "GC", 3), (700, "raw", 4)])
def test_oracle_mlapm_equals_live_reference(N, ver, seed):
    """MLAPM.step (mlapm.py:10-58) live on seeded crowds (incl. stationary agents): 1e-5 per agent, operand-relative."""
    H = _harness()
    _, _, MLAPM, _, _ = H.import_reference()
    g = torch.Generator().manual_seed(seed)
    side = (N / 0.5) ** 0.5
    p, d = torch.rand(N, 2, generator=g) * side, torch.rand(N, 2, generator=g) * side
    v = torch.randn(N, 2, generator=g)
    v[torch.rand(N, generator=g) < 0.1] = 0
    ds = 1.34 + 0.3 * torch.randn(N, 1, generator=g)
    kw = dict(version=ver, tau=0.5, A=7.55, B=-3.00, C=0.2, D=-0.3, theta=56)
    ref = MLAPM.MLAPM(**kw).step(p.clone(), v.clone(), ds.clone(), d.clone(), 0.08).numpy()
    got = O.mlapm_step(p.numpy(), v.numpy(), ds.numpy(), d.numpy(), 0.08, ver)
    num = np.linalg.norm(got.astype(np.float64) - ref, axis=-1)
    den = np.maximum(np.maximum(np.linalg.norm(ref, axis=-1), np.linalg.norm(v.numpy(), axis=-1)), 1e-6)
    assert float((num / den).max()) < 1e-5


@pytest.mark.parametrize("kind", ["pinnsf_bm", "pinnsf_m", "pinnsf_bottleneck", "pinnsf"])
def test_oracle_network_equals_live_reference_module(kind):
    """The four PINNSF forwards (model.py:762, :1104, :1185, :1271) instantiated live with a fresh seed, eval mode, on
    random features with zero-padded slots: every output of the oracle within 1e-5."""
    from piml_b200 import models as M
    from tests.golden_args import base_args
    from tests.util import accel_err, rel_vec_err
    H = _harness()
    _, MODEL, _, _, _ = H.import_reference()
    cls = {"pinnsf_bm": "PINNSF_bottleneck_multitask", "pinnsf_m": "PINNSF_multitask",
           "pinnsf_bottleneck": "PINNSF_bottleneck", "pinnsf": "PINNSF"}[kind]
    args = base_args(model=kind, dataset_name="gc1560")
    torch.manual_seed(1234)
    net = getattr(MODEL, cls)(args).eval()
    g = torch.Generator().manual_seed(5)
    R = 37
    ped, obs, slf = torch.randn(R, 6, 6, generator=g), torch.randn(R, 10, 6, generator=g), torch.randn(R, 7, generator=g)
    ped[:, 4:] = 0
    obs[::2] = 0
    with torch.no_grad():
        ref = net(ped.clone(), obs.clone(), slf.clone())
    spec = M.spec_from_module(net)
    desc = O.net_desc(spec.enc_dims, spec.proc_mode, spec.dec_dims, spec.coll_dims, spec.kind)
    out = O.pinnsf_forward(desc, M.pack_state_dict(net.state_dict(), spec).numpy(), spec.tau, ped.numpy(), obs.numpy(),
                           slf.numpy(), spec.has_obs)
    assert len(out) == len(ref)
    assert accel_err(out[0], ref[0].numpy(), slf.numpy(), spec.tau) < 1e-5
    for o, r_ in zip(out[1:], ref[1:]):
        r_ = r_.numpy()
        o = o.reshape(r_.shape)
        err = rel_vec_err(o, r_, floor=1e-3) if r_.ndim >= 2 and r_.shape[-1] > 1 else float(np.abs(o - r_).max())
        assert err < 1e-5, (kind, err)
