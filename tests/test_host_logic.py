"""CPU tests of the host-side logic: parameter packing, the module mirrors' state_dict/initialisation parity with
the reference, spec derivation and the cos-threshold constant."""
import numpy as np
import pytest
import torch

from tests.golden_args import base_args, model_args
from tests.util import golden, group, reference_available


def test_cos_threshold_matches_reference_constant():
    from piml_b200 import cos_threshold
    assert np.float32(cos_threshold(90)) == np.float32(7.9632673e-4)      # SURVEY.md A.1
    assert cos_threshold(100) < 0 < cos_threshold(60)


@pytest.mark.parametrize("kind", ["pinnsf_bm", "pinnsf_m", "pinnsf_bottleneck", "pinnsf"])
def test_mirror_modules_share_keys_and_seeded_init_with_reference(kind):
    """Same state_dict keys/shapes as the reference classes, and torch.manual_seed(666) reproduces the reference's
    initial weights bit-for-bit (sub-modules are created in the reference's order)."""
    from piml_b200 import models as M
    g = group(golden("models"), kind)
    args = model_args(kind, g["cfg"], str(g["dataset_name"]))
    torch.manual_seed(666)
    m = M.CLASSES[kind](args)
    sd = m.state_dict()
    ref = {k[3:]: v for k, v in g.items() if k.startswith("sd/")}
    assert sorted(sd) == sorted(ref)
    for k in sd:
        assert np.array_equal(sd[k].numpy(), ref[k]), k
    assert m.tau == pytest.approx(float(g["tau"]))


def test_pack_layouts():
    from piml_b200 import models as M
    g = group(golden("models"), "pinnsf_bm")
    args = model_args("pinnsf_bm", g["cfg"], "gc1560")
    spec = M.spec_from_args("pinnsf_bm", args)
    sd = {k[3:]: torch.from_numpy(v) for k, v in g.items() if k.startswith("sd/")}
    b = M.pack_state_dict(sd, spec)
    n_branch = 6 * 128 + 128 + 2 * (128 * 128 + 128) + 128 * 64 + 64 + 64 * 64 + 64 + 64 * 2 + 2
    assert b.numel() == 2 * n_branch + 64 * 64 + 64 + 64 + 1
    w0 = sd["ped_encoder.mlp.0.weight"]
    assert torch.equal(b[:768].view(128, 6), w0)
    # the device layout pads every Linear to 16*NJ columns (+ a padded bias); size comes from the library (no GPU)
    from piml_b200 import _lib
    desc = spec.desc()
    n_dev = _lib.load().piml_pinnsf_packed_floats(_lib.C.byref(desc))
    pad = lambda k, o: (k + 1) * (16 * (8 if o > 64 else 4 if o > 32 else 2 if o > 16 else 1))   # noqa: E731
    n_branch_dev = pad(6, 128) + 2 * pad(128, 128) + pad(128, 64) + pad(64, 64) + pad(64, 2)
    assert n_dev == 2 * n_branch_dev + pad(64, 64) + pad(64, 1)
    # dead weights (ResDNN block-0 Linear when processor_hidden_layers > 1) are not packed
    assert spec.proc_mode == 0 and not any("processor" in k for k in M.linear_keys(spec))


def test_spec_from_module_matches_spec_from_args():
    from piml_b200 import models as M
    for kind, over in (("pinnsf_bm", {}), ("pinnsf_m", {}), ("pinnsf", dict(processor_hidden_layers=1,
                                                                              encoder_hidden_size=32,
                                                                              processor_hidden_size=32))):
        args = base_args(model=kind, **over)
        m = M.CLASSES[kind](args)
        s1, s2 = M.spec_from_args(kind, args), M.spec_from_module(m)
        for f in ("enc_dims", "proc_mode", "dec_dims", "coll_dims", "kind", "has_obs", "tau"):
            assert getattr(s1, f) == getattr(s2, f), (kind, f)


@pytest.mark.skipif(not reference_available(), reason="reference tree not present")
@pytest.mark.parametrize("layers", [16, 3, 1])
def test_train_mode_dropout_masks_follow_the_reference_rng_stream(layers):
    """ResDNN.forward draws one Dropout mask per block and applies only the last (model.py:115-119).  Under the same
    seed the multipliers the CUDA path applies must be the reference's, and torch's RNG must end in the same state."""
    import sys, os
    sys.path.insert(0, os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden"))
    import _refharness as H
    import torch
    from piml_b200 import models as M
    DATA, MODEL, *_ = H.import_reference()
    args = H.default_args(model="pinnsf_bm", dataset_name="gc1560", processor_hidden_layers=layers)
    torch.manual_seed(1)
    net = MODEL.PINNSF_bottleneck_multitask(args).train()
    spec = M.spec_from_module(net)
    assert spec.n_blocks == layers and M.spec_from_args("pinnsf_bm", args).n_blocks == layers
    ped, obs, slf = torch.randn(9, 6, 6), torch.randn(9, 10, 6), torch.randn(9, 7)
    seen = []
    hook = lambda mod, inp, out: seen.append((out / inp[0]).detach().clone())
    handles = [net.ped_processor.dropout.register_forward_hook(hook), net.obs_processor.dropout.register_forward_hook(hook)]
    torch.manual_seed(123)
    net(ped, obs, slf)
    after_ref = torch.rand(4)
    for h in handles:
        h.remove()
    assert len(seen) == 2 * layers                        # one draw per block and branch
    torch.manual_seed(123)
    dp, do = M._dropout_multipliers(spec, True, ped, obs)
    after = torch.rand(4)
    want_p, want_o = torch.nan_to_num(seen[layers - 1], nan=0.0), torch.nan_to_num(seen[-1], nan=0.0)
    ok_p, ok_o = seen[layers - 1].isfinite(), seen[-1].isfinite()          # 0/0 where the block output is exactly 0
    assert torch.equal(dp[ok_p], want_p[ok_p]) and torch.equal(do[ok_o], want_o[ok_o])
    assert ok_p.float().mean() > 0.9
    assert torch.equal(after, after_ref)


@pytest.mark.parametrize("case,kind", [("pinnsf_bm_train", "pinnsf_bm"), ("pinnsf_m_train", "pinnsf_m")])
def test_train_mode_dropout_masks_equal_the_recorded_reference_masks(case, kind):
    """The same draw as above against the masks the reference module applied in train() mode (training_step.npz,
    16 processor blocks; make_golden.py seeds torch with 666 + 1 right before that forward)."""
    from piml_b200 import models as M
    from tests.test_training_ref import drop_masks
    z = golden("training_step")
    g = group(z, case)
    spec = M.spec_from_args(kind, base_args(model=kind, dataset_name=str(g["dataset_name"])))
    assert spec.n_blocks == 16
    ped, obs = torch.from_numpy(z["ped"]), torch.from_numpy(z["obs"])
    torch.manual_seed(667)
    dp, do = M._dropout_multipliers(spec, True, ped, obs)
    want_p, want_o = drop_masks(g)
    assert torch.equal(dp, want_p) and torch.equal(do, want_o)


def test_non_relu_single_block_processor_is_rejected():
    """args.activation only reaches the forward through the single-block processor; the kernels implement ReLU."""
    import argparse
    from piml_b200 import models as M
    a = argparse.Namespace(model='pinnsf_bm', dataset_name='gc1560', dropout=0.5, encoder_hidden_size=128,
                           processor_hidden_size=128, decoder_hidden_size=64, encoder_hidden_layers=3,
                           processor_hidden_layers=1, decoder_hidden_layers=2, ped_feature_dim=6, obs_feature_dim=6,
                           self_feature_dim=7, activation='sigmoid')
    with pytest.raises(NotImplementedError):
        M.spec_from_args('pinnsf_bm', a)
    a.activation = 'relu'
    assert M.spec_from_args('pinnsf_bm', a).proc_mode == 1
    a.processor_hidden_layers, a.activation = 16, 'leaky_relu'       # discarded Linear: activation never applied
    assert M.spec_from_args('pinnsf_bm', a).proc_mode == 0


def test_fused_step_host_side():
    """piml_nn_step_supported (pure host logic of the library, no GPU needed): per-slot-decoder networks with widths the
    16-bit tensor-core kernel runs are accepted, the summed-embedding kind and odd widths are not; NNStep has no CPU
    fallback; the graphed training step insists on a capturable optimizer before it touches the device."""
    import argparse
    from piml_b200 import _lib as L, models as M
    from piml_b200.rollout import NNStep
    from piml_b200.train_graph import GraphedRolloutTraining
    base = dict(dataset_name='gc1560', dropout=0.5, encoder_hidden_size=128, processor_hidden_size=128,
                decoder_hidden_size=64, encoder_hidden_layers=3, processor_hidden_layers=16, decoder_hidden_layers=2,
                ped_feature_dim=6, obs_feature_dim=6, self_feature_dim=7)
    lib = L.load()
    ok = lambda model, **kw: bool(lib.piml_nn_step_supported(
        L.C.byref(M.spec_from_args(model, argparse.Namespace(model=model, **dict(base, **kw))).desc())))
    assert ok('pinnsf_bm') and ok('pinnsf_bottleneck')
    assert ok('pinnsf_bm', encoder_hidden_size=64, processor_hidden_size=64, decoder_hidden_size=32)
    assert not ok('pinnsf_m')                                             # summed embeddings: not a per-slot decoder
    assert not ok('pinnsf_bm', decoder_hidden_size=48)                    # width the kernel has no tile shape for
    assert not ok('pinnsf_bm', processor_hidden_layers=1)                 # single-block processor: FP32-pipe path only
    if not torch.cuda.is_available():
        spec = M.spec_from_args('pinnsf_bm', argparse.Namespace(model='pinnsf_bm', **base))
        z = torch.zeros(1, 8, 2)
        with pytest.raises(RuntimeError, match="no CPU fallback"):
            NNStep(spec, torch.zeros(4), z, z.clone(), z.clone(), z.clone(), torch.zeros(1, 8, dtype=torch.int64),
                   z.clone(), torch.ones(1, 8, dtype=torch.int64), z[:, None].clone(), torch.ones(1, 8), torch.zeros(3, 2),
                   0.08, 6, 90, 4, 10, 90, 4)
    opt = torch.optim.Adam([torch.nn.Parameter(torch.zeros(2))], lr=1e-3)
    with pytest.raises(ValueError, match="capturable"):
        GraphedRolloutTraining(argparse.Namespace(), opt, argparse.Namespace())
