"""Randomised self-consistency sweep on the GPU (bounded by --seconds): pairs of independent evaluations that must agree
   1. MLAPM symmetric kernel vs ordered-pair kernel, random N in [2, 40000], versions raw / GC, stationary / NaN agents
   2. cell-list vs all-pairs neighbour features, random N, M, k, angles, thresholds: bit-identical
   3. tensor-core forward compact vs dense (pinnsf_bm row level, pinnsf_m agent level), the dense reference evaluated
      in chunks whose dense tiles fit one wave: bit-identical
   4. persistent social-force rollout kernel vs the per-step route: bit-identical
   5. fused NN step (piml_nn_step_f32) vs state_features -> pinnsf_forward -> integrate_step, and the rollout loop with the
      fused step forced vs the per-stage loop: random scenes / sizes / k / angles / thresholds, absent agents: bit-identical
   6. tensor-core forwards vs the FP32-pipe forward: random rows / topk / zero patterns: 1e-5 of the summed operands
Prints one line per family; exits non-zero on the first disagreement."""
import argparse, os, sys, time
import numpy as np
import torch
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import piml_b200 as P
from piml_b200 import _lib as L, models as M
from tests.golden_args import base_args

ap = argparse.ArgumentParser(); ap.add_argument("--seconds", type=float, default=60); ap.add_argument("--seed", type=int, default=0)
a = ap.parse_args()
rng = np.random.default_rng(a.seed)
dev = torch.device("cuda")
cu = lambda x, dt=torch.float32: torch.as_tensor(np.asarray(x), dtype=dt).to(dev)
budget = a.seconds / 6


def crowd(N, rho):
    side = np.sqrt(N / rho)
    p = (rng.random((N, 2)) * side).astype(np.float32)
    d = (rng.random((N, 2)) * side).astype(np.float32)
    v = rng.normal(0, 1, (N, 2)).astype(np.float32)
    v[rng.random(N) < 0.05] = 0
    return p, v, d, side


def fuzz_mlapm():
    t0, n, worst = time.time(), 0, 0.0
    while time.time() - t0 < budget:
        N = int(rng.integers(2, 40000)); ver = "GC" if rng.random() < 0.8 else "raw"
        p, v, d, _ = crowd(N, float(rng.choice([0.1, 0.5, 2.0])))
        ds = (1.34 + 0.3 * rng.normal(0, 1, (N, 1))).astype(np.float32)
        model = P.MLAPM(version=ver, tau=0.5, A=7.55, B=-3.0, C=0.2, D=-0.3, theta=56)
        out = {}
        for algo in (2, 1):
            L.check(L.load().piml_set_mlapm_algorithm(algo), "algo")
            out[algo] = model.step(cu(p), cu(v), cu(ds), cu(d), 0.08).cpu().numpy()
        L.load().piml_set_mlapm_algorithm(0)
        num = np.linalg.norm(out[2].astype(np.float64) - out[1], axis=-1)
        den = np.maximum(np.maximum(np.linalg.norm(out[1], axis=-1), np.linalg.norm(v, axis=-1)), 1e-6)
        e = float((num / den).max()); worst = max(worst, e); n += 1
        assert np.isfinite(out[2]).all() and e < 1e-5, ("mlapm", N, ver, e)
    print(f"mlapm symmetric vs ordered: {n} crowds, worst operand-relative difference {worst:.2e}")


def fuzz_features():
    t0, n = time.time(), 0
    ped = P.Pedestrians()
    while time.time() - t0 < budget:
        N = int(rng.integers(1, 6000)); Mo = int(rng.integers(0, 1500))
        kp, ko = int(rng.integers(1, 12)), int(rng.integers(1, 16))
        ang_p, ang_o = float(rng.choice([60, 90, 100, 150])), float(rng.choice([60, 90, 120]))
        thr_p, thr_o = float(rng.choice([1.0, 4.0, 7.5])), float(rng.choice([2.0, 4.0]))
        p, v, d, side = crowd(N, float(rng.choice([0.2, 0.5, 3.0])))
        p[rng.random(N) < 0.1] = np.nan
        acc = rng.normal(0, 1, (N, 2)).astype(np.float32); acc[rng.random(N) < 0.05] = np.nan
        obs = (rng.random((Mo, 2)) * side).astype(np.float32)
        res = {}
        for algo in (1, 2):
            L.check(L.load().piml_set_feature_algorithm(algo), "algo")
            vv, aa = cu(v[None]), cu(acc[None])
            res[algo] = ped.get_relative_features(cu(p[None]), vv, aa, cu(d[None]), cu(obs), kp, ang_p, thr_p, ko, ang_o, thr_o) + (vv, aa)
        L.load().piml_set_feature_algorithm(0)
        for x, y in zip(res[1], res[2]):
            assert torch.equal(x.view(torch.int32), y.view(torch.int32)), ("features", N, Mo, kp, ko, ang_p, thr_p)
        n += 1
    print(f"cell-list vs all-pairs features: {n} scenes, bit-identical")


def fuzz_tc():
    from tests.util import tc_forward_in_dense_chunks
    t0, n = time.time(), 0
    sms = torch.cuda.get_device_properties(dev).multi_processor_count
    nets = {}
    for kind in ("pinnsf_bm", "pinnsf_m"):
        torch.manual_seed(1)
        net = M.CLASSES[kind](base_args(model=kind, dataset_name="gc1560")).to(dev).eval()
        nets[kind] = (net, M.pack_device(net.state_dict(), net.spec, dev), M.pack_device_tc(net.state_dict(), net.spec, dev))
    while time.time() - t0 < budget:
        kind = "pinnsf_bm" if rng.random() < 0.5 else "pinnsf_m"
        net, packed, ptc = nets[kind]
        R = int(rng.integers(3500, 30000)); pz = float(rng.random())
        g = torch.Generator().manual_seed(int(rng.integers(1 << 30)))
        ped = torch.randn(R, 6, 6, generator=g); obs = torch.randn(R, 10, 6, generator=g)
        ped[torch.rand(R, 6, generator=g) < pz] = 0; obs[torch.rand(R, 10, generator=g) < pz] = 0
        ped[torch.rand(R, generator=g) < pz] = 0; obs[torch.rand(R, generator=g) < 0.9] = 0
        slf = torch.randn(R, 7, generator=g)
        ped, obs, slf = ped.to(dev), obs.to(dev), slf.to(dev)
        compact = M.pinnsf_forward(net.spec, packed, ped, obs, slf, need_msgs=False, packed_tc=ptc)[0]
        dense = tc_forward_in_dense_chunks(net.spec, packed, ptc, ped, obs, slf, sms)[0]
        assert torch.equal(compact, dense), ("tc compact", kind, R, pz)
        n += 1
    print(f"tensor-core forward compact vs dense: {n} batches, bit-identical")


def fuzz_sfm_rollout():
    from piml_b200.rollout import rollout_scenes, state_features
    import argparse as ap2
    t0, n = time.time(), 0
    spec = P.SocialForce("gc1560").spec
    rargs = ap2.Namespace(time_unit=0.08, topk_ped=6, sight_angle_ped=90, dist_threshold_ped=4, topk_obs=10,
                          sight_angle_obs=90, dist_threshold_obs=4)
    while time.time() - t0 < budget:
        S, T, Ns, Mo = int(rng.integers(1, 9)), int(rng.integers(5, 60)), int(rng.integers(2, 250)), int(rng.integers(1, 300))
        g = torch.Generator().manual_seed(int(rng.integers(1 << 30)))
        side = float(np.sqrt(Ns / 0.3)) + 2
        ob = (torch.rand(Mo, 2, generator=g) * side).to(dev)
        P0 = (torch.rand(S, T, Ns, 2, generator=g) * side).to(dev)
        absent = torch.rand(S, 1, Ns, generator=g) < 0.3
        P0[absent.expand(S, T, Ns).to(dev)] = float('nan')
        entry = (torch.rand(S, T, Ns, generator=g) < 0.02).float().to(dev)
        scene = {"position": P0, "velocity": (torch.randn(S, T, Ns, 2, generator=g) * 0.8).to(dev),
                 "acceleration": (torch.randn(S, T, Ns, 2, generator=g) * 0.2).to(dev),
                 "destination": (torch.rand(S, T, Ns, 2, generator=g) * side).to(dev),
                 "dest_idx": torch.zeros(S, T, Ns, dtype=torch.int64, device=dev),
                 "waypoints": (torch.rand(S, 2, Ns, 2, generator=g) * side).to(dev),
                 "dest_num": torch.full((S, Ns), 2, dtype=torch.int64, device=dev), "obstacles": ob,
                 "mask_p": torch.ones(S, T, Ns, device=dev), "mask_p_pred": 1 - entry,
                 "desired_speed": (1.0 + torch.rand(S, Ns, generator=g)).to(dev)}
        v0 = scene["velocity"][:, 0].contiguous()
        f0 = state_features(P0[:, 0].contiguous(), v0, scene["acceleration"][:, 0].contiguous(),
                            scene["destination"][:, 0].contiguous(), ob, v0.clone(), scene["desired_speed"], 6, 90, 4, 10, 90, 4)
        scene["ped_features0"], scene["obs_features0"], scene["self_features0"] = f0
        outs = {}
        for mode in ("1", "0"):
            os.environ["PIML_SFM_PERSISTENT"] = mode
            outs[mode] = [x.clone() for x in rollout_scenes(spec, None, rargs, scene, 0, T)]
        os.environ.pop("PIML_SFM_PERSISTENT", None)
        for x, y in zip(outs["1"], outs["0"]):
            assert torch.equal(x.view(torch.int32), y.view(torch.int32)), ("sfm rollout", S, T, Ns, Mo)
        n += 1
    print(f"persistent social-force rollout vs per-step route: {n} scene batches, bit-identical")


def fuzz_nn_step():
    from piml_b200.rollout import NNStep, integrate_step, rollout_scenes, state_features
    import argparse as ap2
    t0, n, nr = time.time(), 0, 0
    torch.manual_seed(1)
    net = M.CLASSES["pinnsf_bm"](base_args(model="pinnsf_bm", dataset_name="gc1560")).to(dev).eval()
    packed, ptc = M.pack_device(net.state_dict(), net.spec, dev), M.pack_device_tc(net.state_dict(), net.spec, dev)
    while time.time() - t0 < budget:
        g = torch.Generator().manual_seed(int(rng.integers(1 << 30)))
        if n % 4 == 3:                         # whole rollouts: fused loop forced vs per-stage loop
            S, T, Ns, Mo = int(rng.integers(1, 6)), int(rng.integers(5, 40)), int(rng.integers(12, 200)), int(rng.integers(10, 200))
            side = float(np.sqrt(Ns / 0.3)) + 2
            ob = (torch.rand(Mo, 2, generator=g) * side).to(dev)
            P0 = (torch.rand(S, T, Ns, 2, generator=g) * side).to(dev)
            P0[(torch.rand(S, 1, Ns, generator=g) < 0.3).expand(S, T, Ns).to(dev)] = float('nan')
            entry = (torch.rand(S, T, Ns, generator=g) < 0.02).float().to(dev)
            scene = {"position": P0, "velocity": (torch.randn(S, T, Ns, 2, generator=g) * 0.8).to(dev),
                     "acceleration": (torch.randn(S, T, Ns, 2, generator=g) * 0.2).to(dev),
                     "destination": (torch.rand(S, T, Ns, 2, generator=g) * side).to(dev),
                     "dest_idx": torch.zeros(S, T, Ns, dtype=torch.int64, device=dev),
                     "waypoints": (torch.rand(S, 2, Ns, 2, generator=g) * side).to(dev),
                     "dest_num": torch.full((S, Ns), 2, dtype=torch.int64, device=dev), "obstacles": ob,
                     "mask_p": torch.ones(S, T, Ns, device=dev), "mask_p_pred": 1 - entry,
                     "desired_speed": (1.0 + torch.rand(S, Ns, generator=g)).to(dev)}
            v0 = scene["velocity"][:, 0].contiguous()
            f0 = state_features(P0[:, 0].contiguous(), v0, scene["acceleration"][:, 0].contiguous(),
                                scene["destination"][:, 0].contiguous(), ob, v0.clone(), scene["desired_speed"], 6, 90, 4, 10, 90, 4)
            scene["ped_features0"], scene["obs_features0"], scene["self_features0"] = f0
            rargs = ap2.Namespace(time_unit=0.08, topk_ped=6, sight_angle_ped=90, dist_threshold_ped=4, topk_obs=10,
                                  sight_angle_obs=90, dist_threshold_obs=4)
            outs = {}
            for mode in ("1", "0"):
                os.environ["PIML_ROLLOUT_FUSED"] = mode
                outs[mode] = [x.clone() for x in rollout_scenes(net.spec, packed, rargs, scene, 0, T, packed_tc=ptc)]
            os.environ.pop("PIML_ROLLOUT_FUSED", None)
            for x, y in zip(outs["1"], outs["0"]):
                assert torch.equal(x.view(torch.int32), y.view(torch.int32)), ("fused rollout", S, T, Ns, Mo)
            nr += 1
        else:
            S = int(rng.choice([1, 1, 2, 5])); N = int(rng.integers(7, 20000 // S)); Mo = int(rng.integers(11, 1500))
            kp, ko = int(rng.integers(1, 7)), int(rng.integers(1, 11))
            ang = int(rng.choice([60, 90, 90, 120, 170])); thr = float(rng.choice([1.5, 4.0, 6.0]))
            side = float(np.sqrt(N / float(rng.choice([0.2, 0.5, 2.0]))))
            p = torch.rand(S, N, 2, generator=g) * side
            p[torch.rand(S, N, generator=g) < 0.1] = float('nan')
            v = torch.randn(S, N, 2, generator=g); v[torch.rand(S, N, generator=g) < 0.05] = 0
            acc = torch.randn(S, N, 2, generator=g) * 0.3
            dest = torch.rand(S, N, 2, generator=g) * side
            ob = torch.rand(*((S, Mo, 2) if rng.random() < 0.3 else (Mo, 2)), generator=g) * side
            ds = 1.0 + torch.rand(S, N, generator=g)
            st = lambda: [x.clone().to(dev) for x in (p, v, acc, dest)] + [torch.zeros(S, N, dtype=torch.int64, device=dev),
                                                                          torch.nan_to_num(v).to(dev)]
            A, B = st(), st()
            dn, wp, dsd, obd = torch.ones(S, N, dtype=torch.int64, device=dev), dest[:, None].to(dev).contiguous(), ds.to(dev), ob.to(dev)
            fa = (kp, ang, thr, ko, ang, thr)
            step = NNStep(net.spec, ptc, *B, dn, wp, dsd, obd, 0.08, *fa)
            for _ in range(2):
                pf, of, sf = state_features(A[0], A[1], A[2], A[3], obd, A[5], dsd, *fa)
                an = M.pinnsf_forward(net.spec, packed, pf.view(S * N, -1, 6), of.view(S * N, -1, 6), sf.view(S * N, 7),
                                      need_msgs=False, packed_tc=ptc)[0].view(S, N, 2)
                integrate_step(A[0], A[1], A[2], an, A[3], A[4], dn, wp, 0.08, True, hist_v=A[5])
                step.step()
            for x, y in zip(A, B):
                assert torch.equal(x.view(torch.int32) if x.dtype == torch.float32 else x,
                                   y.view(torch.int32) if y.dtype == torch.float32 else y), ("fused step", S, N, Mo, kp, ko, ang, thr)
        n += 1
    print(f"fused NN step vs three calls: {n - nr} crowds; fused rollout loop vs per-stage loop: {nr} scene batches; bit-identical")


def fuzz_tc_vs_fp32():
    """6. both tensor-core forwards (dense and compact as the size decides) vs the FP32-pipe kernel: pinnsf_bm on the
    fp16-split kernel and, at width 96, on the 3xTF32 kernel; pinnsf_m on the 3xTF32 kernel.  Random row counts, topk,
    zero-slot patterns, with and without the per-slot messages; 1e-5 of the summed operands."""
    from tests.util import accel_err
    t0, n, worst = time.time(), 0, 0.0
    nets = {}
    for key, kind, width in (("pinnsf_bm", "pinnsf_bm", 128), ("pinnsf_bm_w96", "pinnsf_bm", 96),
                             ("pinnsf_m", "pinnsf_m", 128)):
        torch.manual_seed(2)
        args = base_args(model=kind, dataset_name="gc1560", encoder_hidden_size=width, processor_hidden_size=width)
        net = M.CLASSES[kind](args).to(dev).eval()
        nets[key] = (net, M.pack_device(net.state_dict(), net.spec, dev), M.pack_device_tc(net.state_dict(), net.spec, dev))
    while time.time() - t0 < budget:
        kind = "pinnsf_bm" if rng.random() < 0.6 else "pinnsf_m"
        R = int(rng.integers(1, 9000)); kp = int(rng.integers(1, 9)); ko = int(rng.integers(1, 13)); pz = float(rng.random())
        g = torch.Generator().manual_seed(int(rng.integers(1 << 30)))
        ped = torch.randn(R, kp, 6, generator=g); obs = torch.randn(R, ko, 6, generator=g)
        ped[torch.rand(R, kp, generator=g) < pz] = 0; obs[torch.rand(R, ko, generator=g) < pz] = 0
        slf = torch.randn(R, 7, generator=g)
        ped, obs, slf = ped.to(dev), obs.to(dev), slf.to(dev)
        for key in (("pinnsf_bm", "pinnsf_bm_w96") if kind == "pinnsf_bm" else ("pinnsf_m",)):
            net, packed, ptc = nets[key]
            ref = M.pinnsf_forward(net.spec, packed, ped, obs, slf, need_msgs=True)[0]
            for need in ((False, True) if kind == "pinnsf_bm" else (False,)):
                got = M.pinnsf_forward(net.spec, packed, ped, obs, slf, need_msgs=need, packed_tc=ptc)[0]
                err = accel_err(got.cpu().numpy(), ref.cpu().numpy(), slf.cpu().numpy(), net.spec.tau)
                worst = max(worst, err)
                assert err < 1e-5, ("tc vs fp32", key, R, kp, ko, pz, need, err)
        n += 1
    print(f"tensor-core forwards vs FP32-pipe forward: {n} batches, worst operand-scaled error {worst:.2e}")


fuzz_mlapm(); fuzz_features(); fuzz_tc(); fuzz_sfm_rollout(); fuzz_nn_step(); fuzz_tc_vs_fp32()
print("fuzz ok")
