"""Debug helper: random small crowds through the fused NN step and the three calls; prints the first disagreement in detail."""
import os, sys
import numpy as np
import torch
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import piml_b200 as P
from piml_b200 import _lib as L, models as M
from piml_b200.rollout import NNStep, integrate_step, state_features
from tests.golden_args import base_args

dev = torch.device("cuda")
rng = np.random.default_rng(int(sys.argv[1]) if len(sys.argv) > 1 else 0)
torch.manual_seed(1)
net = M.CLASSES["pinnsf_bm"](base_args(model="pinnsf_bm", dataset_name="gc1560")).to(dev).eval()
packed, ptc = M.pack_device(net.state_dict(), net.spec, dev), M.pack_device_tc(net.state_dict(), net.spec, dev)
bad = 0
for it in range(400):
    g = torch.Generator().manual_seed(int(rng.integers(1 << 30)))
    S = int(rng.choice([1, 1, 2, 5])); N = int(rng.integers(7, 6000 // S)); Mo = int(rng.integers(11, 1500))
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
    kpp, kop = min(kp, N), min(ko, Mo)
    dense = (torch.empty(S, N, kpp, 6, device=dev), torch.empty(S, N, kop, 6, device=dev), torch.empty(S, N, 7, device=dev),
             torch.empty(S, N, 2, device=dev))
    a_out = torch.empty(S, N, 2, device=dev)
    step = NNStep(net.spec, ptc, *B, dn, wp, dsd, obd, 0.08, *fa, a_next=a_out, dense=dense)
    for s_ in range(2):
        pf, of, sf = state_features(A[0], A[1], A[2], A[3], obd, A[5], dsd, *fa)
        an = M.pinnsf_forward(net.spec, packed, pf.view(S * N, -1, 6), of.view(S * N, -1, 6), sf.view(S * N, 7),
                              need_msgs=False, packed_tc=ptc)[0].view(S, N, 2)
        integrate_step(A[0], A[1], A[2], an, A[3], A[4], dn, wp, 0.08, True, hist_v=A[5])
        step.step()
        torch.cuda.synchronize()
        eq = lambda x, y: bool(torch.equal(torch.nan_to_num(x, nan=-7.0), torch.nan_to_num(y, nan=-7.0)))
        names = ["ped_f", "obs_f", "self_f", "a_next"]
        pairs = [(dense[0], pf), (dense[1], of), (dense[2], sf), (a_out, an)]
        msgs = [nm for nm, (x, y) in zip(names, pairs) if not eq(x, y)]
        if msgs:
            d = (torch.nan_to_num(a_out) - torch.nan_to_num(an)).abs()
            print(f"it {it} step {s_}: S={S} N={N} Mo={Mo} kp={kp} ko={ko} ang={ang} thr={thr}: differ: {msgs}; "
                  f"a_next max diff {float(d.max()):.3e} on {int((d > 0).any(-1).sum())} agents", flush=True)
            bad += 1
            break
    if bad >= 6:
        break
print("done, mismatching configs:", bad)
