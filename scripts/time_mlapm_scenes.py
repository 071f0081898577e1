"""Many independent MLAPM scenes per launch (MLAPM.advance_scenes) against MLAPM.advance looped over scenes.

    python scripts/time_mlapm_scenes.py [--reps 50] [--out DIR]

Seeded workloads, every shape warmed up first:
  circle   the main_mlapm.py scene (7 agents on a 10 m circle, v ~ U[0,1)^2, GC constants), 65 536 seeds
  gc122    4096 scenes of 122 slots from bench.synthetic_crowd's recipe (rho = 0.5), 10-30 % of the slots inactive
  sweep    one 2000-agent crowd x 256 constant sets (params (256, 6))
  split    8 scenes x 8192 agents (each scene's rows split over 32 CTAs)
Per workload: ms per step of advance_scenes on the initial state (CUDA events around `reps` calls), agent-steps/s,
evaluated ordered pairs/s (sum over scenes of active^2, self pairs included, as the kernel evaluates them), the share
of launched lanes that own an active row, and MLAPM.advance looped over the first 256 compacted scenes in the same
run (an extrapolation to all S scenes is labelled as such).  The circle also runs rollout_scenes for 200 steps.
For scale: the dense ordered-pair kernel (piml_set_mlapm_algorithm(1)) at N = 8192.  GPU name and power limit are read
in the same run; the JSON goes to --out.
"""
import argparse
import json
import math
import os
import subprocess
import sys

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

import bench  # noqa: E402
import piml_b200 as P  # noqa: E402
from piml_b200 import _lib as L  # noqa: E402
from piml_b200.mlapm import rollout_scenes  # noqa: E402

GC_KW = dict(version='GC', tau=0.5, A=7.55, B=-3.00, C=0.2, D=-0.3, theta=56)
DT, RADIUS = 0.08, 0.3


def lanes(S, N):
    """Lanes the kernel launches for S scenes of N slots (msc_shape in csrc/mlapm.cu)."""
    nchunk = (N + 255) // 256
    if N <= 32:
        C = 1 << (N - 1).bit_length()
    else:
        C = (-(-N // nchunk) + 31) // 32 * 32
    k = 256 // C if nchunk == 1 else 1
    return -(-S // k) * nchunk * k * C


def circle(S, seed=0):
    n = 7
    th = torch.linspace(0, 2 * math.pi * (1 - 1. / n), n)
    p = torch.stack([10 * th.cos(), 10 * th.sin()], -1).expand(S, n, 2).contiguous()
    g = torch.Generator().manual_seed(seed)
    v = torch.rand(S, n, 2, generator=g)
    ds = torch.full((S, n, 2), 1.5)
    return p, v, ds, -p, torch.ones(S, n, dtype=torch.bool), None


def gc122(S=4096, N=122):
    ps, vs, dss, ds_ = [], [], [], []
    for s in range(S):
        p, v, ds, d, _ = bench.synthetic_crowd(N, M=0, seed=1000 + s)
        ps.append(p); vs.append(v); dss.append(ds); ds_.append(d)
    g = torch.Generator().manual_seed(7)
    frac = 0.1 + 0.2 * torch.rand(S, 1, generator=g)
    act = torch.rand(S, N, generator=g) >= frac
    return torch.stack(ps), torch.stack(vs), torch.stack(dss), torch.stack(ds_), act, None


def sweep(S=256, N=2000):
    p, v, ds, d, _ = bench.synthetic_crowd(N, M=0, seed=5)
    g = torch.Generator().manual_seed(9)
    base = torch.tensor([GC_KW[k] for k in ("tau", "A", "B", "C", "D", "theta")])
    prm = base * (0.7 + 0.6 * torch.rand(S, 6, generator=g))
    rep = [x.expand(S, *x.shape).contiguous() for x in (p, v, ds, d)]
    return (*rep, torch.ones(S, N, dtype=torch.bool), prm)


def split(S=8, N=8192):
    xs = [bench.synthetic_crowd(N, M=0, seed=300 + s)[:4] for s in range(S)]
    return (*[torch.stack([x[i] for x in xs]) for i in range(4)], torch.ones(S, N, dtype=torch.bool), None)


def events_ms(fn, reps):
    fn()
    torch.cuda.synchronize()
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record()
    for _ in range(reps):
        fn()
    b.record()
    torch.cuda.synchronize()
    return a.elapsed_time(b) / reps


def gpu_info():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True)
    return q.stdout.strip().splitlines()[0] if q.returncode == 0 and q.stdout.strip() else torch.cuda.get_device_name()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=50)
    ap.add_argument("--out", default="mlapm_scenes_out", help="directory for the JSON summary")
    a = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("time_mlapm_scenes.py measures on the GPU; no CUDA device found")
    L.check(L.load().piml_set_mlapm_algorithm(0), "piml_set_mlapm_algorithm")
    model = P.MLAPM(**GC_KW)
    res = {"gpu": gpu_info(), "workloads": {}}
    for name, make in (("circle", lambda: circle(65536)), ("gc122", gc122), ("sweep", sweep), ("split", split)):
        p, v, ds, d, act, prm = [None if x is None else x.cuda() for x in make()]
        S, N = act.shape
        n_act = act.sum(1).double()
        pairs, agents = float((n_act ** 2).sum()), float(n_act.sum())
        step = lambda: model.advance_scenes(p, v, ds, d, act, DT, RADIUS, prm)   # noqa: E731
        ms = min(events_ms(step, a.reps) for _ in range(3))
        # MLAPM.advance looped over the first 256 scenes, each compacted to its active agents (as rollout does)
        K = min(S, 256)
        comp = [(p[s][act[s]], v[s][act[s]], ds[s][act[s]], d[s][act[s]]) for s in range(K)]
        models = [model if prm is None else P.MLAPM(**dict(zip(("version", "tau", "A", "B", "C", "D", "theta"),
                                                               ["GC"] + prm[s].tolist()))) for s in range(K)]

        def loop():
            for s in range(K):
                models[s].advance(*comp[s], DT, RADIUS)
        loop_ms = min(events_ms(loop, 3) for _ in range(2))
        w = {"S": S, "N": N, "active_agents": agents, "ms_per_step": ms, "agent_steps_per_s": agents / ms * 1e3,
             "pairs_per_step": pairs, "pairs_per_s": pairs / ms * 1e3, "row_lane_share": agents / lanes(S, N),
             "advance_loop_first_scenes": K, "advance_loop_ms": loop_ms,
             "advance_loop_ms_extrapolated_to_S": loop_ms * S / K,
             "speedup_vs_advance_loop_extrapolated": loop_ms * S / K / ms}
        if name == "circle":
            rollout_scenes(model, p, v, ds, d, 2, DT, RADIUS)
            torch.cuda.synchronize()
            w["rollout_200_steps_ms"] = events_ms(lambda: rollout_scenes(model, p, v, ds, d, 200, DT, RADIUS), 1)
        res["workloads"][name] = w
        print(name, json.dumps(w), flush=True)
        del p, v, ds, d, act, prm, comp
        torch.cuda.empty_cache()
    # the dense ordered-pair kernel on one 8192-agent crowd, for scale
    p, v, ds, d, _ = [x.cuda() for x in bench.synthetic_crowd(8192, M=0, seed=1)]
    L.check(L.load().piml_set_mlapm_algorithm(1), "piml_set_mlapm_algorithm")
    try:
        ms = min(events_ms(lambda: model.advance(p, v, ds, d, DT, RADIUS), a.reps) for _ in range(3))
    finally:
        L.check(L.load().piml_set_mlapm_algorithm(0), "piml_set_mlapm_algorithm")
    res["dense_ordered_N8192"] = {"ms_per_step": ms, "pairs_per_s": 8192.0 ** 2 / ms * 1e3}
    print("dense_ordered_N8192", json.dumps(res["dense_ordered_N8192"]))
    os.makedirs(a.out, exist_ok=True)
    with open(os.path.join(a.out, "time_mlapm_scenes.json"), "w") as f:
        json.dump(res, f, indent=1)
    print(json.dumps(res))


if __name__ == "__main__":
    main()
