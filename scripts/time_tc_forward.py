"""Device time of each route of the tensor-core forward (piml_pinnsf_forward_tc_f32) on bench.py's crowd.

    python scripts/time_tc_forward.py [--agents 100000] [--rounds 5] [--iters 20] [--dump DIR]

The features are state_features of bench.synthetic_crowd (k = 6 / 10, 90 deg, 4 m).  The library picks the kernel
and its mode from the network and the batch; at 10^5 agents the dense tiles exceed one wave, so a call without
messages runs in compact mode and a call with messages in dense mode:
    tc16_compact        pinnsf_bm (widths 128 / 64), no messages     16-bit kernel, slot-row compaction
    tc16_dense          pinnsf_bm, with messages                     16-bit kernel, dense tiles
    tf32_agent_compact  pinnsf_m, no messages                        tf32 kernel, agent compaction
    tf32_kind0_compact  pinnsf_bm at width 96, no messages           tf32 kernel, slot-row compaction
    tf32_kind0_dense    pinnsf_bm at width 96, with messages         tf32 kernel, dense tiles
(the 16-bit kernel takes widths 32, 64 and 128 only, so width 96 runs on the tf32 kernel).  bench.py times only the
first route.  The library entry is called directly, as pinnsf_forward(..., packed_tc=...) calls it: pinnsf_forward
sends a request for messages from pinnsf_bm, which has a collision head, to the FP32-pipe kernel.

Rounds alternate the routes; each call has its own CUDA-event pair, preceded by a 160 MB L2 flush outside it.  Prints
one JSON line with the card, its power limit and min / median / max ms per route; the kernels each route launched are
read from a torch.profiler run after the timing and checked against the route.  --dump DIR writes every route's
outputs as DIR/<route>/<name>.npy (seeded inputs: two builds compare output for output).
"""
import argparse
import json
import os
import statistics
import subprocess
import sys

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

import bench  # noqa: E402
from piml_b200 import _lib as L, models as M  # noqa: E402
from piml_b200.rollout import state_features  # noqa: E402

# route -> (network, messages requested, kernel that must run, compaction kernel that must run or None)
ROUTES = {
    "tc16_compact": ("pinnsf_bm", False, "pinnsf_tc16_kernel", "tc_compact_kernel"),
    "tc16_dense": ("pinnsf_bm", True, "pinnsf_tc16_kernel", None),
    "tf32_agent_compact": ("pinnsf_m", False, "pinnsf_tc_kernel", "tc_compact_agents_kernel"),
    "tf32_kind0_compact": ("pinnsf_bm_w96", False, "pinnsf_tc_kernel", "tc_compact_kernel"),
    "tf32_kind0_dense": ("pinnsf_bm_w96", True, "pinnsf_tc_kernel", None),
}
NETS = {"pinnsf_bm": ("pinnsf_bm", {}), "pinnsf_m": ("pinnsf_m", {}),
        "pinnsf_bm_w96": ("pinnsf_bm", {"encoder_hidden_size": 96, "processor_hidden_size": 96})}


def card(dev):
    q = subprocess.run(["nvidia-smi", "--query-gpu=power.limit,clocks.max.sm", "--format=csv,noheader",
                        "-i", str(dev.index or 0)], capture_output=True, text=True)
    return {"name": torch.cuda.get_device_name(dev), "power_limit_and_max_sm_clock": q.stdout.strip() or None}


def kernel_names(fn):
    with torch.profiler.profile(activities=[torch.profiler.ProfilerActivity.CUDA]) as prof:
        fn()
        torch.cuda.synchronize()
    names = set()
    for e in prof.events():
        if e.device_type == torch.autograd.DeviceType.CUDA:
            n = e.name.split("(")[0].split("<")[0]
            names.add(n.rsplit("::", 1)[-1])
    return sorted(names)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--agents", type=int, default=100000)
    ap.add_argument("--rounds", type=int, default=5)
    ap.add_argument("--iters", type=int, default=20)
    ap.add_argument("--dump", metavar="DIR", help="write each route's outputs as DIR/<route>/<name>.npy")
    a = ap.parse_args()
    if not torch.cuda.is_available():
        sys.exit("time_tc_forward.py needs a CUDA device")
    dev = torch.device("cuda")
    N = a.agents
    p, v, ds, dest, obs = [x.to(dev) for x in bench.synthetic_crowd(N)]
    pf, of, sf = state_features(p[None], v[None], torch.zeros_like(p)[None], dest[None], obs, v[None].clone(),
                                ds.view(1, N), *bench.NN_FEATURE_ARGS)
    kp, ko = bench.NN_FEATURE_ARGS[0], bench.NN_FEATURE_ARGS[3]
    pf, of, sf = pf.view(N, kp, 6), of.view(N, ko, 6), sf.view(N, 7)
    nets = {}
    for key, (kind, over) in NETS.items():
        torch.manual_seed(666)
        net = M.CLASSES[kind](argparse.Namespace(**{**bench.NN_ARGS, "model": kind, **over})).to(dev).eval()
        ptc = M.pack_device_tc(net.state_dict(), net.spec, dev)
        assert ptc is not None, key
        nets[key] = (net.spec, net.spec.desc(), ptc)
    outs = {route: {"acc": torch.empty(N, 2, device=dev)} for route in ROUTES}
    for route, (_, msgs, _, _) in ROUTES.items():
        if msgs:
            outs[route].update(ped_msgs=torch.empty(N, kp, 2, device=dev), obs_msgs=torch.empty(N, ko, 2, device=dev))

    def call(route):
        spec, desc, ptc = nets[ROUTES[route][0]]
        o = outs[route]
        L.check(L.load().piml_pinnsf_forward_tc_f32(
            L.C.byref(desc), L.ptr(ptc), 1, spec.tau, L.ptr(pf), L.ptr(of), L.ptr(sf), N, kp, ko, 0,
            L.ptr(o["acc"]), L.ptr(o.get("ped_msgs")), L.ptr(o.get("obs_msgs")), L.stream_ptr(dev)),
            "piml_pinnsf_forward_tc_f32")

    flush = torch.empty(bench.FLUSH_MB << 20, dtype=torch.uint8, device=dev)
    for route in ROUTES:                                           # warm-up: module load, scratch buffers
        for _ in range(3):
            call(route)
    torch.cuda.synchronize()
    ms = {route: [] for route in ROUTES}
    for _ in range(a.rounds):
        for route in ROUTES:
            pairs = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(a.iters)]
            for e0, e1 in pairs:
                flush.zero_()
                e0.record()
                call(route)
                e1.record()
            torch.cuda.synchronize()
            ms[route] += [e0.elapsed_time(e1) for e0, e1 in pairs]
    report = {"card": card(dev), "agents": N, "rounds": a.rounds, "iters": a.iters, "routes": {}}
    for route, (net, msgs, kernel, compaction) in ROUTES.items():
        names = kernel_names(lambda: call(route))
        assert kernel in names and (compaction in names if compaction else "compact" not in " ".join(names)), \
            (route, names)
        t = ms[route]
        report["routes"][route] = {"network": net, "messages": msgs, "kernels": names, "ms_min": min(t),
                                   "ms_median": statistics.median(t), "ms_max": max(t), "n": len(t)}
    if a.dump:
        for route in ROUTES:
            call(route)
            bench.dump_outputs(os.path.join(a.dump, route), outs[route])
    print(json.dumps(report), flush=True)


if __name__ == "__main__":
    main()
