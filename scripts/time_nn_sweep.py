"""A network sweep (piml_b200.rollout.sweep_networks) on the GC clip against looping rollout_scenes over the same networks.

    python scripts/time_nn_sweep.py [--out DIR]

The clip is tests/golden/rollout_gc_bm.npz (N = 122 slots, 725 frames from t_start = 25 to T = 750).  The networks are
pinnsf_bm with the golden rollout's widths (encoder / processor 128, decoder 64, 16 processor blocks): the golden
weights, each weight scaled by a seeded factor in [0.875, 1.125).  Per S in {1, 16, 64, 256}, after one warm-up call
of every S: ms per score-only sweep (CUDA events around whole calls, packing the S networks included), set-steps per
second (S x 725 / time) and the peak device memory torch allocated during the call; against rollout_scenes called
once per network in a Python loop over the same S networks (their tensor-core vectors packed beforehand, outside the
timed window).  GPU name, power limit and maximum SM clock are read in the same run (read-only nvidia-smi query);
the JSON goes to --out.
"""
import argparse
import copy
import json
import os
import subprocess
import sys

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

from piml_b200 import models as M  # noqa: E402
from piml_b200.rollout import rollout_scenes, sweep_networks  # noqa: E402
from tests.golden_args import base_args  # noqa: E402
from tests.util import golden, group  # noqa: E402


def clip():
    i = group(golden("rollout_gc_bm"), "in")
    cu = lambda x, dt=torch.float32: torch.as_tensor(np.asarray(x), dtype=dt).cuda()   # noqa: E731
    scene = {k: cu(i[k])[None] for k in ("position", "velocity", "acceleration", "destination", "waypoints",
                                          "mask_p", "mask_p_pred", "desired_speed", "ped_features0", "obs_features0",
                                          "self_features0")}
    scene["dest_idx"] = cu(i["dest_idx"], torch.int64)[None]
    scene["dest_num"] = cu(i["dest_num"], torch.int64)[None]
    scene["obstacles"] = cu(i["obstacles"])
    args = base_args(model="pinnsf_bm", dataset_name="gc1560", time_unit=float(i["time_unit"]))
    return scene, args, int(i["t_start"]), int(i["num_frames"])


def networks(S, args):
    gold = M.CLASSES["pinnsf_bm"](args)
    sd = {k[3:]: torch.from_numpy(v) for k, v in group(golden("models"), "pinnsf_bm").items() if k.startswith("sd/")}
    gold.load_state_dict(sd)
    nets = []
    for s in range(S):
        g = torch.Generator().manual_seed(s)
        m = copy.deepcopy(gold)
        m.load_state_dict({k: v * (0.875 + 0.25 * torch.rand(v.shape, generator=g)) for k, v in sd.items()})
        nets.append(m.eval())
    return nets


def events_ms(fn, reps):
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    torch.cuda.synchronize()
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
    ap.add_argument("--out", default="nn_sweep_out", help="directory for the JSON summary")
    a = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("time_nn_sweep.py measures on the GPU; no CUDA device found")
    scene, args, t0, T = clip()
    steps = T - t0
    sizes = ((1, 5), (16, 3), (64, 2), (256, 1))
    nets = networks(max(S for S, _ in sizes), args)
    spec = M.spec_from_module(nets[0])
    res = {"gpu": gpu_info(), "clip": {"N": scene["position"].shape[2], "t_start": t0, "T": T, "steps": steps},
           "sweep": {}}
    for S, _ in sizes:                                          # warm-up of every shape the timed windows use
        sweep_networks(scene, nets[:S], args, t0, T)
    torch.cuda.synchronize()
    packed = [M.pack_device_tc(m.state_dict(), spec) for m in nets]
    rollout_scenes(spec, None, args, scene, t0, T, packed_tc=packed[0])
    for S, reps in sizes:
        torch.cuda.synchronize()
        base = torch.cuda.memory_allocated()
        torch.cuda.reset_peak_memory_stats()
        ms = events_ms(lambda: sweep_networks(scene, nets[:S], args, t0, T), reps)
        peak = torch.cuda.max_memory_allocated() - base

        def loop():
            for p in packed[:S]:
                rollout_scenes(spec, None, args, scene, t0, T, packed_tc=p)
        loop_ms = events_ms(loop, 1)
        w = {"ms_per_sweep": ms, "set_steps_per_s": S * steps / ms * 1e3, "peak_bytes_during_sweep": peak,
             "rollout_scenes_loop_ms": loop_ms, "rollout_scenes_loop_set_steps_per_s": S * steps / loop_ms * 1e3,
             "speedup": loop_ms / ms}
        res["sweep"][str(S)] = w
        print(S, json.dumps(w), flush=True)
    os.makedirs(a.out, exist_ok=True)
    with open(os.path.join(a.out, "time_nn_sweep.json"), "w") as f:
        json.dump(res, f, indent=1)
    print(json.dumps(res))


if __name__ == "__main__":
    main()
