"""A social-force constants sweep (piml_b200.sfm.sweep) on the synthetic config-2 clip against looping rollout_scenes.

    python scripts/time_sfm_sweep.py [--out DIR]

The clip is tests/golden/rollout_syn_sfm.npz (N = 110 slots, 725 frames from t_start = 25 to T = 750).  The constant
sets are SocialForce('gc1560')'s A_ped, B_ped, A_obs, B_obs, tau, each scaled by a seeded factor in [0.7, 1.3).
Per S in {64, 4096, 65536}: ms per score-only sweep (CUDA events around whole calls, after one warm-up call of the
same shape), set-steps per second (S x 725 / time), the route the library takes (S <= 2 waves of 148 SMs: the
persistent kernel; more: per-step launches), and the peak device memory torch allocated during the call.  For
comparison: rollout_scenes looped over 16 sets, one call per set with SfmSpec(set), and the same 16 sets as one sweep.
GPU name and power limit are read in the same run; the JSON goes to --out.
"""
import argparse
import json
import os
import subprocess
import sys

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

from piml_b200 import sfm  # noqa: E402
from piml_b200.rollout import rollout_scenes  # noqa: E402
from tests.golden_args import base_args  # noqa: E402
from tests.util import golden, group  # noqa: E402

DEFAULT = [8.75, -2.5, 50.0, -5.0, 0.5]


def clip():
    i = group(golden("rollout_syn_sfm"), "in")
    cu = lambda x, dt=torch.float32: torch.as_tensor(np.asarray(x), dtype=dt).cuda()   # noqa: E731
    scene = {k: cu(i[k])[None] for k in ("position", "velocity", "acceleration", "destination", "waypoints",
                                          "mask_p", "mask_p_pred", "desired_speed", "ped_features0", "obs_features0",
                                          "self_features0")}
    scene["dest_idx"] = cu(i["dest_idx"], torch.int64)[None]
    scene["dest_num"] = cu(i["dest_num"], torch.int64)[None]
    scene["obstacles"] = cu(i["obstacles"])
    args = base_args(model="sfm", dataset_name="gc1560", time_unit=float(i["time_unit"]))
    return scene, args, int(i["t_start"]), int(i["num_frames"])


def constant_sets(S, seed=0):
    g = torch.Generator().manual_seed(seed)
    return torch.tensor(DEFAULT) * (0.7 + 0.6 * torch.rand(S, 5, generator=g))


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
    ap.add_argument("--out", default="sfm_sweep_out", help="directory for the JSON summary")
    a = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("time_sfm_sweep.py measures on the GPU; no CUDA device found")
    scene, args, t0, T = clip()
    steps = T - t0
    sms = torch.cuda.get_device_properties(0).multi_processor_count
    res = {"gpu": gpu_info(), "clip": {"N": scene["position"].shape[2], "t_start": t0, "T": T, "steps": steps},
           "sweep": {}}
    for S, reps in ((64, 10), (4096, 3), (65536, 1)):
        prm = constant_sets(S).cuda()
        run = lambda: sfm.sweep(scene, prm, args, t0, T)                               # noqa: E731
        run()
        torch.cuda.synchronize()
        torch.cuda.reset_peak_memory_stats()
        base = torch.cuda.memory_allocated()
        ms = events_ms(run, reps)
        w = {"ms_per_sweep": ms, "set_steps_per_s": S * steps / ms * 1e3,
             "route": "persistent" if S <= 2 * sms else "per_step",
             "peak_bytes_during_sweep": torch.cuda.max_memory_allocated() - base}
        res["sweep"][str(S)] = w
        print(S, json.dumps(w), flush=True)
        del prm
        torch.cuda.empty_cache()
    K = 16
    prm = constant_sets(K, seed=1)
    specs = [sfm.SfmSpec(*r[:4].tolist(), sfm.EPS, float(r[4])) for r in prm]

    def loop():
        for sp in specs:
            rollout_scenes(sp, None, args, scene, t0, T)
    loop_ms = events_ms(loop, 2)
    prm_d = prm.cuda()
    one_ms = events_ms(lambda: sfm.sweep(scene, prm_d, args, t0, T), 5)
    res["rollout_scenes_loop"] = {"sets": K, "ms": loop_ms, "ms_per_set": loop_ms / K,
                                  "set_steps_per_s": K * steps / loop_ms * 1e3, "same_sets_as_one_sweep_ms": one_ms}
    print("loop", json.dumps(res["rollout_scenes_loop"]))
    os.makedirs(a.out, exist_ok=True)
    with open(os.path.join(a.out, "time_sfm_sweep.json"), "w") as f:
        json.dump(res, f, indent=1)
    print(json.dumps(res))


if __name__ == "__main__":
    main()
