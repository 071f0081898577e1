"""Culled against dense symmetric MLAPM steps on bench.py's crowd (one GPU).

    python scripts/time_mlapm_cull.py [--sizes 100000,1000000] [--rounds 5] [--steps 20] [--out DIR]

Per size: culled (algorithm 2) and dense (algorithm 3) steps alternate in one process, `rounds` x `steps` each, with
a 160 MB L2 flush before every step outside its CUDA-event pair; min / median / max ms per step.  The dense arm at
N >= 10^6 runs one step per round (about 0.7 s each).  Then the work-list length, the evaluated pairs and their rate
against the dense kernel's, a torch.profiler run for the per-kernel split (written under --out), and 50 consecutive
culled steps on the moving crowd.
"""
import argparse
import ctypes as C
import json
import os
import statistics
import sys

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

import bench  # noqa: E402
import piml_b200 as P  # noqa: E402
from piml_b200 import _lib as L  # noqa: E402

STAGE_PAIRS = 512 * 128          # (row block, column stage) item


def algo(a):
    L.check(L.load().piml_set_mlapm_algorithm(a), "piml_set_mlapm_algorithm")


def groups(name):
    if "cull_keys" in name or "RadixSort" in name:
        return "keys + sort"
    if "prep_cull" in name:
        return "prep + boxes"
    if "Select" in name or "Compact" in name or "ScanTileState" in name or "InitKernel" in name:
        return "list build"
    if "sym_list" in name:
        return "pair kernel (culled)"
    if "mlapm_sym_kernel" in name:
        return "pair kernel (dense)"
    if "prep_sym" in name:
        return "prep (dense)"
    if "finalize" in name:
        return "finalize (both arms)"
    return None


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--sizes", default="100000,1000000")
    ap.add_argument("--rounds", type=int, default=5)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--out", default="mlapm_cull_out", help="directory for the JSON summary and the traces")
    a = ap.parse_args()
    if not torch.cuda.is_available():
        sys.exit("time_mlapm_cull.py needs a CUDA device")
    dev = torch.device("cuda")
    os.makedirs(a.out, exist_ok=True)
    flush = torch.empty(bench.FLUSH_MB << 20, dtype=torch.uint8, device=dev)
    report = {"device": torch.cuda.get_device_name(dev)}
    for N in [int(x) for x in a.sizes.split(",")]:
        p, v, ds, dest, _ = [x.to(dev) for x in bench.synthetic_crowd(N)]
        model = P.MLAPM(**bench.MLAPM_KW)

        def run(al, steps, state=None):
            algo(al)
            try:
                times = []
                for _ in range(steps):
                    pp, vv = state if state else (p, v)
                    flush.zero_()
                    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                    e0.record()
                    act, pn, _ = model.advance(pp, vv, ds, dest, bench.DT, bench.RADIUS)
                    e1.record()
                    e1.synchronize()
                    times.append(e0.elapsed_time(e1))
                    if state is not None:
                        state[0], state[1] = pn, act
                return times
            finally:
                algo(0)

        dense_steps = a.steps if N < 1000000 else 1
        run(2, 2), run(3, 1)                                         # warm-up: module load, CUB, workspace
        ms = {"culled": [], "dense": []}
        for _ in range(a.rounds):
            ms["culled"] += run(2, a.steps)
            ms["dense"] += run(3, dense_steps)
        res = {k: {"min": min(t), "median": statistics.median(t), "max": max(t), "n": len(t)} for k, t in ms.items()}
        res["speedup_median"] = res["dense"]["median"] / res["culled"]["median"]
        # work list of the culled step on the bench crowd
        run(2, 1)
        items = C.c_int64()
        L.check(L.load().piml_mlapm_cull_items(L.ptr(model._ws), N, C.byref(items)), "piml_mlapm_cull_items")
        T = (N + 511) // 512
        cand = T * (T // 2 + 1) * 4
        ordered = items.value * 2 * STAGE_PAIRS - 4 * T * STAGE_PAIRS   # diagonal items: one direction
        res.update({"items": items.value, "candidates": cand, "item_share": items.value / cand,
                    "unordered_pairs_evaluated": items.value * STAGE_PAIRS,
                    "ordered_pair_equivalents": ordered})
        # per-kernel split (a separate, traced run)
        prof_steps = 5
        with torch.profiler.profile(activities=[torch.profiler.ProfilerActivity.CUDA]) as prof:
            run(2, prof_steps)
            run(3, 1 if N >= 1000000 else prof_steps)
        split = {}
        for ev in prof.key_averages():
            g = groups(ev.key)
            if g:
                d = split.setdefault(g, {"us_total": 0.0, "calls": 0, "kernels": []})
                d["us_total"] += ev.device_time_total if hasattr(ev, "device_time_total") else ev.cuda_time_total
                d["calls"] += ev.count
                d["kernels"].append(ev.key[:80])
        dn = 1 if N >= 1000000 else prof_steps
        for g, d in split.items():
            d["us_per_step"] = d["us_total"] / (dn if "dense" in g else prof_steps)
        res["split"] = split
        t_pair = split.get("pair kernel (culled)", {}).get("us_per_step")
        t_dense = split.get("pair kernel (dense)", {}).get("us_per_step")
        if t_pair and t_dense:
            res["ordered_pairs_per_s_culled"] = ordered / (t_pair * 1e-6)
            res["ordered_pairs_per_s_dense"] = float(N) * N / (t_dense * 1e-6)
            res["rate_ratio"] = res["ordered_pairs_per_s_culled"] / res["ordered_pairs_per_s_dense"]
        prof.export_chrome_trace(os.path.join(a.out, f"cull_N{N}.pt.trace.json"))
        # 50 consecutive culled steps on the moving crowd
        run_ms = run(2, 50, state=[p.clone(), v.clone()])
        res["moving_50"] = {"first10_median": statistics.median(run_ms[:10]),
                            "last10_median": statistics.median(run_ms[-10:]), "max": max(run_ms)}
        report[f"N{N}"] = res
        print(json.dumps({f"N{N}": res}), flush=True)
        del model
        torch.cuda.empty_cache()
    with open(os.path.join(a.out, "time_mlapm_cull.json"), "w") as f:
        json.dump(report, f, indent=1)


if __name__ == "__main__":
    main()
