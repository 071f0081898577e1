#!/usr/bin/env python
"""bench.py -- agent-steps/s of the PIML crowd-rollout hot path on B200 (contract in the task statement, tier (4)).

Headline workload (BASELINE.json configs[3], the one the north-star target is quoted on): the discovered MLAPM
model's rollout loop (reference src/main_mlapm.py:18-36 -> src/models/mlapm.py:10-58) on a synthetic crowd of
N = 100 000 agents (SURVEY.md 8d recipe, rho = 0.5 ped/m^2).  A "step" is one iteration of that loop: dense all-pairs
force (N^2 ordered pairs), destination term, v' = v + F dt, p' = p + v' dt, arrival test.

  value     device-resident agent-steps/s over all ranks (N agents * K steps / max-over-ranks device time)
  e2e       the same step through the public host-buffer API (piml_b200.MLAPM.advance with pinned CPU tensors),
            H2D + kernels + D2H inside the timed region
  roofline  the all-pairs kernel against the FP32 FMA peak measured live by an FMA-chain probe (the kernel is
            FP32/MUFU-pipe bound, DRAM traffic is O(N)); algorithmic work = 51 FLOP per ordered pair (SURVEY 8d)
  cpu_baseline  the oracle's C port of MLAPM.step timed on the host cores on a bounded row sample (rank 0, N=1 only)

  parity    the step the bench times, checked in the same run against oracle rows (action AND force level)
  reference_pytorch  the UNMODIFIED reference (baseline/_ref, PyTorch CPU) timed on the host cores at the sizes it can run

Multi-GPU (--gpus N under torchrun): the crowd is agent-sharded.  Default exchange "push": the symmetric evaluation
splits the unordered block pairs over the ranks, column-direction shares and the new state are stored into the owners'
buffers over NVLink peer memory by the pair / finalize kernels (no collective); "--exchange nccl": ordered rows + one NCCL
all-gather per step.  Strong scaling at fixed N.  --impl reference times the reference's CPU algorithm (the oracle's
C/OpenMP port of MLAPM.step on all host threads: the Python reference cannot run N = 100k).
"""
import argparse
import json
import math
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

METRIC = "agent_steps_per_sec"
UNIT = "agent-steps/s"
FLOP_PER_PAIR = 51.0          # SURVEY.md 8d, MLAPM-GC per ordered pair
MLAPM_KW = dict(version='GC', tau=0.5, A=7.55, B=-3.00, C=0.2, D=-0.3, theta=56)     # main_mlapm.py:16
DT, RADIUS = 0.08, 0.3
FLUSH_MB = 160                 # L2 is 126 MB
MLAPM_DRAM_BYTES_PER_LAUNCH = 5629952 + 1383680     # ordered-pair kernel: ncu --set full, N = 100k (profiles/r01b_...)
MLAPM_SYM_DRAM_BYTES_PER_LAUNCH = 6473472 + 27649792   # symmetric kernel (profiles/r02i_ncu_mlapm_sym_kernel.txt)


def synthetic_crowd(N, M=2000, seed=666, rho=0.5):
    """SURVEY.md 8d config 4: p ~ U[0,L)^2, L = sqrt(N/rho); v = 1.34 e_dest U(0.5,1) + N(0,0.1^2);
    desired_speed ~ max(0.7, 1.34 + sqrt(0.26) N(0,1)); destination ~ U[0,L)^2; M obstacle points on rings."""
    import torch
    g = torch.Generator().manual_seed(seed)
    L = math.sqrt(N / rho)
    p = torch.rand(N, 2, generator=g) * L
    dest = torch.rand(N, 2, generator=g) * L
    e = dest - p
    e = e / e.norm(dim=-1, keepdim=True).clamp_min(1e-6)
    v = 1.34 * e * (0.5 + 0.5 * torch.rand(N, 1, generator=g)) + 0.1 * torch.randn(N, 2, generator=g)
    ds = (1.34 + math.sqrt(0.26) * torch.randn(N, 1, generator=g)).clamp_min(0.7)
    rings = max(M // 200, 1)
    per = max(M // rings, 1)
    ang = torch.arange(per) * (2 * math.pi / per)
    obs = torch.cat([torch.stack([(r % 5 + 0.5) * L / 5 + 2.75 * ang.cos(),
                                  (r // 5 + 0.5) * L / 2 + 2.75 * ang.sin()], -1) for r in range(rings)], 0)[:M]
    return p.float(), v.float(), ds.float(), dest.float(), obs.float()


DUMP_BYTES = 64 << 20
NPY_HEADER_BYTES = 4096        # per file; a .npy header is 128 bytes for these shapes


def dump_outputs(out_dir, arrays):
    """Write arrays that share their leading (agent) dimension as <out_dir>/<name>.npy in float32, for comparing two
    builds output for output.  Above 64 MB on disk in all, every array keeps the same seeded sample of agents, whose
    indices go to rows.npy (float64)."""
    import numpy as np
    host = {k: v.detach().float().cpu().numpy() for k, v in arrays.items()}
    n = len(next(iter(host.values())))
    total = sum(x.nbytes for x in host.values())
    if total + len(host) * NPY_HEADER_BYTES > DUMP_BYTES:
        budget = DUMP_BYTES - (len(host) + 1) * NPY_HEADER_BYTES
        rows = np.sort(np.random.default_rng(0).choice(n, budget // (total // n + 8), replace=False))
        host = {k: x[rows] for k, x in host.items()}
        host["rows"] = rows.astype(np.float64)
    os.makedirs(out_dir, exist_ok=True)
    for k, x in host.items():
        np.save(os.path.join(out_dir, k + ".npy"), x)


class ClockSampler(threading.Thread):
    """nvidia-smi clocks / throttle reasons sampled DURING the timed region (B200_PROFILING.md recipe)."""
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index):
        super().__init__(daemon=True)
        self.gpu, self.rows, self.proc = gpu_index, [], None

    def run(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits",
                                          "-i", str(self.gpu), "-lms", "100"], stdout=subprocess.PIPE, text=True)
            for line in self.proc.stdout:
                self.rows.append([x.strip() for x in line.split(",")])
        except Exception:
            pass

    def stop(self):
        if self.proc:
            self.proc.terminate()
        self.join(timeout=2)

    def summary(self):
        sm, mx, reasons = [], [], set()
        for r in self.rows:
            try:
                sm.append(float(r[1])); mx.append(float(r[2]))
            except (ValueError, IndexError):
                continue
            for name, val in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), r[5:9]):
                if val.lower().startswith("active"):
                    reasons.add(name)
        if not sm:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"], "samples": 0}
        sm.sort()
        return {"sm_mhz": sm[len(sm) // 2], "sm_max_mhz": max(mx), "reasons": sorted(reasons), "samples": len(sm)}


def cpu_baseline(N, seconds=12.0, threads=None):
    """Oracle C port of MLAPM.step (mlapm.py:10-58) on the host cores, rows [0,R) against all N columns."""
    from oracle import oracle as O
    import numpy as np
    O.set_num_threads(threads or len(os.sched_getaffinity(0)))
    cores = O.num_threads()
    p, v, ds, dest, _ = [x.numpy() for x in synthetic_crowd(N)]
    probe = max(64, cores * 16)
    O.mlapm_step(p, v, ds, dest, DT, "GC", rows=(0, probe))       # spin up the OpenMP team
    t0 = time.perf_counter()
    O.mlapm_step(p, v, ds, dest, DT, "GC", rows=(0, probe))
    rate = probe / max(time.perf_counter() - t0, 1e-6)            # rows/s
    R = int(min(N, max(probe, rate * seconds)))
    t0 = time.perf_counter()
    out = O.mlapm_step(p, v, ds, dest, DT, "GC", rows=(0, R))
    dt = time.perf_counter() - t0
    assert np.isfinite(out).all()
    return {"value": R / dt, "unit": UNIT, "cores": cores, "kind": "port",
            "sample": f"oracle C port (OpenMP, {cores} threads) of MLAPM.step: rows [0,{R}) x all {N} columns, "
                      f"{R * N / dt / 1e6:.1f} Mpairs/s, {dt:.1f} s"}, out


BIG_DT = float(2 ** 20)       # F dt exact, v below the rounding of F dt: F = (action - v) / 2^20 to 6e-8


def parity_block(torch, dev, N, model, oracle_rows=None):
    """The timed step against the oracle, in the same run: action = v + F dt on the rows the cpu_baseline leg computed
    anyway, and the FORCE (recovered through dt = 2^20) on row ranges spread over the symmetric kernel's block
    schedule.  strict = ||dF|| / ||F|| per agent; kappa = S / ||F|| with S = |dest term| + sum |pair term| (fp32
    rounding of a row sum is relative to S; tests/test_gpu_parity_sizes.py states the enforced gate)."""
    from oracle import oracle as O
    import numpy as np
    p, v, ds, dest, _ = synthetic_crowd(N)
    pn, vn, dsn, dn = [x.numpy() for x in (p, v, ds, dest)]
    pc, vc, dsc, dc = [x.to(dev) for x in (p, v, ds, dest)]
    act = model.step(pc, vc, dsc, dc, DT).cpu().numpy()
    big = model.step(pc, vc, dsc, dc, BIG_DT).cpu().numpy().astype(np.float64)
    res = {"oracle": "oracle/piml_oracle.c orc_mlapm_step (mlapm.py:10-58 in the reference's fp32 op order, row sums "
                     "in fp64)"}
    if oracle_rows is not None and len(oracle_rows):
        R = len(oracle_rows)
        num = np.linalg.norm(act[:R].astype(np.float64) - oracle_rows, axis=-1)
        den = np.maximum(np.linalg.norm(oracle_rows, axis=-1), 1e-6)
        res.update({"action_rows": R, "max_rel_action": float((num / den).max())})
    block = 512
    T = (N + block - 1) // block
    e_all, nF_all, S_all = [], [], []
    for b in sorted({0, 1, T // 3 | 1, T // 2, (2 * T) // 3, T - 2, T - 1} & set(range(T))):
        lo, hi = b * block, min(N, b * block + block)
        _, force, opsum = O.mlapm_step_diag(pn, vn, dsn, dn, DT, "GC", rows=(lo, hi))
        F = (big[lo:hi] - vn[lo:hi].astype(np.float64)) / BIG_DT
        e_all.append(np.linalg.norm(F - force, axis=-1)); nF_all.append(np.linalg.norm(force, axis=-1))
        S_all.append(opsum)
    e, nF, S = [np.concatenate(x) for x in (e_all, nF_all, S_all)]
    strict = e / np.maximum(nF, 1e-30)
    kappa = S / np.maximum(nF, 1e-30)
    well = kappa <= 16.0
    res.update({"force_rows": int(len(e)), "max_rel_force": float(strict.max()),
                "max_rel_force_kappa": float(kappa[int(np.argmax(strict))]),
                "p999_rel_force": float(np.quantile(strict, 0.999)),
                "max_rel_force_well_conditioned": float(strict[well].max()) if well.any() else None,
                "well_conditioned_share": float(well.mean()),
                "max_force_err_over_operand_sum": float((e / S).max()),
                "gate": "||dF|| <= 1e-5 max(||F||, S/16) per agent; ||d action|| / ||action|| <= 1e-5 per agent",
                "pass": bool((e <= 1e-5 * np.maximum(nF, S / 16.0)).all()
                             and res.get("max_rel_action", 0.0) < 1e-5)})
    return res


def _import_reference():
    """The UNMODIFIED reference: /root/reference in the build container, its verbatim copy baseline/_ref on the GPU box
    (staged by __graft_entry__.build()).  Returns the src dir or None."""
    for root in ("/root/reference", os.path.join(ROOT, "baseline", "_ref")):
        src = os.path.join(root, "src")
        if os.path.isdir(os.path.join(src, "models")):
            if src not in sys.path:
                sys.path.insert(0, src)
            return src
    return None


def reference_pytorch(budget_s=60.0):
    """Time the reference's own PyTorch CPU path on this box's host cores (north star; BASELINE.md 3.1): MLAPM.step at
    N in {1024, 4096, 8192} and Pedestrians.get_relative_features at N in {512, 2048, 4096} (M = 2000), with 1 thread and
    with all threads; min and max of the repeats.  Sizes that would blow the time budget are skipped and say so."""
    import torch
    src = _import_reference()
    if src is None:
        return {"unavailable": "no reference tree (baseline/_ref missing: run __graft_entry__.build() in the container)"}
    from models.mlapm import MLAPM as RefMLAPM
    import data.data as RDATA
    cores = len(os.sched_getaffinity(0))
    keep = torch.get_num_threads()
    t_begin = time.perf_counter()
    out = {"source": src, "torch": torch.__version__, "cores": cores, "mlapm_step": [], "get_relative_features": []}

    def timed(fn, reps):
        ts = []
        for _ in range(reps):
            t0 = time.perf_counter()
            fn()
            ts.append(time.perf_counter() - t0)
        return min(ts), max(ts)
    ref = RefMLAPM(**MLAPM_KW)
    peds = RDATA.Pedestrians()
    try:
        for threads in (cores, 1):
            torch.set_num_threads(threads)
            for N in (1024, 4096, 8192):
                est = (N / 8192.0) ** 2 * (20.0 if threads == 1 else 5.0)
                if time.perf_counter() - t_begin + 2 * est > budget_s:
                    out["mlapm_step"].append({"N": N, "threads": threads, "skipped": "time budget"})
                    continue
                p, v, ds, dest, _ = synthetic_crowd(N)
                with torch.no_grad():
                    ref.step(p, v, ds, dest, DT)
                    lo, hi = timed(lambda: ref.step(p, v, ds, dest, DT), 2)
                out["mlapm_step"].append({"N": N, "threads": threads, "s_min": lo, "s_max": hi,
                                          "mpairs_per_s": N * N / lo / 1e6, "agent_steps_per_s": N / lo})
            for N in (512, 2048, 4096):
                est = (N / 4096.0) ** 2 * (7.0 if threads == 1 else 3.0)
                if time.perf_counter() - t_begin + 2 * est > budget_s:
                    out["get_relative_features"].append({"N": N, "threads": threads, "skipped": "time budget"})
                    continue
                p, v, ds, dest, obs = synthetic_crowd(N)
                a = torch.zeros_like(v)
                f = lambda: peds.get_relative_features(p[None].clone(), v[None].clone(), a[None].clone(),
                                                       dest[None].clone(), obs, 6, 90, 4, 10, 90, 4)
                with torch.no_grad():
                    lo, hi = timed(f, 2)
                out["get_relative_features"].append({"N": N, "M": int(obs.shape[0]), "threads": threads, "s_min": lo,
                                                     "s_max": hi, "agent_steps_per_s": N / lo})
    finally:
        torch.set_num_threads(keep)
    out["seconds"] = time.perf_counter() - t_begin
    return out


def run_reference(a):
    """--impl reference: the reference's CPU algorithm for this path (oracle port; the Python reference itself
    cannot run N = 100k -- one (N,N,2) fp32 temporary is 80 GB -- and does not travel to the GPU box)."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    if a.workload == "nn":
        return run_reference_nn(a)
    from oracle import oracle as O
    import numpy as np
    N = a.agents
    # all the host threads this process may use (torchrun exports OMP_NUM_THREADS=1 to its workers: override it)
    O.set_num_threads(len(os.sched_getaffinity(0)))
    cores = O.num_threads()
    p, v, ds, dest, _ = [x.numpy() for x in synthetic_crowd(N)]
    probe = max(64, cores * 16)
    O.mlapm_step(p, v, ds, dest, DT, "GC", rows=(0, probe))       # spin up the OpenMP team
    t0 = time.perf_counter()
    O.mlapm_step(p, v, ds, dest, DT, "GC", rows=(0, probe))
    rate = probe / max(time.perf_counter() - t0, 1e-6)
    budget = 90.0 / max(a.steps + a.warmup, 1)                     # whole run within a few minutes
    R = int(min(N, max(probe, rate * min(budget, 10.0))))
    for _ in range(a.warmup):
        O.mlapm_step(p, v, ds, dest, DT, "GC", rows=(0, R))
    t0 = time.perf_counter()
    for s in range(a.steps):
        r0 = (s * R) % max(N - R, 1)
        O.mlapm_step(p, v, ds, dest, DT, "GC", rows=(r0, r0 + R))
    dt = time.perf_counter() - t0
    val = R * a.steps / dt
    sample = (f"each step = rows [r0,r0+{R}) x all {N} columns of one MLAPM.step (oracle C port, OpenMP {cores} "
              f"threads); {R * N * a.steps / dt / 1e6:.1f} Mpairs/s")
    print(json.dumps({
        "impl": "reference", "metric": METRIC, "value": val, "unit": UNIT, "n_gpus": a.gpus, "steps": a.steps,
        "warmup": a.warmup, "ms_per_step": dt / a.steps * 1e3, "higher_is_better": True, "scaling": "strong",
        "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": bench_config(N, a.gpus),
        "ms_per_full_step": N / val * 1e3, "sample_rows_per_step": R,
        "note": "value = rows computed per second against all N columns (agent-steps/s of a full step is the same "
                "number); ms_per_step is the time of one SAMPLED step of R rows, ms_per_full_step its extrapolation "
                "to all N rows",
        "cpu_baseline": {"value": val, "unit": UNIT, "cores": cores, "kind": "port", "sample": sample},
        "e2e": {"value": val, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}))


def run_reference_nn(a):
    """--impl reference --workload nn: the oracle's port of one NN rollout step on all host threads, sampled rows."""
    N = a.agents
    _, _, _, _, obs_h = synthetic_crowd(N)
    budget = min(8.0, 90.0 / max(a.steps + a.warmup, 1))
    cpu, R, _, dt = nn_cpu_baseline(N, obs_h, seconds=budget, steps=max(a.steps, 1))
    print(json.dumps({
        "impl": "reference", "metric": METRIC, "value": cpu["value"], "unit": UNIT, "n_gpus": a.gpus, "steps": a.steps,
        "warmup": a.warmup, "ms_per_step": dt * 1e3, "ms_per_full_step": N / cpu["value"] * 1e3,
        "sample_rows_per_step": R, "higher_is_better": True, "scaling": "strong", "vs_baseline": None, "dtype": "f32",
        "data": "synthetic", "config": nn_config(N, int(obs_h.shape[0])), "cpu_baseline": cpu,
        "e2e": {"value": cpu["value"], "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}))


def run_nn(a):
    """--workload nn: the NN-augmented rollout step as the main line (1 GPU: NNCrowd; torchrun: ShardedNNCrowd)."""
    import torch
    import torch.distributed as dist
    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device; the piml_b200 hot path has no CPU fallback")
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    N = a.agents
    _, _, _, _, obs_h = synthetic_crowd(N)
    sampler = ClockSampler(local) if rank == 0 else None
    if sampler:
        sampler.start(); time.sleep(0.3)
    if world == 1:
        blk = nn_workload(torch, dev, N, obs_h, a.steps, a.warmup, with_cpu=not a.no_cpu)
        if sampler:
            sampler.stop()
        line = {"metric": METRIC, "value": blk["value"], "unit": UNIT, "n_gpus": 1, "steps": a.steps,
                "warmup": max(a.warmup, 3), "ms_per_step": blk["ms_per_step"], "higher_is_better": True,
                "scaling": "strong", "vs_baseline": None, "dtype": "f32", "data": "synthetic"}
        line.update({k: v for k, v in blk.items() if k not in line})
        line["clocks"] = sampler.summary() if sampler else None
        print(json.dumps(line))
        return
    dist.init_process_group("nccl", device_id=dev)
    blk = nn_path_sharded(torch, dist, dev, N, obs_h, world, iters=a.steps)
    if rank == 0:
        sampler.stop()
        ms = blk.get("ms_per_step")
        print(json.dumps({"metric": METRIC, "value": (N / ms * 1e3) if ms else None, "unit": UNIT, "n_gpus": world,
                          "steps": a.steps, "warmup": 3, "ms_per_step": ms, "higher_is_better": True,
                          "scaling": "strong", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
                          "config": nn_config(N, int(obs_h.shape[0])), "detail": blk, "clocks": sampler.summary()}))
    dist.destroy_process_group()


def bench_config(N, world):
    """The workload both arms run (identical keys and values in `ours` and `--impl reference`)."""
    return {"workload": f"mlapm_gc_rollout_N{N}", "agents": N,
            "reference": "src/main_mlapm.py:18-36 + src/models/mlapm.py:10-58, version GC",
            "crowd": "SURVEY 8d config 4: seed 666, rho 0.5 ped/m^2, dt 0.08",
            "l2": f"{FLUSH_MB} MB memset between steps, inside the timed region (GPU arm)"}


def probe_peaks(L, torch, dev):
    """FP32 FMA and MUFU pipe peaks, measured live with the library's probe kernels (best of 5)."""
    sms = torch.cuda.get_device_properties(dev).multi_processor_count
    ctas, iters = sms * 8, 4096
    out = torch.empty(ctas * 256, device=dev)
    res = {}
    for which, name, per in ((0, "fp32_tflops", 2.0), (1, "mufu_tops", 1.0)):
        best = 0.0
        for _ in range(6):
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            L.check(L.load().piml_pipe_probe(which, ctas, iters, L.ptr(out), L.stream_ptr(dev)), "piml_pipe_probe")
            e1.record()
            torch.cuda.synchronize()
            ms = e0.elapsed_time(e1)
            best = max(best, ctas * 256 * iters * 32 * per / (ms * 1e-3) / 1e12)
        res[name] = best
    return res


NN_ARGS = dict(model='pinnsf_bm', dataset_name='gc1560', dropout=0.5, encoder_hidden_size=128,
               processor_hidden_size=128, decoder_hidden_size=64, encoder_hidden_layers=3, processor_hidden_layers=16,
               decoder_hidden_layers=2, ped_feature_dim=6, obs_feature_dim=6, self_feature_dim=7, topk_ped=6,
               topk_obs=10, sight_angle_ped=90, sight_angle_obs=90, dist_threshold_ped=4, dist_threshold_obs=4,
               time_unit=DT)
NN_FEATURE_ARGS = (6, 90, 4, 10, 90, 4)
NN_FLOP_PER_AGENT = 1.52e6            # SURVEY.md 8d: pinnsf_bm forward, 6 ped + 10 obstacle slots
# algorithmic HBM bytes per agent-step, stage by stage (DESIGN.md 4.2-4.5): features read 44 B of state and write
# (6 + 10) slots x 24 B + 28 B self + 8 B dest; the forward reads those 420 B and writes 8 B; integrate reads 68 B and
# writes 48 B.  A fully fused step would move 44 + 48 = 92 B (SURVEY.md 8d "68-92 B").
NN_BYTES_PER_AGENT = 44 + 384 + 28 + 8 + 420 + 8 + 68 + 48
NN_BYTES_PER_AGENT_FUSED = 92


def nn_config(N, M=2000):
    return {"workload": f"pinnsf_bm_nn_rollout_N{N}", "agents": N, "obstacle_points": M,
            "reference": "src/models/simulators.py:595-652 (model forward -> Euler / arrival -> get_relative_features), "
                         "src/models/model.py:1185-1221, src/data/data.py:466-512",
            "crowd": "SURVEY 8d config 4: seed 666, rho 0.5 ped/m^2, dt 0.08, k 6/10, 90 deg, 4 m; seed-666 weights",
            "l2": f"{FLUSH_MB} MB memset before every step; each step has its own CUDA-event pair (GPU arm)"}


class NNCrowd(object):
    """One NN-augmented rollout step (simulators.py:602-652) on the synthetic crowd: pinnsf_bm forward (tcgen05),
    integrate, cell-list feature rebuild.  Device-resident state; `step()` enqueues the stage kernels."""

    def __init__(self, torch, dev, N, obs_h):
        import argparse as ap
        from piml_b200 import models as M
        from piml_b200.rollout import integrate_step, state_features
        self.torch, self.dev, self.N, self.models = torch, dev, N, M
        self._integrate, self._features = integrate_step, state_features
        torch.manual_seed(666)
        self.net = M.PINNSF_bottleneck_multitask(ap.Namespace(**NN_ARGS)).to(dev).eval()
        self.packed = M.pack_device(self.net.state_dict(), self.net.spec, dev)
        self.packed_tc = M.pack_device_tc(self.net.state_dict(), self.net.spec, dev)
        p, v, ds, dest, _ = synthetic_crowd(N)
        # the crowd's state in ONE device buffer [p | v | a | dest | desired speed] (9 N floats) with a pinned host twin:
        # a host-side loop then pays one H2D and one D2H per step instead of five + three
        self.h_state = torch.cat([p.reshape(-1), v.reshape(-1), torch.zeros(2 * N), dest.reshape(-1),
                                  ds.reshape(-1)]).pin_memory()
        self.d_state = self.h_state.to(dev)
        self.p, self.v, self.acc, self.dest = [self.d_state[2 * N * k:2 * N * (k + 1)].view(1, N, 2) for k in range(4)]
        self.ds = self.d_state[8 * N:].view(1, N)
        self.hist = self.v.clone()
        self.obs = obs_h.to(dev)
        self.didx = torch.zeros(1, N, dtype=torch.int64, device=dev)
        self.dnum = torch.ones(1, N, dtype=torch.int64, device=dev)
        self.wp = self.dest[:, None].contiguous()
        self.bufs = tuple(self._features(self.p, self.v, self.acc, self.dest, self.obs, self.hist, self.ds,
                                         *NN_FEATURE_ARGS)) + (torch.empty(1, N, 2, device=dev),)
        self.a_next = None
        self._fused = None
        self.h_out = torch.empty(6 * N).pin_memory()           # new p | v | a

    def forward(self):
        N, M = self.N, self.models
        pf, of, sf = self.bufs[:3]
        self.a_next = M.pinnsf_forward(self.net.spec, self.packed, pf.view(N, 6, 6), of.view(N, -1, 6), sf.view(N, 7),
                                       need_msgs=False, packed_tc=self.packed_tc)[0].view(1, N, 2)

    def integrate(self):
        self._integrate(self.p, self.v, self.acc, self.a_next, self.dest, self.didx, self.dnum, self.wp, DT, False,
                        hist_v=self.hist)

    def features(self):
        self._features(self.p, self.v, self.acc, self.dest, self.obs, self.hist, self.ds, *NN_FEATURE_ARGS,
                       out=self.bufs)

    def step(self):
        self.forward(); self.integrate(); self.features()

    def step_fused(self):
        """The same step as ONE library call (piml_nn_step_f32): features -> forward -> integrate on the state."""
        if self._fused is None:
            from piml_b200.rollout import NNStep
            self._fused = NNStep(self.net.spec, self.packed_tc, self.p, self.v, self.acc, self.dest, self.didx,
                                 self.hist, self.dnum, self.wp, self.ds, self.obs, DT, *NN_FEATURE_ARGS,
                                 remove_on_arrival=False)
        self._fused.step()

    def e2e_step(self):
        """Host state in (pinned), one step, new p / v / a out: what a host-side simulation loop pays per step."""
        self.d_state.copy_(self.h_state, non_blocking=True)
        self.hist.copy_(self.v)
        self.step_fused()
        self.h_out.copy_(self.d_state[:6 * self.N])

    @property
    def e2e_bytes(self):
        return self.N * 4 * (2 + 2 + 2 + 2 + 1), self.N * 4 * 6


def nn_cpu_baseline(N, obs_h, seconds=8.0, steps=1, rows0=0):
    """Oracle C port of one NN rollout step on the host cores for rows [r0, r0+R) against all N agents / M obstacles:
    get_relative_features (data.py:466-512) -> pinnsf_bm forward (model.py:1185-1221) -> Euler update
    (simulators.py:603-604).  Returns (block, rows, (features, acceleration) of those rows for the parity check)."""
    import argparse as ap
    import numpy as np
    import torch
    from oracle import oracle as O
    from piml_b200 import models as M
    O.set_num_threads(len(os.sched_getaffinity(0)))
    cores = O.num_threads()
    torch.manual_seed(666)
    net = M.PINNSF_bottleneck_multitask(ap.Namespace(**NN_ARGS)).eval()
    desc = O.net_desc(net.spec.enc_dims, net.spec.proc_mode, net.spec.dec_dims, net.spec.coll_dims, net.spec.kind)
    flat = M.pack_state_dict(net.state_dict(), net.spec).cpu().numpy()
    p, v, ds, dest, _ = [x.numpy() for x in synthetic_crowd(N)]
    a, obs = np.zeros_like(v), obs_h.numpy()

    def rows_step(r0, r1):
        w = O.relative_features_rows(p, v, a, dest, obs, (r0, r1), *NN_FEATURE_ARGS)
        slf = np.concatenate([w[2], v[r0:r1], a[r0:r1], ds[r0:r1]], -1)
        acc = O.pinnsf_forward(desc, flat, net.spec.tau, w[0], w[1], slf)[0]
        R = r1 - r0
        O.integrate_step(p[r0:r1], v[r0:r1], a[r0:r1], acc, dest[r0:r1], np.zeros(R, np.int64), np.ones(R, np.int64),
                         dest[None, r0:r1], DT, remove_on_arrival=False)
        return w, slf, acc
    probe = max(64, cores * 8)
    rows_step(0, probe)
    t0 = time.perf_counter()
    rows_step(0, probe)
    rate = probe / max(time.perf_counter() - t0, 1e-6)
    R = int(min(N, max(probe, rate * seconds)))
    t0 = time.perf_counter()
    for s_ in range(steps):
        r0 = (rows0 + s_ * R) % max(N - R, 1)
        w, slf, acc = rows_step(r0, r0 + R)
    dt = (time.perf_counter() - t0) / steps
    return ({"value": R / dt, "unit": UNIT, "cores": cores, "kind": "port",
             "sample": f"oracle C port (OpenMP, {cores} threads) of one NN rollout step: rows [r0,r0+{R}) x all {N} "
                       f"agents + {obs.shape[0]} obstacles (features), {R} x 16 slot rows through pinnsf_bm, Euler; "
                       f"{dt:.1f} s per sampled step"}, R, (r0, w, slf, acc), dt)


def nn_workload(torch, dev, N, obs_h, steps, warmup, with_cpu=True):
    """The NN-augmented rollout step as a full bench block (value / e2e / roofline / cpu_baseline / parity)."""
    from piml_b200 import _lib as L
    import numpy as np
    crowd = NNCrowd(torch, dev, N, obs_h)
    flush = torch.empty(FLUSH_MB << 20, dtype=torch.uint8, device=dev)
    ev = lambda: torch.cuda.Event(enable_timing=True)
    # ---- the three-call route (state_features / pinnsf_forward / integrate_step): per-stage times, and the forward
    # stage's time for the tensor roofline (the fused step launches the same forward kernel inside one C call)
    for _ in range(max(warmup, 3)):
        flush.zero_(); crowd.step()
    torch.cuda.synchronize()
    marks = [[ev() for _ in range(4)] for _ in range(steps)]
    u0, u1 = ev(), ev()
    u0.record()
    for s_ in range(steps):
        flush.zero_()
        marks[s_][0].record(); crowd.forward()
        marks[s_][1].record(); crowd.integrate()
        marks[s_][2].record(); crowd.features()
        marks[s_][3].record()
    u1.record()
    torch.cuda.synchronize()
    ms3 = u0.elapsed_time(u1) / steps
    st = [sum(m[i].elapsed_time(m[i + 1]) for m in marks) / steps for i in range(3)]
    # ---- the timed path: the fused step, ONE library call per step (piml_nn_step_f32)
    for _ in range(max(warmup, 3)):
        flush.zero_(); crowd.step_fused()
    torch.cuda.synchronize()
    launches0 = L.launch_count()
    pairs = [(ev(), ev()) for _ in range(steps)]
    for s_ in range(steps):
        flush.zero_()                                       # L2 flushed before every step, outside its event pair
        pairs[s_][0].record(); crowd.step_fused(); pairs[s_][1].record()
    torch.cuda.synchronize()
    launches = L.launch_count() - launches0
    ms = sum(a_.elapsed_time(b_) for a_, b_ in pairs) / steps
    assert torch.isfinite(crowd.p[0]).sum() > 0
    # ---- end to end with host buffers
    for _ in range(2):
        crowd.e2e_step()
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    g0, g1 = ev(), ev()
    g0.record()
    for _ in range(steps):
        crowd.e2e_step()
    g1.record()
    torch.cuda.synchronize()
    e2e_ms = max(g0.elapsed_time(g1), (time.perf_counter() - t0) * 1e3) / steps
    h2d, d2h = crowd.e2e_bytes
    peak_gbs, peak_src, bf16 = 6550.0, "fallback (B200_PROFILING.md)", 1650.0
    try:
        with open(os.path.join(ROOT, "MEASURED_PEAKS.json")) as f:
            pk = json.load(f)
            peak_gbs, bf16, peak_src = float(pk["hbm_gbs"]), float(pk["bf16_tflops"]), "MEASURED_PEAKS.json"
    except Exception:
        pass
    gbs = NN_BYTES_PER_AGENT_FUSED * N / (ms * 1e-3) / 1e9
    fwd_tf = NN_FLOP_PER_AGENT * N / (st[0] * 1e-3) / 1e12
    # what the tensor cores actually execute: the non-empty slot rows only, 3 fp16 MMA terms per product
    live_rows = int((crowd.bufs[0].abs().sum(-1) > 0).sum()) + int((crowd.bufs[1].abs().sum(-1) > 0).sum())
    exec_tf = 3.0 * live_rows * (NN_FLOP_PER_AGENT / 16.0) / (st[0] * 1e-3) / 1e12
    block = {
        "metric": METRIC, "value": N / ms * 1e3, "unit": UNIT, "ms_per_step": ms, "steps": steps,
        "config": nn_config(N, int(obs_h.shape[0])), "dtype": "f32 (network contractions as 3-term split products on "
                                                               "the tensor cores, fp32 accumulate)",
        "api": "piml_b200.rollout.NNStep.step -> piml_nn_step_f32: cell-list features (compact slot rows) -> tcgen05 "
               "forward -> slot sums + destination term + Euler, 7 launches",
        "three_call_route": {"ms_per_step": ms3, "stage_ms": {"forward": st[0], "integrate": st[1], "features": st[2]},
                             "note": "state_features -> pinnsf_forward -> integrate_step (12 stream operations); the "
                                     "fused step is bit-identical to it (parity.fused_step_bit_identical)"},
        "roofline": {"bound": "tensor", "kernel": "pinnsf_tc16_kernel (+ compaction, finish: the forward stage of the "
                                                  "three-call route, same kernel on the same rows)",
                     "achieved": fwd_tf, "peak": bf16 / 2.0, "unit": "TFLOP/s", "frac": fwd_tf / (bf16 / 2.0),
                     "peak_source": peak_src + " bf16_tflops / 2 (dense tf32 rate)",
                     "note": "achieved = 1.52 MFLOP per agent (SURVEY 8d, all 16 slots) / forward stage time; the "
                             "kernel evaluates only non-empty slot rows (compact mode) but spends 3 MMAs per product "
                             "(3-term split for fp32-grade results), so executed tensor FLOPs differ from algorithmic",
                     "traffic": None,
                     "executed": {"slot_rows_evaluated": live_rows, "slot_rows_dense": 16 * N,
                                  "fp16_tensor_tflops_executed": exec_tf, "fp16_peak_tflops": bf16,
                                  "frac_of_fp16_peak": exec_tf / bf16, "tensor_pipe_busy_ncu": 0.429,
                                  "source": "profiles/r02m_ncu_pinnsf_tc16_kernel.txt; 36 of a tile's 87 MMAs are N = 64 "
                                            "(half a pipe pass each), so pipe-busy sits below the FLOP fraction"},
                     "hbm": {"bytes_per_agent_step": NN_BYTES_PER_AGENT, "bytes_per_agent_step_fused": NN_BYTES_PER_AGENT_FUSED,
                             "achieved": gbs, "peak": peak_gbs, "unit": "GB/s", "frac": gbs / peak_gbs,
                             "note": "whole fused step, its algorithmic bytes (state in / out, bytes_per_agent_step_fused) "
                                     "against the HBM copy peak: the step is tensor / instruction bound, not HBM bound, "
                                     "at this size; bytes_per_agent_step is what the unfused stages move"}},
        "e2e": {"value": N / e2e_ms * 1e3, "unit": UNIT, "ms_per_step": e2e_ms, "h2d_bytes_per_step": h2d,
                "d2h_bytes_per_step": d2h,
                "api": "pinned host state [p | v | a | dest | desired speed] (one buffer, one H2D) -> NNStep.step "
                       "(piml_nn_step_f32) -> host [p | v | a] (one D2H)"},
        "gpu_launches": launches,
    }
    if with_cpu:
        cpu, R, (r0, w, slf, acc_ref), _ = nn_cpu_baseline(N, obs_h)
        block["cpu_baseline"] = cpu
        # parity of the timed path on the rows the CPU leg just computed (fresh crowd, first step)
        chk = NNCrowd(torch, dev, N, obs_h)
        pf, of, sf = [x[0, r0:r0 + R].cpu().numpy() for x in chk.bufs[:3]]
        chk.forward()
        acc = chk.a_next[0, r0:r0 + R].cpu().numpy().astype(np.float64)
        n = np.linalg.norm(slf[:, :2], axis=-1, keepdims=True)
        dterm = (slf[:, 6:7] * slf[:, :2] / np.where(n == 0, 0.1, n) - slf[:, 2:4]) / chk.net.spec.tau
        err = np.linalg.norm(acc - acc_ref, axis=-1)
        scale = np.maximum(np.maximum(np.linalg.norm(acc_ref, axis=-1), np.linalg.norm(dterm, axis=-1)), 1e-3)
        block["parity"] = {"rows": R, "features_bit_exact": bool(np.array_equal(pf, w[0]) and np.array_equal(of, w[1])
                                                                  and np.array_equal(sf, slf)),
                           "max_rel_acceleration_operand_scaled": float((err / scale).max()),
                           "max_rel_acceleration_strict": float((err / np.maximum(np.linalg.norm(acc_ref, axis=-1),
                                                                                  1e-6)).max()),
                           "gate": "features bit-exact; ||da|| <= 1e-5 max(||a||, ||dest term||) per agent"}
        # the fused step against the three calls on fresh crowds: every state tensor bit for bit after 2 steps
        c3, cf = NNCrowd(torch, dev, N, obs_h), NNCrowd(torch, dev, N, obs_h)
        for _ in range(2):
            c3.features(); c3.forward(); c3.integrate()
            cf.step_fused()
        same = all(np.array_equal(x.cpu().numpy(), y.cpu().numpy(), equal_nan=True)
                   for x, y in ((c3.p, cf.p), (c3.v, cf.v), (c3.acc, cf.acc), (c3.dest, cf.dest), (c3.hist, cf.hist)))
        block["parity"]["fused_step_bit_identical"] = bool(same)
        block["parity"]["pass"] = bool(block["parity"]["features_bit_exact"] and same
                                       and block["parity"]["max_rel_acceleration_operand_scaled"] < 1e-5)
    return block


def nn_path_sharded(torch, dist, dev, N, obs_h, world, iters=10):
    """Under torchrun: the same NN rollout step agent-sharded (piml_b200.sharded.ShardedNNCrowd: the fused step on the
    rank's own rows, new state pushed to the peers from the last kernel's epilogue)."""
    import argparse as ap
    from piml_b200 import models as M
    from piml_b200.sharded import ShardedNNCrowd
    args = ap.Namespace(model='pinnsf_bm', dataset_name='gc1560', dropout=0.5, encoder_hidden_size=128,
                        processor_hidden_size=128, decoder_hidden_size=64, encoder_hidden_layers=3,
                        processor_hidden_layers=16, decoder_hidden_layers=2, ped_feature_dim=6, obs_feature_dim=6,
                        self_feature_dim=7, topk_ped=6, topk_obs=10, sight_angle_ped=90, sight_angle_obs=90,
                        dist_threshold_ped=4, dist_threshold_obs=4, time_unit=DT)
    crowd, err = None, ""
    try:
        torch.manual_seed(666)
        net = M.PINNSF_bottleneck_multitask(args).to(dev).eval()
        p, v, ds, dest, _ = [x.to(dev) for x in synthetic_crowd(N)]
        crowd = ShardedNNCrowd(net, args, N, obs_h.to(dev), device=dev)
        crowd.load(p, v, torch.zeros_like(v), dest, torch.zeros(N, dtype=torch.int64),
                   torch.ones(N, dtype=torch.int64), dest[None], ds)
        with torch.no_grad():
            crowd.step(remove_on_arrival=False) if world == 1 else None
    except Exception as e:
        crowd, err = None, f"{type(e).__name__}: {e}"[:300]
    ok = torch.tensor([1 if crowd is not None else 0], device=dev)
    dist.all_reduce(ok, op=dist.ReduceOp.MIN)               # all ranks take the collective steps, or none does
    if int(ok) == 0:
        return {"error": err or "setup failed on another rank"}
    try:
        with torch.no_grad():
            for _ in range(3):
                crowd.step(remove_on_arrival=False)
            dist.barrier(); torch.cuda.synchronize()
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            for _ in range(iters):
                crowd.step(remove_on_arrival=False)
            e1.record()
            dist.barrier(); torch.cuda.synchronize()
        ms = torch.tensor([e0.elapsed_time(e1) / iters], device=dev)
        dist.all_reduce(ms, op=dist.ReduceOp.MAX)
        ms = float(ms)
        how = ("fused step per rank (piml_nn_step_shard_f32): cell list over all agents, own rows in sorted order -> "
               "tcgen05 forward -> Euler; new p, v, a pushed into every rank's next state over NVLink peer memory "
               "(24 B/agent/peer), one barrier") if getattr(crowd, "fused", False) else \
              ("own-row cell-list features + tcgen05 forward, NCCL all-gather of the accelerations (8 B/agent), "
               "replicated integrate")
        return {"workload": f"pinnsf_bm NN rollout step, N={N}, agent-sharded x{world}: {how}",
                "ms_per_step": ms, "agent_steps_per_sec": N / ms * 1e3}
    except Exception as e:                               # secondary evidence must never take the headline down
        return {"error": f"{type(e).__name__}: {e}"[:300]}


def crowd_1m_block(torch, dist, dev, world, rank, steps=3):
    """BASELINE configs[4] (a): one MLAPM crowd of 1 000 000 agents, agent-sharded over the ranks (ShardedCrowd: block
    ownership, shares and new state pushed over NVLink peer memory); one GPU: the unsharded symmetric kernel."""
    import piml_b200 as P
    N = 1000000
    try:
        p, v, ds, dest, _ = [x.to(dev) for x in synthetic_crowd(N)]
        model = P.MLAPM(**MLAPM_KW)
        crowd = None
        if world > 1:
            from piml_b200.sharded import ShardedCrowd
            crowd = ShardedCrowd(N, device=dev)
            crowd.load(p, v)
        state = [p, v]

        def one():
            if crowd is not None:
                crowd.step(model, ds, dest, DT, RADIUS)
            else:
                act, pn, _ = model.advance(state[0], state[1], ds, dest, DT, RADIUS)
                state[0], state[1] = pn, act
        one()
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(steps):
            one()
        e1.record()
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()
        ms = torch.tensor([e0.elapsed_time(e1) / steps], device=dev)
        if world > 1:
            dist.all_reduce(ms, op=dist.ReduceOp.MAX)
        ms = float(ms)
        fin = crowd.position if crowd is not None else state[0]
        ok = bool(torch.isfinite(fin).all())
        ws = (crowd._sym_ws.numel() if crowd is not None else model._ws.numel())
        del crowd, model
        torch.cuda.empty_cache()
        return {"workload": f"mlapm_gc_rollout_N{N}, agent-sharded x{world}", "agents": N, "steps": steps,
                "ms_per_step": ms, "agent_steps_per_sec": N / ms * 1e3, "scaling": "strong",
                "tflops_algorithmic": FLOP_PER_PAIR * N * N / (ms * 1e-3) / 1e12, "workspace_bytes_per_rank": int(ws),
                "finite": ok}
    except Exception as e:                                   # secondary block: never take the headline down
        return {"error": f"{type(e).__name__}: {e}"[:300]}


def nn_crowd_1m_block(torch, dist, dev, world, rank, steps=5):
    """BASELINE configs[4] (a) on the path the metric names: one crowd of 1 000 000 agents through the NN-augmented
    rollout step -- one GPU: the fused step (NNStep); torchrun: agent-sharded (ShardedNNCrowd, new state pushed over
    NVLink peer memory)."""
    N = 1000000
    try:
        _, _, _, _, obs_h = synthetic_crowd(N)
        if world > 1:
            blk = nn_path_sharded(torch, dist, dev, N, obs_h, world, iters=steps)
        else:
            crowd = NNCrowd(torch, dev, N, obs_h)
            for _ in range(2):
                crowd.step_fused()
            torch.cuda.synchronize()
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            for _ in range(steps):
                crowd.step_fused()
            e1.record()
            torch.cuda.synchronize()
            ms = e0.elapsed_time(e1) / steps
            assert torch.isfinite(crowd.p[0]).sum() > 0
            blk = {"workload": f"pinnsf_bm NN rollout step, N={N}, one GPU: fused step (piml_nn_step_f32); no explicit L2 "
                               "flush: the step's working set (compact rows, messages, maps: ~0.4 GB) is larger than L2",
                   "ms_per_step": ms, "agent_steps_per_sec": N / ms * 1e3}
            del crowd
        torch.cuda.empty_cache()
        return blk
    except Exception as e:                                   # secondary block: never take the headline down
        return {"error": f"{type(e).__name__}: {e}"[:300]}


def clip_rollouts_block(torch, dev):
    """BASELINE configs[0] / [1] as the reference runs them: ONE clip rolled from t = 25 to its last frame through
    `piml_rollout_f32` -- the GC clip (N = 122 slots, 750 frames, pinnsf_bm with the golden run's weights) and the
    synthetic social-force clip (N = 110, 750 frames, the pure social-force model in the persistent kernel).  A single
    scene is launch-latency bound; the reference takes 13-20 ms per step on CPU (BASELINE.md)."""
    import argparse as ap
    import numpy as np
    import piml_b200 as P
    from piml_b200 import models as M
    from piml_b200.rollout import rollout_scenes
    out = {}
    for name, key in (("rollout_gc_bm", "gc_clip_pinnsf_bm"), ("rollout_syn_sfm", "synthetic_clip_social_force")):
        try:
            z = np.load(os.path.join(ROOT, "tests", "golden", name + ".npz"))
            t0, T = int(z["in/t_start"]), int(z["in/position"].shape[0])
            cu = lambda k, dt=torch.float32: torch.as_tensor(z["in/" + k]).to(dev, dt)
            scene = {k: cu(k)[None].contiguous() for k in ("position", "velocity", "acceleration", "destination",
                                                           "mask_p", "mask_p_pred", "waypoints", "desired_speed")}
            scene["dest_idx"], scene["dest_num"] = cu("dest_idx", torch.int64)[None], cu("dest_num", torch.int64)[None]
            scene["obstacles"] = cu("obstacles")
            for k in ("ped_features0", "obs_features0", "self_features0"):
                scene[k] = cu(k)[None]
            args = ap.Namespace(**dict(NN_ARGS, time_unit=float(z["in/time_unit"])))
            if str(z["in/model"]) == "sfm":
                spec, packed, packed_tc = P.SocialForce(str(z["in/dataset_name"])).spec, None, None
            else:
                torch.manual_seed(666)
                net = M.PINNSF_bottleneck_multitask(args).to(dev).eval()
                net.load_state_dict({k[3:]: torch.from_numpy(z[k]) for k in z.files if k.startswith("sd/")})
                spec, packed = net.spec, M.pack_device(net.state_dict(), net.spec, dev)
                packed_tc = M.pack_device_tc(net.state_dict(), net.spec, dev)
            run = lambda: rollout_scenes(spec, packed, args, scene, t0, T, packed_tc=packed_tc)
            run()
            torch.cuda.synchronize()
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            res = run()
            e1.record()
            torch.cuda.synchronize()
            ms, N, steps = e0.elapsed_time(e1), int(scene["position"].shape[2]), T - t0
            out[key] = {"slots": N, "frames": steps, "ms_total": ms, "ms_per_step": ms / steps,
                        "agent_steps_per_sec": N * steps / ms * 1e3, "finite_positions": int(torch.isfinite(res[0]).sum())}
        except Exception as e:                               # secondary block: never take the headline down
            out[key] = {"error": f"{type(e).__name__}: {e}"[:300]}
    return out


def scenes_block(torch, dist, dev, world, rank, S_total=4096, steps=100):
    """BASELINE configs[4] (b): 4096 independent GC-shaped scenes (the GC clip's own state at t = 25, jittered per scene
    by seeded N(0, 0.05 m)) rolled `steps` frames with pinnsf_bm; scene s runs on rank s mod G, no communication."""
    import argparse as ap
    import numpy as np
    from piml_b200 import models as M
    from piml_b200.rollout import rollout_scenes, state_features
    try:
        z = np.load(os.path.join(ROOT, "tests", "golden", "rollout_gc_bm.npz"))
        t0 = int(z["in/t_start"])
        T = t0 + steps + 1
        mine = list(range(rank, S_total, world))
        S = len(mine)
        g = torch.Generator().manual_seed(1234)
        jitter = (0.05 * torch.randn(S_total, int(z["in/position"].shape[1]), 2, generator=g))[mine].to(dev)
        cu = lambda k, dt=torch.float32: torch.as_tensor(z["in/" + k][:T] if z["in/" + k].ndim and z["in/" + k].shape[0] >= T
                                                          and k not in ("waypoints", "obstacles", "dest_num", "desired_speed")
                                                          else z["in/" + k]).to(dev, dt)
        scene = {k: cu(k)[None].expand(S, *cu(k).shape).contiguous() for k in ("position", "velocity", "acceleration",
                                                                              "destination", "mask_p", "mask_p_pred")}
        scene["position"][:, t0] += jitter
        scene["dest_idx"] = cu("dest_idx", torch.int64)[None].expand(S, -1, -1).contiguous()
        scene["waypoints"] = cu("waypoints")[None].expand(S, -1, -1, -1).contiguous()
        scene["dest_num"] = cu("dest_num", torch.int64)[None].expand(S, -1).contiguous()
        scene["obstacles"] = cu("obstacles")
        scene["desired_speed"] = cu("desired_speed")[None].expand(S, -1).contiguous()
        args = ap.Namespace(**dict(NN_ARGS, time_unit=float(z["in/time_unit"])))
        torch.manual_seed(666)
        net = M.PINNSF_bottleneck_multitask(args).to(dev).eval()
        net.load_state_dict({k[3:]: torch.from_numpy(z[k]) for k in z.files if k.startswith("sd/")})
        packed = M.pack_device(net.state_dict(), net.spec, dev)
        packed_tc = M.pack_device_tc(net.state_dict(), net.spec, dev)
        hist0 = cu("self_features0")[None, :, 2:4].expand(S, -1, -1).contiguous()
        f0 = state_features(scene["position"][:, t0].contiguous(), scene["velocity"][:, t0].contiguous(),
                            scene["acceleration"][:, t0].contiguous(), scene["destination"][:, t0].contiguous(),
                            scene["obstacles"], hist0, scene["desired_speed"], *NN_FEATURE_ARGS)
        scene["ped_features0"], scene["obs_features0"], scene["self_features0"] = f0
        Ns = scene["position"].shape[2]
        run = lambda: rollout_scenes(net.spec, packed, args, scene, t0, T, packed_tc=packed_tc)
        run()
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        res = run()
        e1.record()
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()
        ms = torch.tensor([e0.elapsed_time(e1)], device=dev)
        if world > 1:
            dist.all_reduce(ms, op=dist.ReduceOp.MAX)
        ms = float(ms)
        nsteps = T - t0
        active = float(res[3][:, t0:T].sum()) / max(S * nsteps, 1)
        del scene, res
        torch.cuda.empty_cache()
        return {"workload": f"{S_total} GC-shaped scenes x {Ns} slots, pinnsf_bm rollout of {nsteps} frames from t = {t0}, "
                            f"scene-parallel x{world} (no communication)", "scenes": S_total, "slots": int(Ns),
                "frames": nsteps, "ms_total": ms, "ms_per_step": ms / nsteps, "scaling": "strong",
                "agent_steps_per_sec": S_total * Ns * nsteps / ms * 1e3, "mean_active_agents_per_scene": active}
    except Exception as e:
        return {"error": f"{type(e).__name__}: {e}"[:300]}


def sharded_timeline(torch, dist, dev, crowd, model, ds, dest, world, steps=5):
    """Per-rank stage times of the agent-sharded MLAPM step (CUDA events at the stage boundaries inside
    ShardedCrowd.step): pairs + share push | barrier 1 | finalize + state push | barrier 2, averaged over `steps`."""
    names = ["pairs_and_share_push", "barrier_1", "finalize_and_state_push", "barrier_2"] if crowd.symmetric else \
        ["rows_and_state_push", "barrier"]
    acc = [0.0] * len(names)
    for _ in range(steps):
        tr = []
        crowd.step(model, ds, dest, DT, RADIUS, trace=tr)
        torch.cuda.synchronize()
        for i in range(len(names)):
            acc[i] += tr[i].elapsed_time(tr[i + 1]) / steps
    mine = torch.tensor(acc, device=dev)
    allr = [torch.zeros_like(mine) for _ in range(world)]
    dist.all_gather(allr, mine)
    return {"stages": names, "ms_per_rank": [[round(float(x), 4) for x in r] for r in allr]}


def training_block(torch, dev, with_reference=True):
    """BASELINE configs[2]: one rollout-training step (UCY clip, pinnsf_bm, channelled windows of 5 steps, 144 slots):
    test_multiple_rollouts_for_training + loss.backward() + Adam, every kernel from libpiml_b200.so, on the reference's own
    batch (tests/golden/training_rollout.npz, 6 channels) tiled to the config's batch of C = 32 channels; next to it the
    UNMODIFIED reference (baseline/_ref, PyTorch CPU, all host threads) on the 6-channel batch it was generated from."""
    import argparse as ap
    try:
        import piml_b200 as P
        from piml_b200 import train_rollout as TRO
        from tests.golden_args import base_args
        from tests.test_gpu_training import _batch_from_golden, mirror
        from tests.util import golden, group
        g = group(golden("training_rollout"), "ucy_bm")
        kind, dsn = str(g["in/model"]), str(g["in/dataset_name"])
        x = g["in/args"]
        args = base_args(model=kind, dataset_name=dsn, reg_weight=float(x[0]), collision_threshold=float(x[1]),
                         collision_loss_weight=float(x[2]), hard_collision_penalty=float(x[3]),
                         teacher_weight=float(x[4]), collision_pred_weight=float(x[5]),
                         collision_focus_weight=float(x[6]), new_collision_loss_flag=int(x[7]), time_decay=float(x[8]),
                         collision_loss_version=str(g["in/collision_loss_version"]))
        net = mirror(kind, dsn, None, True)
        opt = torch.optim.Adam(net.parameters(), lr=4e-6, capturable=True)
        sim = ap.Namespace(args=args, model=net, collision_count=0, hard_collision_count=0, epoch=0, batch_idx=0)
        base = _batch_from_golden(g)
        C0 = base.position.shape[0]
        rep = (32 + C0 - 1) // C0

        def make_batch():
            b = type(base)()
            for k, v in base.__dict__.items():
                if torch.is_tensor(v) and v.dim() >= 1 and v.shape[0] == C0 and k not in ("obstacles", "dest_num"):
                    v = v.repeat(rep, *([1] * (v.dim() - 1)))[:32].clone()
                elif torch.is_tensor(v):
                    v = v.clone()
                setattr(b, k, v)
            return b

        def step():
            opt.zero_grad(set_to_none=True)
            res = TRO.test_multiple_rollouts_for_training(sim, make_batch())
            res[0].backward()
            opt.step()
            return res
        for _ in range(3):
            step()
        torch.cuda.synchronize()
        l0, t0, n = P._lib.launch_count(), time.perf_counter(), 10
        for _ in range(n):
            res = step()
        torch.cuda.synchronize()
        ms_eager = (time.perf_counter() - t0) / n * 1e3
        launches = (P._lib.launch_count() - l0) / n
        # the same step captured once into a CUDA graph (piml_b200.train_graph) and replayed per batch
        from piml_b200.train_graph import GraphedRolloutTraining
        import gc
        res = None                      # the eager steps' autograd graph (AccumulateGrad nodes bound to this stream)
        opt.zero_grad(set_to_none=True)
        gc.collect()
        graphed = GraphedRolloutTraining(sim, opt, make_batch())
        batches = [make_batch() for _ in range(n)]
        for b in batches[:2]:
            graphed.step(b)
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        for b in batches:
            res = graphed.step(b)
        torch.cuda.synchronize()
        ms = (time.perf_counter() - t0) / n * 1e3
        b = make_batch()
        C, T, N = [int(v) for v in b.position.shape[:3]]
        blk = {"workload": f"rollout-training step {kind}/{dsn}: C={C} channels x T={T} steps x N={N} slots, forward rollout + "
                           "losses + backward + Adam, the whole step replayed as ONE captured CUDA graph "
                           "(piml_b200.train_graph; batch copied into static buffers, one read-back per step)",
               "ms_per_step": ms, "agent_steps_per_sec": C * T * N / ms * 1e3, "ms_per_step_eager": ms_eager,
               "library_launches_per_step": launches, "loss": float(res[0])}
    except Exception as e:
        return {"error": f"{type(e).__name__}: {e}"[:300]}
    if with_reference and _import_reference():
        try:
            sys.path.insert(0, os.path.join(ROOT, "tests", "golden"))
            import _refharness as H
            DATA, MODEL, MLAPM_MOD, SIM, UTILS = H.import_reference()
            keep = torch.get_num_threads()
            torch.set_num_threads(len(os.sched_getaffinity(0)))
            rargs = H.default_args(model=kind, dataset_name=dsn, valid_steps=T)
            data = H.make_time_indexed(rargs, H.load_raw(H.UCY_CLIP))
            ch = DATA.ChanneledTimeIndexedPedData()
            with H.quiet():
                ch.load_from_time_indexed_peddata(data, stride=T, mode='slice')
            batch = DATA.ChanneledTimeIndexedPedData.slice(ch, slice(200, 200 + C0))
            torch.manual_seed(666)
            with H.quiet():
                rsim = SIM.BaseSimulator(rargs)
            rsim.collision_count, rsim.hard_collision_count, rsim.epoch, rsim.batch_idx = 0, 0, 0, 0
            t0 = time.perf_counter()
            with H.quiet():
                out = rsim.test_multiple_rollouts_for_training(batch)
            t1 = time.perf_counter()
            out[0].backward()
            t2 = time.perf_counter()
            torch.set_num_threads(keep)
            blk["reference_pytorch"] = {"channels": C0, "steps": T, "slots": N, "threads": len(os.sched_getaffinity(0)),
                                        "forward_s": t1 - t0, "backward_s": t2 - t1,
                                        "agent_steps_per_sec": C0 * T * N / (t2 - t0),
                                        "note": "the unmodified reference on the host cores, ONE run of the 6-channel batch "
                                                "(its C = 32, T = 10 batch takes 19.2 s + 0.48 s in the build container, "
                                                "SURVEY 8a row a12)"}
        except Exception as e:
            blk["reference_pytorch"] = {"error": f"{type(e).__name__}: {e}"[:300]}
    return blk


def run_ours(a):
    import torch
    import torch.distributed as dist
    import piml_b200 as P
    from piml_b200 import _lib as L

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device; the piml_b200 hot path has no CPU fallback")
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if world > 1:
        if a.dump_outputs:
            raise SystemExit("--dump-outputs runs on one GPU")
        dist.init_process_group("nccl", device_id=dev)
    N = a.agents
    if N % world:
        raise SystemExit(f"--agents {N} must be divisible by the number of ranks {world}")
    from piml_b200.sharded import allgather_state, shard_rows
    shard = N // world
    r0, r1 = shard_rows(N, world, rank)

    p_h, v_h, ds_h, dest_h, obs_h = [x.pin_memory() for x in synthetic_crowd(N)]
    pos, vel, ds, dest = p_h.to(dev), v_h.to(dev), ds_h.to(dev), dest_h.to(dev)
    model = P.MLAPM(**MLAPM_KW)
    flush = torch.empty(FLUSH_MB << 20, dtype=torch.uint8, device=dev)  # > 126 MB L2
    pos_next, vel_next = torch.empty_like(pos), torch.empty_like(vel)
    # Multi-GPU exchange: "push" = the finalize kernel stores each new row into every rank's next-state arrays over
    # NVLink peer memory (piml_mlapm_advance_push_f32) + one barrier; "nccl" = separate all-gathers after the step.
    crowd, exchange, exchange_note = None, "none", ""
    if world > 1:
        exchange = a.exchange
        if exchange == "push":
            try:
                from piml_b200.sharded import ShardedCrowd
                crowd = ShardedCrowd(N, device=dev)
                crowd.load(pos, vel)
            except Exception as e:                                      # no peer mapping on this box: use NCCL
                crowd, exchange, exchange_note = None, "nccl", f"push unavailable: {type(e).__name__}: {e}"[:200]
            ok = torch.tensor([1 if crowd is not None else 0], device=dev)
            dist.all_reduce(ok, op=dist.ReduceOp.MIN)
            if int(ok) == 0 and crowd is not None:
                crowd, exchange, exchange_note = None, "nccl", "push unavailable on another rank"

    arrived = None

    def advance_step():
        """One step incl. the exchange; returns nothing (state is updated in place / swapped)."""
        nonlocal pos, vel, pos_next, vel_next, arrived
        if crowd is not None:
            crowd.step(model, ds, dest, DT, RADIUS)
            return
        act, pnew, arrived = model.advance(pos, vel, ds, dest, DT, RADIUS, rows=(r0, r1))
        if world > 1:                                                   # the path's one exchange step
            allgather_state(pos_next, vel_next, pnew, act)
            pos, pos_next = pos_next, pos
            vel, vel_next = vel_next, vel
        else:
            pos, vel = pnew, act

    def step():
        flush.zero_()                                                   # L2 flush between steps
        advance_step()

    def sync_all():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    for _ in range(max(a.warmup, 3)):
        step()
    peaks = probe_peaks(L, torch, dev) if rank == 0 else {}
    sampler = ClockSampler(local) if rank == 0 else None
    if sampler:
        sampler.start()
        time.sleep(0.3)
    # ---- device-resident timed region: EXACTLY K steps --------------------------------------------------------
    sync_all()
    launches0 = L.launch_count()
    k_ev = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(a.steps)]
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for s in range(a.steps):
        flush.zero_()
        k_ev[s][0].record()
        advance_step()
        k_ev[s][1].record()
    e1.record()
    sync_all()
    launches = L.launch_count() - launches0
    ms = torch.tensor([e0.elapsed_time(e1)], device=dev)
    kernel_ms = torch.tensor([sum(x.elapsed_time(y) for x, y in k_ev) / a.steps], device=dev)
    if world > 1:
        dist.all_reduce(ms, op=dist.ReduceOp.MAX)
        dist.all_reduce(kernel_ms, op=dist.ReduceOp.MAX)
    ms, kernel_ms = float(ms), float(kernel_ms)
    final_pos = crowd.position if crowd is not None else pos
    assert torch.isfinite(final_pos).all(), "non-finite positions after the timed rollout"
    if world > 1:                       # every rank must hold the same crowd after the exchange
        chk = final_pos.double().sum().reshape(1)
        lo, hi = chk.clone(), chk.clone()
        dist.all_reduce(lo, op=dist.ReduceOp.MIN)
        dist.all_reduce(hi, op=dist.ReduceOp.MAX)
        assert float(hi - lo) == 0.0, "ranks disagree on the crowd state after the exchange"
    if a.dump_outputs:                  # one GPU: pos / vel are what the last timed MLAPM.advance returned
        dump_outputs(a.dump_outputs, {"action": vel, "new_position": pos, "arrived": arrived})

    # ---- end-to-end through the public host-buffer API ------------------------------------------------------------
    act_h = torch.empty(shard, 2).pin_memory()
    pnew_h = torch.empty(shard, 2).pin_memory()
    arr_h = torch.empty(shard, dtype=torch.bool).pin_memory()

    if crowd is not None:                  # the agent-sharded public API: host state in, this rank's rows out
        cr0, cr1 = crowd.rows
        act_h = torch.empty(cr1 - cr0, 2).pin_memory()
        pnew_h = torch.empty(cr1 - cr0, 2).pin_memory()
        arr_h = torch.empty(cr1 - cr0, dtype=torch.bool).pin_memory()

    e2e_scatter = crowd is not None
    if crowd is not None:          # this rank's rows only: pinned host slices
        own_h = [x[cr0:cr1].clone().pin_memory() for x in (p_h, v_h, ds_h, dest_h)]

    def e2e_step():
        nonlocal e2e_scatter
        if crowd is not None:
            if e2e_scatter:
                try:               # 1/G of the state over PCIe, the rest over NVLink peer stores
                    crowd.scatter_rows(own_h[0], own_h[1], own_h[3])
                    ds[cr0:cr1].copy_(own_h[2], non_blocking=True)
                    arrived = crowd.step(model, ds, crowd.dest_buf, DT, RADIUS)
                except Exception:  # no get_buffer on this torch: whole state from the host
                    e2e_scatter = False
            if not e2e_scatter:
                crowd.position.copy_(p_h, non_blocking=True); crowd.velocity.copy_(v_h, non_blocking=True)
                ds.copy_(ds_h, non_blocking=True); dest.copy_(dest_h, non_blocking=True)
                arrived = crowd.step(model, ds, dest, DT, RADIUS)
            act_h.copy_(crowd.velocity[cr0:cr1]); pnew_h.copy_(crowd.position[cr0:cr1]); arr_h.copy_(arrived)
            return
        act, pnew, arrived = model.advance(p_h, v_h, ds_h, dest_h, DT, RADIUS, rows=(r0, r1))   # host in, host out
        act_h.copy_(act); pnew_h.copy_(pnew); arr_h.copy_(arrived)
    for _ in range(2):
        e2e_step()
    sync_all()
    t0 = time.perf_counter()
    g0, g1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    g0.record()
    for _ in range(a.steps):
        e2e_step()
    g1.record()
    sync_all()
    wall = (time.perf_counter() - t0) * 1e3
    e2e_ms = torch.tensor([max(g0.elapsed_time(g1), wall)], device=dev)
    if world > 1:
        dist.all_reduce(e2e_ms, op=dist.ReduceOp.MAX)
    e2e_ms = float(e2e_ms)
    if sampler:
        sampler.stop()
    h2d = (p_h.numel() + v_h.numel() + ds_h.numel() + dest_h.numel()) * 4
    if crowd is not None and e2e_scatter:
        h2d = sum(x.numel() for x in own_h) * 4 * world          # every rank uploads its own rows only
    d2h = (act_h.numel() + pnew_h.numel()) * 4 + arr_h.numel()

    sym_used = (world == 1 and N >= 16384) or (crowd is not None and crowd.symmetric)
    nn_sharded = nn_path_sharded(torch, dist, dev, N, obs_h, world) if world > 1 else None   # collective: all ranks
    timeline = sharded_timeline(torch, dist, dev, crowd, model, ds, dest, world) if crowd is not None else None
    extra = {}
    if not a.no_config5:
        extra["crowd_1m"] = crowd_1m_block(torch, dist, dev, world, rank)
        extra["nn_crowd_1m"] = nn_crowd_1m_block(torch, dist, dev, world, rank)
        extra["scenes_4096"] = scenes_block(torch, dist, dev, world, rank)
    if rank == 0:
        pairs = float(shard) * N                       # ordered pairs one launch of the pairs kernel evaluates
        achieved = FLOP_PER_PAIR * pairs / (kernel_ms * 1e-3) / 1e12
        peak = peaks.get("fp32_tflops") or None
        line = {
            "metric": METRIC, "value": N * a.steps / (ms * 1e-3), "unit": UNIT, "n_gpus": world, "steps": a.steps,
            "warmup": max(a.warmup, 3), "ms_per_step": ms / a.steps, "higher_is_better": True, "scaling": "strong",
            "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "config": bench_config(N, world),
            "parallelism": {"mode": f"agent-sharded rows x{world}" + (
                                "" if world == 1 else (" + exchange fused into the finalize kernel (NVLink peer stores) + "
                                                       "1 barrier/step" if exchange == "push" and not sym_used else
                                                       " + symmetric evaluation: column-direction shares and new state "
                                                       "stored into the owners' buffers over NVLink peer memory by the "
                                                       "pair / finalize stages + 2 barriers/step" if exchange == "push"
                                                       else " + NCCL all-gather/step")),
                            "exchange": exchange, "exchange_note": exchange_note},
            "roofline": {"bound": "fp32",
                         "kernel": ("mlapm_sym_kernel<GC> (every unordered pair once for both rows, packed FP32; +prep, "
                                    "finalize)" if sym_used else
                                    "mlapm_pairs2_kernel<GC, packed FP32> (ordered pairs of this rank's rows; +prep, "
                                    "finalize)"),
                         "achieved": achieved, "peak": peak, "unit": "TFLOP/s",
                         "peak_nominal": 148 * 128 * 2 * 1.965e9 / 1e12,
                         "frac": (achieved / peak) if peak else None,
                         "traffic": (None if N != 100000 else MLAPM_SYM_DRAM_BYTES_PER_LAUNCH / world if sym_used
                                     else MLAPM_DRAM_BYTES_PER_LAUNCH * (shard / N)),
                         "traffic_unit": "bytes of DRAM traffic per launch (ncu dram__bytes_read+write, profiles/"
                                         "r02i_ncu_mlapm_sym_kernel.txt / r01b_ncu_mlapm_pairs2_kernel.txt); "
                                         "algorithmic work is FLOPs",
                         "note": "achieved = 51 algorithmic FLOP per ORDERED pair (SURVEY 8d) x N^2 / kernel time.  "
                                 "The symmetric kernel evaluates the n<->m-symmetric part of the formula once per "
                                 "unordered pair, so it executes fewer FLOP than the algorithmic count and the "
                                 "fraction can exceed 1; ncu: FMA pipe 66.6 % busy, MUFU 49 %, ALU 32 % "
                                 "(profiles/r02i_ncu_mlapm_sym_kernel.txt)",
                         "peak_source": "live FFMA-chain probe (piml_pipe_probe), best of 6; FP32 is not in "
                                        "MEASURED_PEAKS.json",
                         "executed": ({"fp32_lane_instructions_per_ordered_pair": 16.3,
                                       "fma_pipe_busy_ncu": 0.670, "mufu_pipe_busy_ncu": 0.488,
                                       "source": "profiles/r02i_ncu_mlapm_sym_kernel.txt (32 packed FP32 instructions "
                                                 "per 128 ordered pairs + 9 FADD per 256 and warp)"} if sym_used else
                                      {"fp32_lane_instructions_per_ordered_pair": 24.0, "fma_pipe_busy_ncu": 0.718,
                                       "source": "profiles/r01b_ncu_mlapm_pairs2_kernel.txt"}),
                         "flop_per_pair": FLOP_PER_PAIR, "pairs_per_launch": pairs, "kernel_ms": kernel_ms,
                         "pairs_per_sec": pairs / (kernel_ms * 1e-3), "mufu_peak_tops": peaks.get("mufu_tops")},
            "e2e": {"value": N * a.steps / (e2e_ms * 1e-3), "unit": UNIT, "h2d_bytes_per_step": h2d,
                    "d2h_bytes_per_step": d2h, "ms_per_step": e2e_ms / a.steps,
                    "api": ("piml_b200.MLAPM.advance(pinned host tensors) -> host tensors" if crowd is None else
                            "piml_b200.sharded.ShardedCrowd: each rank uploads ITS rows (pinned host), scatter_rows over "
                            "NVLink, step, this rank's rows out")},
            "gpu_launches": launches,
            "clocks": sampler.summary() if sampler else None,
        }
        if world == 1:
            line["nn_path"] = nn_workload(torch, dev, N, obs_h, 10, 3, with_cpu=not a.no_cpu)
            line["clip_rollouts"] = clip_rollouts_block(torch, dev)
        else:
            line["nn_path"] = nn_sharded
            line["timeline"] = timeline
        line.update(extra)
        if world == 1:
            line["training"] = training_block(torch, dev, with_reference=not a.no_cpu)
        if world == 1 and not a.no_cpu:
            line["cpu_baseline"], rows = cpu_baseline(N)
            line["parity"] = parity_block(torch, dev, N, model, rows)
            line["cpu_baseline"]["reference_pytorch"] = reference_pytorch()
        print(json.dumps(line))
    if world > 1:
        dist.destroy_process_group()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--agents", type=int, default=100000)
    ap.add_argument("--workload", default="mlapm", choices=["mlapm", "nn"],
                    help="mlapm: BASELINE configs[3] headline (MLAPM rollout); nn: the NN-augmented rollout step")
    ap.add_argument("--no-cpu", action="store_true", help="skip the cpu_baseline leg")
    ap.add_argument("--no-config5", action="store_true", help="skip the crowd_1m / scenes_4096 blocks")
    ap.add_argument("--exchange", default="push", choices=["push", "nccl"],
                    help="multi-GPU exchange: fused peer-memory push (default) or NCCL all-gather")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="after the timed steps, write what the last one returned (action, new_position, arrived) "
                         "as DIR/<name>.npy; inputs are seeded, so runs with the same arguments compare output for "
                         "output")
    a = ap.parse_args()
    if a.steps < 1:
        ap.error("--steps must be at least 1")
    if a.dump_outputs and (a.impl != "ours" or a.workload != "mlapm"):
        ap.error("--dump-outputs applies to the default workload (--impl ours --workload mlapm)")
    if a.impl == "reference":
        run_reference(a)
    elif a.workload == "nn":
        run_nn(a)
    else:
        run_ours(a)


if __name__ == "__main__":
    main()
