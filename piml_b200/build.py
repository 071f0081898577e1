"""Builds piml_b200/lib/libpiml_b200.so with nvcc for sm_100a (in-tree, so it travels to the GPU box).

    python -m piml_b200.build [--force] [--verbose]

cudart is linked statically: the library loads (and its symbols can be enumerated) on a machine without a GPU or
driver; only calling a compute entry point needs the device.
"""
import os
import subprocess
import sys

HERE = os.path.dirname(os.path.abspath(__file__))
CSRC = os.path.join(HERE, "csrc")
LIBDIR = os.path.join(HERE, "lib")
LIB = os.path.join(LIBDIR, "libpiml_b200.so")
SOURCES = ["api.cu", "features.cu", "features_cells.cu", "mlapm.cu", "mlp.cu", "mlp_bwd.cu", "mlp_tc.cu", "mlp_tc16.cu", "integrate.cu", "nn_step.cu", "losses.cu", "metrics.cu", "rollout.cu", "rollout_sfm.cu", "sfm.cu", "sfm_sweep.cu"]
NVCC_FLAGS = ["-gencode", "arch=compute_100a,code=sm_100a", "-O3", "-lineinfo", "-std=c++17",
              "-Xcompiler", "-fPIC,-fvisibility=hidden", "--expt-relaxed-constexpr", "-cudart", "static"]


def _nvcc():
    for c in (os.environ.get("NVCC"), "/usr/local/cuda/bin/nvcc", "nvcc"):
        if c and (os.path.isabs(c) and os.path.exists(c) or not os.path.isabs(c)):
            return c
    return "nvcc"


def needs_build():
    if not os.path.exists(LIB):
        return True
    t = os.path.getmtime(LIB)
    deps = [os.path.join(CSRC, f) for f in os.listdir(CSRC)] + [
        os.path.join(HERE, "..", "include", "piml_b200.h"), os.path.abspath(__file__)]
    return any(os.path.getmtime(d) > t for d in deps)


def build(force=False, verbose=False):
    if not force and not needs_build():
        return LIB
    os.makedirs(LIBDIR, exist_ok=True)
    objdir = os.path.join(HERE, "build")
    os.makedirs(objdir, exist_ok=True)
    env = dict(os.environ)
    procs = []
    for src in SOURCES:
        obj = os.path.join(objdir, src.replace(".cu", ".o"))
        cmd = [_nvcc(), *NVCC_FLAGS, "-ccbin", "/usr/bin/g++", "-c", os.path.join(CSRC, src), "-o", obj]
        if verbose:
            cmd.insert(1, "-Xptxas=-v")
        procs.append((src, obj, subprocess.Popen(cmd, env=env, stdout=subprocess.PIPE, stderr=subprocess.STDOUT)))
    objs = []
    for src, obj, p in procs:
        out = p.communicate()[0].decode()
        if p.returncode != 0:
            raise RuntimeError(f"nvcc failed on {src}:\n{out}")
        if verbose and out.strip():
            print(out)
        objs.append(obj)
    cmd = [_nvcc(), "-shared", "-cudart", "static", "-ccbin", "/usr/bin/g++", "-Xcompiler", "-fPIC",
           "-gencode", "arch=compute_100a,code=sm_100a", "-o", LIB, *objs]
    subprocess.check_call(cmd, env=env)
    return LIB


if __name__ == "__main__":
    print(build(force="--force" in sys.argv, verbose="--verbose" in sys.argv))
