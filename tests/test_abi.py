"""CPU-side checks of the drop-in boundary: libpiml_b200.so loads without a GPU and exports exactly the entry points
include/piml_b200.h declares; the ctypes table covers all of them; calling compute without a GPU fails loudly."""
import os
import re

import pytest
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def header_symbols():
    src = open(os.path.join(ROOT, "include", "piml_b200.h")).read()
    src = re.sub(r"/\*.*?\*/", "", src, flags=re.S)
    return sorted(set(re.findall(r"\b(piml_[a-z0-9_]+)\s*\(", src)))


def test_library_loads_and_exports_every_declared_symbol():
    from piml_b200 import _lib
    lib = _lib.load()
    syms = header_symbols()
    assert len(syms) >= 14
    for s in syms:
        assert hasattr(lib, s), f"{s} declared in include/piml_b200.h but not exported"
    assert sorted(_lib.SIGNATURES) == syms, "ctypes table and header disagree"
    assert lib.piml_version() >= 100
    assert lib.piml_mlapm_workspace_bytes(1000) > 0
    assert _lib.launch_count() >= 0


def test_no_cpu_fallback(monkeypatch):
    import piml_b200 as P
    monkeypatch.setattr(torch.cuda, "is_available", lambda: False)      # a machine without a GPU, also on a GPU box
    x = torch.zeros(1, 4, 2)
    with pytest.raises(RuntimeError, match="no CPU fallback"):
        P.Pedestrians().get_relative_features(x, x.clone(), x.clone(), x, torch.zeros(2, 2), 6, 90, 4, 10, 90, 4)
    with pytest.raises(RuntimeError, match="no CPU fallback"):
        P.MLAPM(version='GC', tau=0.5, A=1, B=-1, C=0, D=0, theta=0).step(x[0], x[0], x[0], x[0], 0.08)


def test_product_never_imports_oracle():
    """The oracle is test infrastructure: nothing under piml_b200/ may import, load or link it."""
    pkg = os.path.join(ROOT, "piml_b200")
    pat = re.compile(r"^\s*(from|import)\s+oracle\b|liboracle|piml_oracle|orc_[a-z_]+\(", re.M)
    for dirpath, _, files in os.walk(pkg):
        for f in files:
            if f.endswith((".py", ".cu", ".cuh", ".h")):
                text = open(os.path.join(dirpath, f)).read()
                assert not pat.search(text), f"{f} uses the oracle"
