"""CPU: the C-ABI library builds, loads and exports every symbol include/codlad_b200.h declares
(no compute calls -- there is no GPU here), and the product path refuses to run without CUDA."""
import os
import re

import pytest
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def declared_symbols():
    text = "".join(open(os.path.join(ROOT, "include", h)).read() for h in ("codlad_b200.h", "codlad_b200_train.h"))
    return sorted(set(re.findall(r"CB2_API[^;(]*?\b(cb2t?_\w+)\s*\(", text)))


def test_header_and_binding_agree():
    from codlad_b200 import _native
    names = declared_symbols()
    assert len(names) >= 20
    assert sorted(_native.SIGNATURES) == names


def test_library_builds_loads_and_exports_all_symbols():
    from codlad_b200 import _native, build
    path = build.build()
    assert os.path.exists(path)
    lib = _native.lib()          # resolves every symbol in SIGNATURES or raises
    assert lib.cb2_abi_version() == _native.ABI_VERSION
    import ctypes
    raw = ctypes.CDLL(path)
    for name in declared_symbols():
        assert hasattr(raw, name), name


def test_sass_contains_only_sm100a():
    import subprocess
    from codlad_b200 import build
    cuobjdump = os.path.join(os.path.dirname(build.NVCC), "cuobjdump")      # the toolkit that built the library, whatever PATH says
    out = subprocess.run([cuobjdump, "-lelf", build.build()], capture_output=True, text=True, check=True).stdout
    archs = set(re.findall(r"sm_\d+a?", out))
    assert archs == {"sm_100a"}, archs


@pytest.mark.skipif(torch.cuda.is_available(), reason="checks the no-GPU failure mode")
def test_no_cpu_fallback():
    from codlad_b200 import engine, weights
    with pytest.raises(RuntimeError, match="no CPU fallback"):
        engine.DenoiserEngine(weights.init_denoiser_state(0))
    with pytest.raises(RuntimeError, match="no CPU fallback"):
        engine.knn_topk(torch.zeros(1, 4, 3), None, 4)


def test_product_package_never_imports_the_oracle():
    pkg = os.path.join(ROOT, "codlad_b200")
    for dirpath, _, files in os.walk(pkg):
        for f in files:
            if f.endswith((".py", ".cu", ".cuh", ".h")):
                src = open(os.path.join(dirpath, f)).read()
                assert not re.search(r"^\s*(from|import)\s+oracle", src, re.M), f
                assert "/root/reference" not in src, f
