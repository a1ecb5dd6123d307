"""The C-ABI library builds for sm_100a without a GPU, loads, and exports every declared symbol."""
import ctypes
import os
import re

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _declared_symbols():
    text = open(os.path.join(ROOT, "include", "nlml_hpe_b200.h")).read()
    text = re.sub(r"/\*.*?\*/", "", text, flags=re.S)
    return sorted(set(re.findall(r"\b(nlml_[a-z0-9_]+)\s*\(", text)))


def test_header_declares_expected_entry_points():
    syms = _declared_symbols()
    for s in ("nlml_tucker_plan_create", "nlml_tucker_fit_f32", "nlml_tucker_fit_host_f32",
              "nlml_mlp_plan_create", "nlml_mlp_forward_f32", "nlml_mlp_forward_host_f32"):
        assert s in syms


def test_library_exports_every_declared_symbol(cuda_lib):
    for s in _declared_symbols():
        assert hasattr(cuda_lib, s), f"{s} declared in include/nlml_hpe_b200.h but not exported"
    from nlml_hpe_b200 import _lib
    assert sorted(_lib.EXPORTS) == _declared_symbols()
    assert cuda_lib.nlml_abi_version() == 1


def test_library_is_sm100a_only(cuda_lib):
    import subprocess
    from nlml_hpe_b200 import _build
    cuobjdump = os.path.join(os.path.dirname(_build._nvcc()), "cuobjdump")   # the toolkit that built the library, on PATH or not
    out = subprocess.run([cuobjdump, "-lelf", _build.LIB_PATH], capture_output=True, text=True).stdout
    archs = set(re.findall(r"sm_\d+a?", out))
    assert archs == {"sm_100a"}, archs


def test_no_cpu_fallback_without_device(cuda_lib):
    """On a box without a GPU every compute entry point must fail loudly (no oracle, no CPU path)."""
    import torch
    if torch.cuda.is_available():
        pytest.skip("GPU present")
    W = np.zeros((5, 3, 3, 3, 8), np.float32)
    rows = np.zeros((3, 4), np.float64)
    h = ctypes.c_void_p()
    rc = cuda_lib.nlml_tucker_plan_create(W.ctypes.data, 5, 3, 3, 3, 8, rows.ctypes.data, rows.ctypes.data,
                                          rows.ctypes.data, 0, ctypes.byref(h))
    assert rc == -2 and not h.value
    assert b"no CPU fallback" in cuda_lib.nlml_last_error()
    from nlml_hpe_b200 import TD_Tester, _lib
    with pytest.raises(_lib.NlmlError):
        TD_Tester.optimize_with_sgd(W, np.zeros(8, np.float32), None, 5, rows, rows, rows)


def test_product_never_imports_oracle():
    """The shipped package must not reference oracle/ or the host-check build."""
    pkg = os.path.join(ROOT, "nlml_hpe_b200")
    for dirpath, _, files in os.walk(pkg):
        for f in files:
            if f.endswith((".py", ".cu", ".cuh", ".h")):
                text = open(os.path.join(dirpath, f)).read()
                assert not re.search(r"^\s*(from|import)\s+oracle\b", text, flags=re.M), f
                assert "hostcheck" not in text or f in ("tucker_math.h", "powell_math.h"), f   # headers the host-check build compiles too (comments only)
