"""The C-ABI shared library loads and exports every symbol include/fem_b200.h declares (no compute calls)."""
import os
import re

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def header_symbols():
    src = open(os.path.join(ROOT, "include", "fem_b200.h")).read()
    src = re.sub(r"/\*.*?\*/", "", src, flags=re.S)
    return sorted(set(re.findall(r"\b(fem_[a-z0-9_]+)\s*\(", src)))


def test_library_exports_every_header_symbol():
    from fem_elastoplasticity_b200 import _lib
    if not os.path.isfile(_lib.LIB_PATH):
        import __graft_entry__
        __graft_entry__.build()
    lib = _lib.load()
    names = header_symbols()
    assert len(names) >= 25
    for n in names:
        assert hasattr(lib, n), f"{n} declared in fem_b200.h but not exported"
        assert n in _lib.SIGNATURES, f"{n} has no ctypes signature"
    assert set(_lib.SIGNATURES) <= set(names)
    assert lib.fem_version() >= 100


def test_set_tuning_rejects_removed_kernel_selections():
    """Keys and values that selected deleted assembly, strain and return-map kernels fail loudly instead of silently timing
    the default kernel; the kept assembly variants are still accepted."""
    from fem_elastoplasticity_b200 import _lib
    if not os.path.isfile(_lib.LIB_PATH):
        import __graft_entry__
        __graft_entry__.build()
    lib = _lib.load()
    try:
        for key, value in ((b"assemble_variant", 7), (b"assemble_variant", 8), (b"assemble_canon", 3), (b"assemble_warps", 4),
                           (b"strain_variant", 2), (b"return_map_variant", 1)):
            assert lib.fem_set_tuning(key, value) != 0, (key, value)
        for value in (0, 1, 2, 6):
            assert lib.fem_set_tuning(b"assemble_variant", value) == 0, value
        for value in (0, 2):
            assert lib.fem_set_tuning(b"assemble_canon", value) == 0, value
    finally:
        assert lib.fem_set_tuning(b"assemble_variant", 0) == 0
        assert lib.fem_set_tuning(b"assemble_canon", 0) == 0


def test_no_cpu_fallback_without_device():
    """Without a CUDA device the product path must fail loudly (never fall back to the oracle / CPU)."""
    import torch
    if torch.cuda.is_available():
        pytest.skip("CUDA device present")
    import numpy as np
    from fem_elastoplasticity_b200 import pythonFEM, plan
    with pytest.raises(RuntimeError, match="no CPU fallback"):
        plan.FemPlan(np.array([[0], [1], [2]]), np.array([[0.0, 1.0, 0.0], [0.0, 0.0, 1.0]]),
                     np.array([[-1], [1], [0]]), np.array([[-1], [0], [1]]), np.array([[0.5]]))
    with pytest.raises(RuntimeError):
        pythonFEM.construct_constitutive_problem(np.zeros((3, 4)), np.zeros((4, 4)), np.ones(4), np.ones(4), np.ones(4), np.ones(4))


def test_product_package_never_imports_oracle():
    pkg = os.path.join(ROOT, "fem_elastoplasticity_b200")
    for dirpath, _, files in os.walk(pkg):
        for f in files:
            if f.endswith(".py"):
                txt = open(os.path.join(dirpath, f)).read()
                assert not re.search(r"^\s*(from|import)\s+oracle\b", txt, flags=re.M), f
