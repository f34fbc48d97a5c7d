# coding=utf-8
"""CPU-side checks of the drop-in boundary: libtfgk.so loads and exports every symbol include/tfgk.h declares,
the ctypes table matches the header, and the product refuses to run without a GPU (no silent fallback)."""
import ctypes
import os
import re

import numpy as np
import pytest
import torch

import tf_geometric_b200 as tfg
from tf_geometric_b200 import _ffi

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _header_functions():
    text = open(os.path.join(ROOT, "include", "tfgk.h")).read()
    text = re.sub(r"/\*.*?\*/", "", text, flags=re.S)
    return re.findall(r"\b(?:int|const char \*)\s*(tfgk_\w+)\s*\(([^;]*?)\)\s*;", text, flags=re.S)


def test_library_is_built_and_loads():
    assert os.path.exists(_ffi.library_path()), "run __graft_entry__.build() first"
    lib = _ffi.lib()
    assert lib.tfgk_version() == _ffi.ABI_VERSION


def test_every_declared_symbol_is_exported_and_bound():
    decl = _header_functions()
    names = [n for n, _ in decl]
    assert len(names) >= 25
    handle = ctypes.CDLL(_ffi.library_path())
    for name in names:
        assert hasattr(handle, name), "{} declared in include/tfgk.h but not exported".format(name)
    bound = set(_ffi.SIGNATURES) | {"tfgk_last_error"}
    assert set(names) == bound, "header vs ctypes table differ: {}".format(set(names) ^ bound)


def test_ctypes_arity_matches_header():
    for name, args in _header_functions():
        if name == "tfgk_last_error":
            continue
        n_args = 0 if args.strip() in ("", "void") else len([a for a in args.split(",") if a.strip()])
        assert n_args == len(_ffi.SIGNATURES[name]), "{}: header has {} args, ctypes table {}".format(
            name, n_args, len(_ffi.SIGNATURES[name]))


def test_argument_validation_without_gpu():
    """Entry points validate arguments before touching the device, so these run on a CPU-only box."""
    lib = _ffi.lib()
    out = ctypes.c_size_t()
    assert lib.tfgk_csr_workspace_bytes(1000, 10, ctypes.byref(out)) == 0 and out.value > 0
    assert lib.tfgk_csr_workspace_bytes(-1, 10, ctypes.byref(out)) == 1
    assert b"E" in lib.tfgk_last_error()
    assert lib.tfgk_gemm_workspace_bytes(100, 128, 1 << 20, ctypes.byref(out)) == 0 and out.value > 0
    assert lib.tfgk_spmm_f32(None, None, None, None, 0, -1, 4, 0, 1.0, None, 0, 0.0, None, 0, None, 0, None, None) == 1
    assert lib.tfgk_spmm_f32(None, None, None, None, 0, 5, 4, 7, 1.0, None, 0, 0.0, None, 0, None, 0, None, None) == 1


@pytest.mark.skipif(torch.cuda.is_available(), reason="only meaningful on a CPU-only machine")
def test_operators_fail_loudly_without_gpu():
    x = np.ones((4, 3), dtype=np.float32)
    ei = np.array([[0, 1], [1, 2]], dtype=np.int32)
    with pytest.raises(RuntimeError, match="no CPU fallback"):
        tfg.nn.aggregate_neighbors(x, ei)
    with pytest.raises(RuntimeError, match="no CPU fallback"):
        tfg.nn.segment_softmax(np.ones(2, np.float32), np.array([0, 0]), 1)
    with pytest.raises(RuntimeError, match="no CPU fallback"):
        tfg.layers.GCN(4)([x, ei])


def test_product_never_imports_the_oracle():
    pkg = os.path.join(ROOT, "tf_geometric_b200")
    for dirpath, _, files in os.walk(pkg):
        for f in files:
            if f.endswith((".py", ".cu", ".cuh", ".h")):
                text = open(os.path.join(dirpath, f)).read()
                assert "oracle" not in text.lower() or f in ("index_ops.cu", "__init__.py") and "import" not in \
                    [l for l in text.lower().splitlines() if "oracle" in l][0], \
                    "{} mentions the oracle".format(os.path.join(dirpath, f))


def test_kernel_library_reads_no_environment_variable():
    """Which kernel runs is decided from what the call can observe (shape, alignment, buffer layout), never from the
    environment: a user-set variable must not change results or speed."""
    csrc = os.path.join(ROOT, "tf_geometric_b200", "csrc")
    for f in sorted(os.listdir(csrc)):
        if f.endswith((".cu", ".cuh", ".h")):
            text = open(os.path.join(csrc, f)).read()
            assert "getenv" not in text, "{} reads an environment variable".format(f)
