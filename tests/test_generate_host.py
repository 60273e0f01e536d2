"""rwkv_b200_generate without a GPU: the symbol is exported and declared, a call without a loaded model fails with a
message instead of crashing, and the pybind module exposes `generate`."""
import ctypes
import importlib
import os
import sys

import pytest

from util import PKG_DIR


def test_generate_is_exported_and_declared(pkg):
    lib = pkg.load_library()
    assert "rwkv_b200_generate" in lib._declared
    assert lib.rwkv_b200_generate.restype is ctypes.c_int


def test_generate_fails_cleanly_without_a_model(pkg):
    lib = pkg.load_library()
    out = (ctypes.c_ulonglong * 4)()
    n = ctypes.c_ulonglong(99)
    u = (ctypes.c_double * 4)(0.1, 0.2, 0.3, 0.4)
    rc = lib.rwkv_b200_generate(None, 1, 4, 1, 0.9, u, None, 0, out, ctypes.byref(n), None)
    assert rc != 0
    assert lib.rwkv_b200_last_error()


def test_engine_cannot_be_built_for_generate_without_cuda(pkg, make_model):
    """No model loads without a device (the constructor refuses), so there is nothing to call generate on."""
    lib = pkg.load_library()
    if lib.rwkv_b200_device_count() > 0:
        pytest.skip("a CUDA device is visible")
    with pytest.raises(pkg.EngineError, match="no CUDA device|no CPU fallback"):
        pkg.Engine(make_model(1, 64)).generate(1, 4, pkg.engine.GEN_GREEDY)


def test_pybind_exposes_generate(pkg):
    assert pkg.build.build_pybind()
    d = os.path.join(PKG_DIR, "bindings", "pybind")
    if d not in sys.path:
        sys.path.insert(0, d)
    os.environ["SO_LIB_PATH"] = "rwkv"
    binding = importlib.import_module("binding")
    assert "generate" in dir(binding.CPP_LIB)
    assert callable(binding.ModelWrapper.generate)
