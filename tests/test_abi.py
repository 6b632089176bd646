"""The C-ABI shared library loads on a box without a GPU, exports every symbol
include/mixemt_b200.h declares, and the product path fails loudly (no CPU
fallback) when no device is visible."""
import ctypes
import os
import re

import pytest

import mixemt_b200
from mixemt_b200 import _lib

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def declared_symbols():
    text = open(os.path.join(ROOT, "include", "mixemt_b200.h")).read()
    text = re.sub(r"/\*.*?\*/", "", text, flags=re.S)
    return sorted(set(re.findall(r"\b(mxb_[a-z0-9_]+)\s*\(", text)))


def test_header_symbols_are_exported():
    names = declared_symbols()
    assert len(names) >= 30
    for name in names:
        assert hasattr(_lib.lib, name), "libmixemt_b200.so does not export %s" % name


def test_python_prototypes_cover_the_header():
    assert sorted(_lib.EXPORTED_SYMBOLS) == declared_symbols()


def test_abi_version_2_and_error_string():
    """Version 2: mxb_build_matrix takes route_host after match_host."""
    assert _lib.lib.mxb_abi_version() == 2
    assert isinstance(_lib.last_error(), str)


def test_argument_errors_do_not_need_a_gpu():
    rc = _lib.lib.mxb_sig_count(None, None, -1, None)
    assert rc == _lib.MXB_ERR_ARG
    with pytest.raises(_lib.MixemtB200Error):
        _lib.check(rc)
    assert "mxb_sig_count" in _lib.last_error()


def test_no_cpu_fallback_without_device():
    if _lib.lib.mxb_device_count() > 0:
        pytest.skip("a GPU is visible")
    import numpy as np
    from conftest import make_args
    handle = ctypes.c_void_p()
    assert _lib.lib.mxb_ctx_create(0, ctypes.byref(handle)) != _lib.MXB_OK
    with pytest.raises(_lib.MixemtB200Error):
        mixemt_b200.run_em(np.zeros((2, 2)), np.ones(2), make_args())
    with pytest.raises(_lib.MixemtB200Error):
        mixemt_b200.em_step(np.zeros((2, 2)), np.ones(2), np.log([0.5, 0.5]), np.zeros((2, 2)))


def test_product_package_never_imports_the_oracle():
    pkg = os.path.join(ROOT, "mixemt_b200")
    for dirpath, _, files in os.walk(pkg):
        for name in files:
            if name.endswith((".py", ".cu", ".cuh", ".cpp", ".h")):
                text = open(os.path.join(dirpath, name)).read()
                assert not re.search(r"^\s*(from|import)\s+oracle\b", text, flags=re.M), name
                assert "liboracle" not in text, name
