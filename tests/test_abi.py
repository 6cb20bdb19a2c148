"""CPU-side checks of the C-ABI boundary: the library loads and exports every symbol the header declares
(no compute calls), struct layouts agree, and the product fails loudly without a GPU."""
import ctypes as C
import os
import re
import subprocess

import numpy as np
import pytest

from conftest import ROOT

HEADER = os.path.join(ROOT, "include", "daisyworld_b200.h")


@pytest.fixture(scope="module")
def lib():
    from therldaisyworld_b200 import build, _lib
    build.build()
    return _lib.load()


HEADER_TILED = os.path.join(ROOT, "include", "daisyworld_b200_tiled.h")


def header_symbols(path=HEADER, prefix="dw_"):
    src = open(path).read()
    src = re.sub(r"/\*.*?\*/", "", src, flags=re.S)
    return sorted(set(re.findall(r"\b(" + prefix + r"[A-Za-z0-9_]+)\s*\(", src)))


def test_library_exports_every_declared_symbol(lib):
    from therldaisyworld_b200 import _lib
    declared = header_symbols()
    assert declared, "no symbols parsed from the header"
    assert sorted(_lib.SYMBOLS) == declared, "therldaisyworld_b200/_lib.py and the header disagree"
    out = subprocess.check_output(["nm", "-D", "--defined-only", _lib.LIB_PATH], text=True)
    exported = set(re.findall(r"\bT (dw_[A-Za-z0-9_]+)", out))
    assert set(declared) <= exported, f"missing: {set(declared) - exported}"
    assert lib.dw_abi_version() == 3
    tiled = header_symbols(HEADER_TILED, "dwt_")
    assert tiled and sorted(_lib.TILED_SYMBOLS) == tiled, "_lib.py and daisyworld_b200_tiled.h disagree"
    exported_t = set(re.findall(r"\bT (dwt_[A-Za-z0-9_]+)", out))
    assert set(tiled) <= exported_t, f"missing: {set(tiled) - exported_t}"


def test_struct_layouts_match_header():
    from therldaisyworld_b200._lib import DwClock, DwConfig, DwRunResult, DwtPtrs
    assert C.sizeof(DwtPtrs) == 7 * 8
    assert C.sizeof(DwConfig) == 4 * 4 + 13 * 8 + 27 * 8
    assert C.sizeof(DwClock) == 5 * 8 + 2 * 8 + 2 * 4
    assert C.sizeof(DwRunResult) == 24
    assert DwConfig.daisy_kernel.offset == 16 + 13 * 8


def test_sass_is_sm100a_only(lib):
    from therldaisyworld_b200 import _lib
    out = subprocess.check_output(["cuobjdump", "-lelf", _lib.LIB_PATH], text=True)
    archs = set(re.findall(r"sm_(\d+a?)", out))
    assert archs == {"100a"}, archs


def test_no_cpu_fallback_without_gpu(lib):
    import torch
    if torch.cuda.is_available():
        pytest.skip("GPU present")
    from therldaisyworld_b200 import RLDaisyWorld, DaisyWorldError
    with pytest.raises(DaisyWorldError):
        RLDaisyWorld()


def test_product_does_not_import_oracle():
    """The oracle is test infrastructure: nothing under therldaisyworld_b200/ may reference it."""
    pkg = os.path.join(ROOT, "therldaisyworld_b200")
    for dirpath, _, files in os.walk(pkg):
        for f in files:
            if f.endswith((".py", ".cu", ".cuh", ".inl", ".h")):
                text = open(os.path.join(dirpath, f)).read()
                assert not re.search(r"^\s*(from|import)\s+oracle", text, flags=re.M), f
                assert "daisy_oracle" not in text, f


def test_headers_are_plain_c(tmp_path):
    """The boundary is a C ABI: both headers must compile as C99 on their own (no C++-isms, no CUDA or torch types)."""
    src = tmp_path / "use_headers.c"
    src.write_text('#include "daisyworld_b200.h"\n#include "daisyworld_b200_tiled.h"\n'
                   "int probe(dw_handle *h, dwt_handle *t) { dw_config c; dw_clock k; dwt_ptrs p; (void)c; (void)k; (void)p;\n"
                   "  return dw_abi_version() + (h != 0) + (t != 0) + DW_POLICY_MLP + DW_MLP_PARAMS + DWT_PEER_BUFFERS; }\n")
    subprocess.check_call(["gcc", "-std=c99", "-Wall", "-Werror", "-pedantic", "-fsyntax-only", "-I", os.path.join(ROOT, "include"), str(src)])
