"""CPU-side checks of the drop-in boundary: libusip_b200.so loads without a GPU, exports every symbol that
include/usip_b200.h declares, and the ctypes binding covers exactly that set (no compute calls here)."""
import ctypes
import os
import re

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _declared():
    src = open(os.path.join(ROOT, "include", "usip_b200.h")).read()
    src = re.sub(r"/\*.*?\*/", "", src, flags=re.S)
    return sorted(set(re.findall(r"\b(usip_[a-z0-9_]+)\s*\(", src)))


def test_header_symbols_exported_and_bound():
    from usip_b200 import _lib
    lib = _lib.load()
    declared = _declared()
    assert len(declared) >= 20
    for name in declared:
        assert hasattr(lib, name), "declared in usip_b200.h but not exported: " + name
    assert sorted(_lib.SIGNATURES) == declared, (set(declared) ^ set(_lib.SIGNATURES))
    assert lib.usip_abi_version() == 1
    assert lib.usip_layer_tile_rows() == 128


def test_layer_desc_layout_matches_c_struct():
    """sizeof/offsets of the ctypes mirror must match the C struct (compiled with gcc here)."""
    import subprocess, tempfile
    from usip_b200._lib import LayerDesc
    prog = r'''
#include <stdio.h>
#include <stddef.h>
#include "usip_b200.h"
int main(){ printf("%zu %zu %zu %zu %zu %zu\n", sizeof(usip_layer_desc), offsetof(usip_layer_desc, W),
  offsetof(usip_layer_desc, addend), offsetof(usip_layer_desc, Y), offsetof(usip_layer_desc, gmax),
  offsetof(usip_layer_desc, precision)); return 0; }'''
    with tempfile.TemporaryDirectory() as td:
        c = os.path.join(td, "t.c"); exe = os.path.join(td, "t")
        open(c, "w").write(prog)
        subprocess.check_call(["gcc", "-I", os.path.join(ROOT, "include"), c, "-o", exe])
        out = [int(v) for v in subprocess.check_output([exe]).split()]
    assert out == [ctypes.sizeof(LayerDesc), LayerDesc.W.offset, LayerDesc.addend.offset, LayerDesc.Y.offset,
                   LayerDesc.gmax.offset, LayerDesc.precision.offset]


def test_product_path_fails_loudly_without_cuda():
    import torch
    if torch.cuda.is_available():
        pytest.skip("GPU present")
    from usip_b200 import index_max
    with pytest.raises(RuntimeError):
        index_max.forward_cuda_shared_mem(torch.zeros(1, 1, 4), torch.zeros(1, 4, dtype=torch.int32), 2)


def test_product_code_never_imports_oracle():
    """oracle/ is test infrastructure: nothing under usip_b200/ may import or execute it."""
    pkg = os.path.join(ROOT, "usip_b200")
    for dp, _, fs in os.walk(pkg):
        for f in fs:
            if f.endswith((".py", ".cu", ".cuh", ".h")):
                txt = open(os.path.join(dp, f)).read()
                assert not re.search(r"^\s*(from|import)\s+oracle\b", txt, flags=re.M), os.path.join(dp, f)
                assert "usip_oracle" not in txt or f == "index_max.py", os.path.join(dp, f)


def test_only_ops_calls_the_c_abi():
    """ops.py is the one module that knows the C calling convention: no other Python module of the package calls a usip_*
    entry point (_lib.py only loads the library and reads its error), and ops.py wraps every launch entry point."""
    from usip_b200 import _lib
    pkg = os.path.join(ROOT, "usip_b200")
    for dp, _, fs in os.walk(pkg):
        for f in fs:
            path = os.path.join(dp, f)
            if f.endswith(".py") and os.path.relpath(path, pkg) not in ("ops.py", "_lib.py"):
                assert not re.search(r"\busip_[a-z0-9_]+\(", open(path).read()), path
    ops_src = open(os.path.join(pkg, "ops.py")).read()
    host_only = ("_abi_version", "_last_error", "_scratch_bytes", "_tile_rows", "_stat_slots", "_tc_workspace_bytes")
    unwrapped = [n for n in _lib.SIGNATURES if not n.endswith(host_only) and not re.search(r"\b%s\(" % n, ops_src)]
    assert not unwrapped, unwrapped
