"""CPU: the C-ABI shared library loads, exports every entry point include/maro_b200.h declares (and nothing in the
loader's list is missing from the header), and refuses to create a handle without a GPU instead of falling back."""
import ctypes as C
import os
import re
import subprocess
import sys

from maro_b200 import _abi, _native

ROOT = os.path.abspath(os.path.join(os.path.dirname(__file__), ".."))


def _declared():
    text = open(os.path.join(ROOT, "include", "maro_b200.h")).read()
    text = re.sub(r"/\*.*?\*/", "", text, flags=re.S)  # comments mention entry points too
    return set(re.findall(r"\b(maro_[a-z0-9_]+)\s*\(", text))


def test_header_and_loader_agree():
    declared = _declared()
    assert declared == set(_native.EXPORTS), (sorted(declared - set(_native.EXPORTS)), sorted(set(_native.EXPORTS) - declared))
    assert len(declared) >= 60


def test_library_loads_and_exports_every_declared_symbol():
    L = _native.lib()  # raises NativeLibraryError if the library has not been built
    raw = C.CDLL(_native.LIB_PATH)
    for name in sorted(_declared()):
        assert hasattr(raw, name), name
    assert L.maro_abi_version() == _abi.ABI_VERSION
    assert L.maro_last_error() is not None


def test_create_without_a_gpu_fails_loudly():
    """in a child process that sees no CUDA device (CUDA_VISIBLE_DEVICES=""), so that it runs on GPU machines too"""
    code = ("import pytest\n"
            "from maro_b200.batch import CimBatch\n"
            "from maro_b200.scenarios.cim.topology import build_topology\n"
            "with pytest.raises(RuntimeError, match='no CUDA device'):\n"
            "    CimBatch(build_topology('toy.4p_ssdd_l0.0', 20), 2)\n")
    p = subprocess.run([sys.executable, "-c", code], cwd=ROOT, env=dict(os.environ, CUDA_VISIBLE_DEVICES=""),
                       capture_output=True, text=True, timeout=300)
    assert p.returncode == 0, p.stderr[-3000:]


def test_product_package_never_imports_the_oracle():
    pkg = os.path.join(ROOT, "maro_b200")
    for base, _, files in os.walk(pkg):
        for f in files:
            if f.endswith((".py", ".cu", ".cuh", ".hpp")):
                src = open(os.path.join(base, f), errors="ignore").read()
                assert not re.search(r"^\s*(from|import)\s+oracle\b", src, flags=re.M), os.path.join(base, f)
                assert not re.search(r"#include\s+\"[^\"]*oracle", src), os.path.join(base, f)
