"""The C-ABI library loads and exports every symbol include/motifs_b200.h declares (no compute calls: CPU box)."""
import ctypes
import os
import re
import subprocess
import sys

import motifs_jl_b200 as mb

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def declared_symbols():
    src = open(os.path.join(ROOT, "include", "motifs_b200.h")).read()
    src = re.sub(r"/\*.*?\*/", "", src, flags=re.S)
    return sorted(set(re.findall(r"\b(mb200_[a-z0-9_]+)\s*\(", src)))


def test_header_symbols_are_exported():
    lib = ctypes.CDLL(mb.library_path())
    names = declared_symbols()
    assert len(names) >= 13
    for n in names:
        assert hasattr(lib, n), f"{n} declared in include/motifs_b200.h but not exported"


def test_binding_covers_header():
    lib = mb._lib.load()
    for n in declared_symbols():
        assert getattr(lib, n).argtypes is not None, f"{n} has no ctypes signature in _lib.py"
    assert lib.mb200_version() >= 100


def test_no_device_fails_loudly():
    """No CPU fallback: without a CUDA device the context cannot be created.  Checked in a child process that sees no
    device (CUDA_VISIBLE_DEVICES empty), so it holds on a GPU machine as well."""
    code = "import pytest, motifs_jl_b200 as mb\nwith pytest.raises(mb.MB200Error):\n    mb.Context(0)\n"
    env = dict(os.environ, CUDA_VISIBLE_DEVICES="", PYTHONPATH=os.pathsep.join(filter(None, [ROOT, os.environ.get("PYTHONPATH")])))
    r = subprocess.run([sys.executable, "-c", code], cwd=ROOT, env=env, capture_output=True, text=True, timeout=300)
    assert r.returncode == 0, r.stdout + r.stderr


def test_product_does_not_import_oracle():
    pkg = os.path.join(ROOT, "motifs.jl_b200")
    for dirpath, _, files in os.walk(pkg):
        for f in files:
            if f.endswith((".py", ".cu", ".cuh", ".h", ".cpp")):
                txt = open(os.path.join(dirpath, f)).read()
                assert not re.search(r"^\s*(from|import)\s+oracle\b", txt, flags=re.M), f"{f} imports the oracle"
                assert "liboracle" not in txt, f"{f} references the oracle library"
