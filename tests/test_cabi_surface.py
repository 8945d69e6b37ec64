"""The C-ABI library loads without a GPU and exports every function include/fmb200.h declares (no compute calls here)."""
import ctypes
import os
import re

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _declared_functions():
    src = open(os.path.join(ROOT, "include", "fmb200.h")).read()
    src = re.sub(r"/\*.*?\*/", "", src, flags=re.S)
    names = re.findall(r"\b(fmb_[A-Za-z0-9_]+)\s*\(", src)
    return sorted(set(names))


def test_library_exports_every_declared_symbol():
    import fmb200
    from fmb200 import capi
    declared = _declared_functions()
    assert len(declared) >= 40
    lib = ctypes.CDLL(fmb200.lib_path())
    missing = [n for n in declared if not hasattr(lib, n)]
    assert not missing, f"declared in fmb200.h but not exported: {missing}"
    # the Python binding's list (used by __graft_entry__.build) covers the header too
    assert set(capi.SYMBOLS) == set(declared), sorted(set(capi.SYMBOLS) ^ set(declared))


def test_no_cpu_fallback_without_device():
    """without a CUDA device every compute entry point fails loudly with FMB_ENODEVICE (in a fresh process that sees no device,
    so that the check also runs where a GPU is present)"""
    import subprocess
    import sys
    code = ("import sys; sys.path.insert(0, %r)\n"
            "import numpy as np, fmb200\n"
            "assert fmb200.device_count() == 0\n"
            "try:\n"
            "    fmb200.Index.build(5, np.array([1, 2, 3, 0], dtype=np.uint8))\n"
            "except fmb200.FmbError as e:\n"
            "    print(e.code, e)\n") % ROOT
    r = subprocess.run([sys.executable, "-c", code], env=dict(os.environ, CUDA_VISIBLE_DEVICES=""), capture_output=True, text=True, timeout=300)
    assert r.returncode == 0, r.stdout + r.stderr
    assert r.stdout.startswith("-2 ") and "no CPU fallback" in r.stdout, r.stdout


def test_product_never_imports_the_oracle():
    """oracle/ is test infrastructure: nothing under the package or include/ may reference it"""
    bad = []
    for base in ("fmindex-collection_b200", "include"):
        for root, _, files in os.walk(os.path.join(ROOT, base)):
            if os.path.basename(root) in ("build", "__pycache__"):
                continue
            for f in files:
                if not f.endswith((".py", ".cu", ".cuh", ".hpp", ".h")):
                    continue
                text = open(os.path.join(root, f), errors="ignore").read()
                if re.search(r"fm_oracle|pyoracle|libfmoracle|libfmref|from oracle|import oracle", text):
                    bad.append(os.path.join(root, f))
    assert not bad, bad
