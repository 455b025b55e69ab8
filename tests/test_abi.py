"""CPU suite: the C-ABI library loads and exports every symbol include/accmsm.h declares; without a GPU the
product refuses to run (no CPU fallback)."""
import ctypes as C
import os
import re
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def header_symbols():
    text = open(os.path.join(ROOT, "include", "accmsm.h")).read()
    text = re.sub(r"/\*.*?\*/", "", text, flags=re.S)
    return sorted(set(re.findall(r"\b(accmsm_[a-z0-9_]+)\s*\(", text)))


def test_header_and_loader_agree():
    from accumulation_b200._lib import SYMBOLS
    assert sorted(SYMBOLS) == header_symbols()


def test_library_exports_every_declared_symbol():
    from accumulation_b200 import build
    so = build.build()
    lib = C.CDLL(so)
    for name in header_symbols():
        assert hasattr(lib, name), name
    lib.accmsm_strerror.restype = C.c_char_p
    assert lib.accmsm_strerror(0) == b"ok"
    assert b"CUDA" in lib.accmsm_strerror(-1)


def test_no_cpu_fallback_without_gpu():
    """Context() raises AccmsmError in a process that sees no CUDA device (every device hidden, so the refusal is
    observable on a machine with a GPU too)"""
    code = ("import accumulation_b200 as ab\n"
            "try:\n    ab.Context(0)\nexcept ab.AccmsmError:\n    raise SystemExit(3)\n")
    p = subprocess.run([sys.executable, "-c", code], cwd=ROOT, capture_output=True, text=True, timeout=300,
                       env=dict(os.environ, CUDA_VISIBLE_DEVICES=""))
    assert p.returncode == 3, p.stdout[-2000:] + p.stderr[-2000:]


def test_product_never_imports_the_oracle():
    pkg = os.path.join(ROOT, "accumulation_b200")
    for dirpath, _, files in os.walk(pkg):
        for f in files:
            if f.endswith((".py", ".cu", ".cuh", ".inc", ".hpp", ".h")):
                text = open(os.path.join(dirpath, f), errors="ignore").read()
                assert "oracle" not in text.replace("the oracle", "").replace("with the oracle", "") or f == "__none__", f


def test_rust_ffi_declarations_are_in_sync_with_the_header():
    """accmsm-sys/src/ffi.rs is generated from include/accmsm.h: every declared symbol, no drift"""
    assert subprocess.run([sys.executable, os.path.join(ROOT, "tools", "gen_sys_bindings.py"), "--check"]).returncode == 0
    text = open(os.path.join(ROOT, "accmsm-sys", "src", "ffi.rs")).read()
    for name in header_symbols():
        assert f"pub fn {name}(" in text, name
