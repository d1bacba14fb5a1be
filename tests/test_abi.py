"""The C-ABI library loads without a GPU and exports every symbol include/obboot.h declares (no compute calls)."""
import os
import re
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def header_symbols():
    src = open(os.path.join(ROOT, "include", "obboot.h")).read()
    src = re.sub(r"/\*.*?\*/", "", src, flags=re.S)
    return sorted(set(re.findall(r"\b(ob_[a-z0-9_]+)\s*\(", src)))


def test_library_exports_every_declared_symbol():
    from oaxaca_blinder_rs_b200 import _native
    _native.build()
    lib = _native.lib()
    syms = header_symbols()
    assert len(syms) >= 15
    for s in syms:
        assert hasattr(lib, s), f"{s} declared in include/obboot.h but not exported by libobboot.so"
    assert sorted(_native.SYMBOLS) == [s for s in syms if s in _native.SYMBOLS]
    assert lib.ob_abi_version() == 6


def test_no_cpu_fallback():
    """Without a CUDA device every compute entry point must fail loudly (never route to the oracle).  Checked in a
    child process that sees no device, so that it holds on GPU machines too."""
    code = ("import oaxaca_blinder_rs_b200 as ob\n"
            "try:\n"
            "    ob.Context(0)\n"
            "except ob.OaxacaError as e:\n"
            "    print(e.kind)\n")
    r = subprocess.run([sys.executable, "-c", code], cwd=ROOT, env={**os.environ, "CUDA_VISIBLE_DEVICES": ""},
                       capture_output=True, text=True, timeout=300)
    assert r.returncode == 0, r.stderr
    assert r.stdout.strip() == "NoDevice", (r.stdout, r.stderr)


def test_product_never_imports_the_oracle():
    pkg = os.path.join(ROOT, "oaxaca_blinder_rs_b200")
    for dirpath, _, files in os.walk(pkg):
        for f in files:
            if f.endswith((".py", ".cu", ".cuh", ".h", ".cc", ".cpp")):
                txt = open(os.path.join(dirpath, f), errors="ignore").read()
                assert "pyoracle" not in txt and "ob_oracle" not in txt and "liboracle" not in txt, f


def test_num_stats():
    import ctypes as C
    import numpy as np
    from oaxaca_blinder_rs_b200 import _native
    hb = np.array([1, 0, 1], dtype=np.int32)
    assert _native.lib().ob_num_stats(51, 3, hb.ctypes.data_as(C.POINTER(C.c_int32))) == 5 + 2 * (51 + 2)
