"""CPU-side checks of the C-ABI boundary: the library loads, exports every symbol include/clstm_b200.h declares,
and refuses to run without a CUDA device (no CPU fallback).  No compute calls here."""
import os
import re
import subprocess
import sys

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


@pytest.fixture(scope="module")
def ffi():
    import clstm_b200
    if not os.path.exists(clstm_b200.LIB_PATH):
        clstm_b200.build()
    return clstm_b200


def test_header_symbols_exported(ffi):
    hdr = open(os.path.join(ROOT, "include", "clstm_b200.h")).read()
    declared = set(re.findall(r"\b(clstm_b200_[a-z0-9_]+)\s*\(", hdr))
    declared -= {"clstm_b200_net", "clstm_b200_cfg"}
    out = subprocess.check_output(["nm", "-D", "--defined-only", ffi.LIB_PATH], text=True)
    exported = set(re.findall(r"\bT (clstm_b200_[a-z0-9_]+)", out))
    assert declared, "no declarations parsed"
    assert declared <= exported, sorted(declared - exported)
    assert declared == set(ffi.EXPORTS), sorted(declared ^ set(ffi.EXPORTS))
    ffi.lib()  # binds every symbol with its signature


def test_library_is_sm100a_only(ffi):
    out = subprocess.check_output(["cuobjdump", "-lelf", ffi.LIB_PATH], text=True)
    archs = set(re.findall(r"sm_(\d+a?)", out))
    assert archs == {"100a"}, archs


def test_no_cpu_fallback(ffi):
    # every device hidden, so that the check also runs on a machine with a GPU
    code = ("import clstm_b200\n"
            "try:\n"
            "    clstm_b200.Net(48, 100, 83)\n"
            "except clstm_b200.Error as e:\n"
            "    print(e)\n")
    r = subprocess.run([sys.executable, "-c", code], cwd=ROOT, env=dict(os.environ, CUDA_VISIBLE_DEVICES=""),
                       capture_output=True, text=True, timeout=120)
    assert r.returncode == 0, r.stderr[-2000:]
    assert "no CPU fallback" in r.stdout, r.stdout


def test_product_does_not_touch_oracle():
    # the oracle is test infrastructure: nothing under clstm_b200/ may import, link or execute it
    bad = []
    for d, _, files in os.walk(os.path.join(ROOT, "clstm_b200")):
        if os.sep + "build" in d or os.sep + "lib" in d:
            continue
        for f in files:
            if f.endswith((".py", ".cu", ".cuh", ".h", ".cc", ".cpp", "Makefile")):
                txt = open(os.path.join(d, f), errors="ignore").read()
                if re.search(r"liboracle|oracle/|import oracle|from oracle|clstm_oracle", txt):
                    bad.append(os.path.join(d, f))
    assert not bad, bad
