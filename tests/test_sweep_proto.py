"""CPU test of the two-part sweep's filter for guides whose summary planes are protospacer levels or wildcards
(gsx_core.h summary_eval_proto, tests/sweep_proto_check.cpp): equal to the general filter on random sectors.  No GPU."""
import os
import subprocess

import pytest

from conftest import ROOT

CHECK = os.path.join(ROOT, "tests", "_build", "sweep_proto_check")
LIBDIR = os.path.join(ROOT, "guidescan-cli_b200")


@pytest.mark.timeout(600)
def test_proto_filter_equals_general_filter():
    lib = os.path.join(LIBDIR, "libgsx.so")
    if not os.path.exists(lib):
        pytest.skip("libgsx.so not built (run __graft_entry__.build())")
    src = os.path.join(ROOT, "tests", "sweep_proto_check.cpp")
    os.makedirs(os.path.dirname(CHECK), exist_ok=True)
    subprocess.check_call(["g++", "-O2", "-std=c++17", "-I/usr/local/cuda/include", "-o", CHECK, src, "-L" + LIBDIR, "-lgsx",
                           "-Wl,-rpath," + LIBDIR])
    r = subprocess.run([CHECK], capture_output=True, text=True, timeout=600)
    assert r.returncode == 0, r.stderr
    assert "proto selftest ok" in r.stdout
