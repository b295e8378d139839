"""CPU test of the device job's search plan (tests/search_plan_check.cpp): the path, kernel variants and slice widths
plan_search chooses for synthetic batches and index shapes.  No GPU."""
import os
import subprocess

import pytest

from conftest import ROOT

CHECK = os.path.join(ROOT, "tests", "_build", "search_plan_check")
LIBDIR = os.path.join(ROOT, "guidescan-cli_b200")


@pytest.mark.timeout(600)
def test_search_plan_paths_and_widths():
    lib = os.path.join(LIBDIR, "libgsx.so")
    if not os.path.exists(lib):
        pytest.skip("libgsx.so not built (run __graft_entry__.build())")
    src = os.path.join(ROOT, "tests", "search_plan_check.cpp")
    os.makedirs(os.path.dirname(CHECK), exist_ok=True)
    subprocess.check_call(["g++", "-O2", "-std=c++17", "-I/usr/local/cuda/include", "-o", CHECK, src, "-L" + LIBDIR, "-lgsx",
                           "-Wl,-rpath," + LIBDIR])
    env = {k: v for k, v in os.environ.items() if not k.startswith("GSX_")}
    r = subprocess.run([CHECK], capture_output=True, text=True, timeout=600, env=env)
    assert r.returncode == 0, r.stderr
    assert "search plan selftest ok" in r.stdout
