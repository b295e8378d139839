"""CPU test of the two-part sweep's enumeration plan (tests/split_plan_check.cpp): every alignment within 3 mismatches reached by
exactly one of the two forms, a quarter of the plain sweep's patterns.  No GPU."""
import os
import re
import subprocess

import pytest

from conftest import ROOT

CHECK = os.path.join(ROOT, "tests", "_build", "split_plan_check")
LIBDIR = os.path.join(ROOT, "guidescan-cli_b200")


@pytest.mark.timeout(600)
def test_two_part_plan_reaches_every_site_once():
    lib = os.path.join(LIBDIR, "libgsx.so")
    if not os.path.exists(lib):
        pytest.skip("libgsx.so not built (run __graft_entry__.build())")
    src = os.path.join(ROOT, "tests", "split_plan_check.cpp")
    os.makedirs(os.path.dirname(CHECK), exist_ok=True)
    subprocess.check_call(["g++", "-O2", "-std=c++17", "-I/usr/local/cuda/include", "-o", CHECK, src, "-L" + LIBDIR, "-lgsx",
                           "-Wl,-rpath," + LIBDIR])
    r = subprocess.run([CHECK], capture_output=True, text=True, timeout=600)
    assert r.returncode == 0, r.stderr
    assert "split selftest ok" in r.stdout
    per = [float(x) for x in re.findall(r"patterns per guide and strand ([0-9.]+) \(", r.stdout)]
    assert len(per) == 3
    for p in per:                              # 2 185 (distal half capped) + 496 (PAM-first, proximal half capped)
        assert abs(p - 2681) <= 0.02 * 2681
    assert "plain sweep: patterns per guide and strand 10690" in r.stdout
