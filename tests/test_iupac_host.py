"""IUPAC class letters in PAMs on the host (tests/iupac_check.cpp): letter tables, the device arithmetic of a class character against
brute force, the PAM bytes of A/C/G/T/N lists (unchanged), the search path of class batches, the generator's expansion against
oracle/kmers_oracle.py, and the CLI's validation.  No GPU."""
import os
import re
import subprocess

import pytest

from conftest import ROOT

import kmers_oracle as KO

CHECK = os.path.join(ROOT, "tests", "_build", "iupac_check")
LIBDIR = os.path.join(ROOT, "guidescan-cli_b200")
BIN = os.path.join(LIBDIR, "bin", "guidescan")
IUPAC = {"R": "AG", "Y": "CT", "S": "CG", "W": "AT", "K": "GT", "M": "AC", "B": "CGT", "D": "AGT", "H": "ACT", "V": "ACG"}


@pytest.fixture(scope="module")
def check_output():
    if not os.path.exists(os.path.join(LIBDIR, "libgsx.so")):
        pytest.skip("libgsx.so not built (run __graft_entry__.build())")
    os.makedirs(os.path.dirname(CHECK), exist_ok=True)
    subprocess.check_call(["g++", "-O2", "-std=c++17", "-I/usr/local/cuda/include", "-o", CHECK, os.path.join(ROOT, "tests", "iupac_check.cpp"),
                           "-L" + LIBDIR, "-lgsx", "-Wl,-rpath," + LIBDIR])
    env = {k: v for k, v in os.environ.items() if not k.startswith("GSX_")}
    r = subprocess.run([CHECK], capture_output=True, text=True, timeout=600, env=env)
    assert r.returncode == 0, r.stderr
    assert "iupac selftest ok" in r.stdout
    return r.stdout


def _lists(out, kind):
    return {m.group(1): m.group(2).split() for m in re.finditer(r"^%s (\S+): ?(.*)$" % kind, out, re.M)}


def test_tables_arithmetic_packing_and_paths(check_output):
    pass                      # (the checks ran in the fixture; a failure there names the broken check)


def test_expansion_is_kmers_oracle_for_acgtn(check_output):
    exp = _lists(check_output, "expand")
    for pam, got in exp.items():
        if set(pam) <= set("ACGTN"):
            assert got == KO.pam_set(pam), pam


def test_expansion_of_classes(check_output):
    """breadth first, first expandable letter first, members in the order A, C, T, G; the class-only expansion keeps N"""
    def restated(pam):
        q = [pam]
        first = lambda p: next((i for i, c in enumerate(p) if c == "N" or c in IUPAC), None)
        while any(first(p) is not None for p in q):
            p = q.pop(0)
            at = first(p)
            if at is None:
                q.append(p)
            else:
                q.extend(p[:at] + c + p[at + 1:] for c in "ACTG" if c in IUPAC.get(p[at], "ACGT"))
        return q
    exp, cls = _lists(check_output, "expand"), _lists(check_output, "classes")
    for pam in exp:
        assert exp[pam] == restated(pam), pam
        want = [""]
        for c in pam:
            want = [s + b for s in want for b in IUPAC.get(c, c)]
        assert cls[pam] == want, pam
    assert exp["NRG"][:4] == ["AAG", "AGG", "CAG", "CGG"] and len(exp["NRRH"]) == 4 * 2 * 2 * 3
    assert cls["NNGRRT"] == ["NNGAAT", "NNGAGT", "NNGGAT", "NNGGGT"] and len(cls["NRRH"]) == 12


@pytest.mark.parametrize("args", [["kmers", "g.fa", "--pam", "NXG"], ["kmers", "g.fa", "--pam", "nrg"], ["kmers", "g.fa", "--pam", "NrG"],
                                  ["enumerate", "IDX", "--genome", "g.fa", "--pam", "NUG"],
                                  ["decode", "db.sam", "--genome", "g.fa", "-a", "NZG"], ["decode", "db.sam", "--genome", "g.fa", "-a", "NRGG"]])
def test_cli_rejects_bad_pam_letters(tmp_path, args):
    if not os.path.exists(BIN):
        pytest.skip("guidescan not built")
    r = subprocess.run([BIN] + args + ["-o", os.path.join(str(tmp_path), "o.csv")], capture_output=True, text=True, cwd=str(tmp_path))
    assert r.returncode == 105, r.stderr


def test_cli_accepts_class_letters(tmp_path):
    """kmers --pam NRG passes validation: on a machine without a GPU it fails only for want of a device"""
    if not os.path.exists(BIN):
        pytest.skip("guidescan not built")
    fa = os.path.join(str(tmp_path), "g.fa")
    open(fa, "w").write(">c\nACGTACGTACGTACGTACGTACGTAGG\n")
    r = subprocess.run([BIN, "kmers", "--pam", "NRG", "-o", os.path.join(str(tmp_path), "k.csv"), fa], capture_output=True, text=True)
    import gsx
    if gsx.device_count() == 0:
        assert r.returncode == 1 and "no CUDA device" in r.stderr, r.stderr
    else:
        assert r.returncode == 0, r.stderr
