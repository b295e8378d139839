"""CPU tests of the sweep's summary and parking arithmetic (gsx_core.h, mirrored by tests/host_core_check.cpp) on dense intervals:
a genome with repeat families and low-complexity tracts (synth.add_skew), whose guides reach table entries of more than 16 and more
than 32 rows -- the entries the sweep parks and drains, or passes to the tree search unexamined.  Byte for byte against the oracle."""
import os
import subprocess

import pytest

from conftest import reference_index
from test_host_core import harness  # noqa: F401  (the fixture that builds tests/host_core_check)


@pytest.fixture(scope="module")
def skewed_small(tmp_path_factory):
    """2 Mb, 3 chromosomes, 400 guides (the first 100 with planted copies), add_skew scaled down: 20 repeat families of 10..500
    near-copies and 20 guides drawn from 0.2 Mb of low-complexity tracts"""
    import synth
    d = str(tmp_path_factory.mktemp("skew_host"))
    G = 2_000_000
    g = synth.make_genome(G, 53)
    pos, kmers = synth.sample_guides(g, 400, 53)
    synth.plant(g, kmers[:100], 53)
    kmers, fam, low = synth.add_skew(g, kmers, 53, frac=0.05, lowc_mb=0.2, max_copies=500)
    chroms = synth.chromosome_table(G, 3)
    fa, gcsv = os.path.join(d, "k.fa"), os.path.join(d, "k.guides.csv")
    synth.write_fasta(fa, g, chroms)
    synth.write_guides_csv(gcsv, pos, kmers, chroms)
    reference_index(fa, os.path.join(d, "k"))
    return d, fa, gcsv, fam, low


@pytest.mark.timeout(900)
@pytest.mark.parametrize("m", [2, 3])
def test_sweep_on_skewed_genome_matches_oracle(harness, skewed_small, m):  # noqa: F811
    import oracle as O
    d, fa, gcsv, fam, low = skewed_small
    want = os.path.join(d, "o%d.csv" % m)
    O.Index(fa).enumerate_file(O.make_opts(mismatches=m), gcsv, want, nthreads=os.cpu_count() or 4)
    want_text = open(want, "rb").read()
    # the skew is really there: most family guides have 10+ sites, some guide thousands
    rows = {}
    for line in want_text.decode().splitlines()[1:]:
        k = line.split(",", 1)[0]
        rows[k] = rows.get(k, 0) + 1
    fam_rows = sorted(rows.get("g%d" % i, 0) for i in fam)
    assert fam_rows[len(fam_rows) // 2] >= 10 and max(rows.values()) > 1000
    for tag, extra in (("sweep3", ["--lookahead", "--ftab", "9", "--sweep", "3"]),
                       # a shallow table: most family and tract entries hold more than 32 rows (the "wide" pass-through)
                       ("sweep2", ["--lookahead", "--ftab", "7", "--sweep", "2"])):
        out = os.path.join(d, "%s_m%d.csv" % (tag, m))
        subprocess.run([harness, os.path.join(d, "k"), gcsv, out, "-m", str(m)] + extra, capture_output=True, text=True, check=True)
        assert open(out, "rb").read() == want_text, tag
