"""gsx_enumerate_genome / `guidescan enumerate --genome`: generation and enumeration in one pass, without the guides CSV.

The contract: the output is byte for byte what gsx_generate_kmers -> (rows selected by a BED file) -> gsx_enumerate_file writes, for
every batch size and device list.  select_rows below restates the row selection; the CPU tests pin it on hand-written rows at the
edges, and the GPU tests use it as the reference for the regions."""
import gzip
import json
import os
import subprocess

import pytest

from conftest import ROOT

GOLD = os.path.join(ROOT, "tests", "golden")
EXE = os.path.join(ROOT, "guidescan-cli_b200", "bin", "guidescan")
HEADER = "id,sequence,pam,chromosome,position,sense\n"


def select_rows(csv_text, bed, k, plen, start):
    """Rows of a generated guides CSV whose k-mer lies inside one interval of `bed` ([(chrom, start, end)], 0-based, half-open),
    in their order.  The k-mer of a row at 1-based position p spans [p-1, p-1+k) when it lies before the PAM on the + strand
    ("+" without --start, "-" with it), else [p-1+plen, p-1+plen+k)."""
    lines = csv_text.splitlines(True)
    out = [lines[0]]
    for line in lines[1:]:
        _, _, _, chrom, pos, sense = line.rstrip("\n").split(",")
        before = (sense == "+") != bool(start)
        a = int(pos) - 1 + (0 if before else plen)
        if any(c == chrom and s <= a and a + k <= e for c, s, e in bed):
            out.append(line)
    return "".join(out)


def row(chrom, pos, sense):
    return "x%s:%d:%s,ACGT,NGG,%s,%d,%s\n" % (chrom, pos, sense, chrom, pos, sense)


def kept(rows, bed, k=4, plen=3, start=False):
    return select_rows(HEADER + "".join(rows), bed, k, plen, start)[len(HEADER):]


# ---- CPU: the row selection ----------------------------------------------------------------------------------------------------
def test_select_exact_fit_and_one_base_short():
    # "+" without --start: the k-mer is [p-1, p-1+k)
    assert kept([row("c", 11, "+")], [("c", 10, 14)]) == row("c", 11, "+")          # [10, 14) exactly
    assert kept([row("c", 10, "+")], [("c", 10, 14)]) == ""                          # [9, 13): a base short at the left
    assert kept([row("c", 12, "+")], [("c", 10, 14)]) == ""                          # [11, 15): a base short at the right
    # "-" without --start: the k-mer is behind the PAM, [p-1+plen, p-1+plen+k)
    assert kept([row("c", 8, "-")], [("c", 10, 14)]) == row("c", 8, "-")
    assert kept([row("c", 7, "-")], [("c", 10, 14)]) == ""
    assert kept([row("c", 9, "-")], [("c", 10, 14)]) == ""


def test_select_with_start_swaps_the_senses():
    assert kept([row("c", 8, "+")], [("c", 10, 14)], start=True) == row("c", 8, "+")
    assert kept([row("c", 11, "+")], [("c", 10, 14)], start=True) == ""
    assert kept([row("c", 11, "-")], [("c", 10, 14)], start=True) == row("c", 11, "-")
    assert kept([row("c", 8, "-")], [("c", 10, 14)], start=True) == ""


def test_select_overlapping_and_adjacent_intervals():
    rows = [row("c", p, "+") for p in range(1, 30)]
    # overlapping: each row once, in its order
    got = kept(rows, [("c", 5, 12), ("c", 8, 16), ("c", 5, 12)])
    assert got == "".join(row("c", p, "+") for p in range(6, 14))
    # adjacent: a k-mer across the shared end lies in neither interval
    got = kept(rows, [("c", 0, 10), ("c", 10, 20)])
    assert got == "".join(row("c", p, "+") for p in list(range(1, 8)) + list(range(11, 18)))


def test_select_interval_at_chromosome_end_and_other_chromosomes():
    rows = [row("a", 97, "+"), row("b", 97, "+"), row("a", 96, "-")]       # chromosome a of 100 bases
    assert kept(rows, [("a", 90, 100)]) == row("a", 97, "+")
    assert kept(rows, [("a", 90, 100)], plen=0) == row("a", 97, "+") + row("a", 96, "-")
    assert kept(rows, []) == ""


# ---- CPU: command line errors, before any index or device is touched --------------------------------------------------------
def cli(*args):
    if not os.path.exists(EXE):
        pytest.skip("CLI not built")
    return subprocess.run([EXE] + list(args), capture_output=True, text=True)


def test_cli_kmers_file_and_genome_are_exclusive():
    r = cli("enumerate", "idx", "-f", "k.csv", "--genome", "g.fa", "-o", "out")
    assert r.returncode != 0 and "--genome" in r.stderr and "index" not in r.stdout.lower()


def test_cli_kmer_length_out_of_range():
    r = cli("enumerate", "idx", "--genome", "g.fa", "--kmer-length", "40", "-o", "out")
    assert r.returncode != 0 and "--kmer-length" in r.stderr and "Loading" not in r.stdout


def test_cli_kmers_needs_output():
    r = cli("kmers", "g.fa")
    assert r.returncode != 0 and "--output is required" in r.stderr


def test_cli_unknown_option_after_genome():
    r = cli("enumerate", "idx", "--genome", "g.fa", "--bogus", "-o", "out")
    assert r.returncode != 0 and "--bogus" in r.stderr


def test_cli_neither_kmers_file_nor_genome():
    r = cli("enumerate", "idx", "-o", "out")
    assert r.returncode != 0 and "--kmers-file is required" in r.stderr


def test_cli_help_documents_the_new_surface():
    r = cli("--help")
    for s in ("kmers [OPTIONS] GENOME.fa", "--genome", "--regions", "--min-chr-length", "--kmer-length"):
        assert s in r.stderr


# ---- GPU -----------------------------------------------------------------------------------------------------------------------
CASES = ["g200k", "g150kN"]
# (name, enumerate params, fmt, mode, generator options, BED of the first bases of every chromosome or None)
OPTION_SETS = [
    ("m3_csv", dict(mismatches=3), "csv", "complete", {}, None),
    ("m2_sam", dict(mismatches=2), "sam", "complete", {}, None),
    ("m3_csv_succinct", dict(mismatches=3), "csv", "succinct", {}, None),
    ("m3_sam_succinct", dict(mismatches=3), "sam", "succinct", {}, None),
    ("m3_altNAG_sam", dict(mismatches=3, alt_pams=("NAG",)), "sam", "complete", {}, None),
    ("m1_r1_d1_csv", dict(mismatches=1, rna_bulges=1, dna_bulges=1), "csv", "complete", {}, 800),
    ("m2_start_TTTN_k23", dict(mismatches=2, start=True), "csv", "complete", dict(pam="TTTN", kmer_length=23), None),
]


@pytest.fixture(scope="module")
def gsx():
    import gsx as g
    if g.device_count() < 1:
        pytest.fail("no CUDA device: the product has no CPU path")
    return g


@pytest.fixture(scope="module")
def indexes(gsx, golden_index):
    out = {}
    yield lambda case, devices=(0,): out.setdefault((case, tuple(devices)), gsx.Index.open(golden_index[case], devices=list(devices)))
    for ix in out.values():
        ix.close()


def write_bed(path, intervals, comment=True):
    with open(path, "w") as f:
        if comment:
            f.write("# regions\ntrack name=test\n\n")
        for c, s, e in intervals:
            f.write("%s\t%d\t%d\tname\t0\t+\n" % (c, s, e))
    return path


def head_bed(ix, n):
    return [(c, 0, min(n, L)) for c, L in ix.chromosomes()]


def via_csv(gsx, ix, fa, d, params, fmt, mode, gen, bed, tag):
    """gsx_generate_kmers -> select_rows -> gsx_enumerate_file: the reference of the contract"""
    csv = os.path.join(d, tag + ".kmers.csv")
    gsx.generate_kmers(fa, csv, start=bool(params.start), **gen)
    if bed is not None:
        text = open(csv).read()
        open(csv, "w").write(select_rows(text, bed, gen.get("kmer_length", 20), len(gen.get("pam", "NGG")), bool(params.start)))
    out = os.path.join(d, tag + ".want")
    n, _ = ix.enumerate_file(csv, out, params, fmt=fmt, mode=mode)
    return n, open(out, "rb").read()


@pytest.mark.gpu
@pytest.mark.parametrize("opt", [o[0] for o in OPTION_SETS])
@pytest.mark.parametrize("case", CASES)
def test_genome_enumerate_equals_generate_then_enumerate_file(gsx, golden_dir, indexes, tmp_path, case, opt):
    name, kw, fmt, mode, gen, head = next(o for o in OPTION_SETS if o[0] == opt)
    fa = golden_dir[case][0]
    ix = indexes(case)
    params = gsx.make_params(**kw)
    bed = head_bed(ix, head) if head else None
    bed_path = write_bed(str(tmp_path / "r.bed"), bed) if bed else None
    n_want, want = via_csv(gsx, ix, fa, str(tmp_path), params, fmt, mode, gen, bed, name)
    out = str(tmp_path / "got")
    n, ctr = ix.enumerate_genome(fa, out, params, regions=bed_path, fmt=fmt, mode=mode, **gen)
    assert open(out, "rb").read() == want
    assert n == n_want
    assert n > (100 if head else 1000)


@pytest.mark.gpu
def test_genome_enumerate_equals_cpu_oracle(gsx, golden_dir, indexes, tmp_path):
    import kmers_oracle as K
    import oracle as O
    fa = golden_dir["g150kN"][0]
    ix = indexes("g150kN")
    bed = head_bed(ix, 5000)
    csv = str(tmp_path / "oracle.csv")
    open(csv, "w").write(select_rows(K.generate(fa), bed, 20, 3, False))
    want = str(tmp_path / "oracle.out")
    O.Index(fa).enumerate_file(O.make_opts(mismatches=2), csv, want, nthreads=4)
    got = str(tmp_path / "gpu.out")
    n, _ = ix.enumerate_genome(fa, got, gsx.make_params(mismatches=2), regions=write_bed(str(tmp_path / "r.bed"), bed))
    assert n > 500
    assert open(got, "rb").read() == open(want, "rb").read()


@pytest.mark.gpu
def test_genome_enumerate_independent_of_batches_and_devices(gsx, golden_dir, indexes, tmp_path):
    fa = golden_dir["g150kN"][0]
    params = gsx.make_params(mismatches=3)
    outs = {}
    # the whole genome, large batches; a BED subset near every chromosome's ends with batches of 7 (hundreds of calls that cross
    # chromosome boundaries and leave the sweep for the tree search)
    ix0 = indexes("g150kN")
    bed = [(c, max(0, L - 1500), L) for c, L in ix0.chromosomes()] + [(c, 0, 1500) for c, L in ix0.chromosomes()]
    bed_path = write_bed(str(tmp_path / "ends.bed"), bed)
    for devices in ((0,), (0, 0)):
        ix = indexes("g150kN", devices)
        for batch in (8193, 0):
            out = str(tmp_path / ("all_%d_%d" % (len(devices), batch)))
            outs[("all", devices, batch)] = (ix.enumerate_genome(fa, out, params, batch_guides=batch)[0], open(out, "rb").read())
        for batch in (7, 0):
            out = str(tmp_path / ("ends_%d_%d" % (len(devices), batch)))
            outs[("ends", devices, batch)] = (ix.enumerate_genome(fa, out, params, regions=bed_path, batch_guides=batch)[0], open(out, "rb").read())
    for kind in ("all", "ends"):
        got = {v for k, v in outs.items() if k[0] == kind}
        assert len(got) == 1, kind
    assert outs[("all", (0,), 0)][0] > 15000
    n_ends = outs[("ends", (0,), 0)][0]
    assert 100 < n_ends < 2000
    assert outs[("ends", (0,), 0)][1] == via_csv(gsx, ix0, fa, str(tmp_path), params, "csv", "complete", {}, bed, "ends")[1]


@pytest.mark.gpu
def test_genome_enumerate_regions(gsx, golden_dir, indexes, tmp_path):
    fa = golden_dir["g200k"][0]
    ix = indexes("g200k")
    chroms = ix.chromosomes()
    assert len(chroms) >= 3
    c0, (c1, l1) = chroms[0][0], chroms[1]
    # unsorted, overlapping, one at a chromosome's end, chromosome chroms[2] without intervals
    bed = [(c1, l1 - 3000, l1), (c0, 9000, 12000), (c0, 1000, 4000), (c0, 3000, 6000), (c1, 100, 2000), (c0, 5990, 6010)]
    bed_path = write_bed(str(tmp_path / "r.bed"), bed)
    params = gsx.make_params(mismatches=3)
    n_want, want = via_csv(gsx, ix, fa, str(tmp_path), params, "csv", "complete", {}, bed, "regions")
    out = str(tmp_path / "got")
    n, _ = ix.enumerate_genome(fa, out, params, regions=bed_path)
    assert open(out, "rb").read() == want and n == n_want and n > 500
    assert all(f",{chroms[2][0]}," not in l for l in open(str(tmp_path / "regions.kmers.csv")).readlines()[1:])


@pytest.mark.gpu
@pytest.mark.parametrize("fmt", ["csv", "sam"])
def test_genome_enumerate_nothing_selected_writes_the_header(gsx, golden_dir, indexes, tmp_path, fmt):
    fa = golden_dir["g200k"][0]
    ix = indexes("g200k")
    c, L = ix.chromosomes()[0]
    bed_path = write_bed(str(tmp_path / "r.bed"), [(c, 100, 110), (c, L, L)])      # shorter than a k-mer; empty at the end
    out = str(tmp_path / "got")
    n, _ = ix.enumerate_genome(fa, out, gsx.make_params(), regions=bed_path, fmt=fmt)
    assert n == 0
    assert open(out, "rb").read() == ix.header(fmt=fmt)
    # the CSV path on a kmers file holding only its header line writes the same
    csv = str(tmp_path / "empty.csv")
    open(csv, "w").write(HEADER)
    out2 = str(tmp_path / "got2")
    assert ix.enumerate_file(csv, out2, gsx.make_params(), fmt=fmt)[0] == 0
    assert open(out2, "rb").read() == ix.header(fmt=fmt)


@pytest.mark.gpu
def test_genome_enumerate_argument_errors(gsx, golden_dir, indexes, tmp_path):
    fa = golden_dir["g200k"][0]
    ix = indexes("g200k")
    chroms = ix.chromosomes()
    text = open(fa).read()
    renamed = str(tmp_path / "renamed.fa")
    open(renamed, "w").write(text.replace(">" + chroms[1][0], ">other", 1))
    shortened = str(tmp_path / "short.fa")
    lines = text.splitlines(True)
    last = max(i for i, l in enumerate(lines) if not l.startswith(">"))
    open(shortened, "w").write("".join(lines[:last] + [lines[last][:-2] + "\n"]))
    params = gsx.make_params()
    bad = [
        (dict(fasta=renamed), "other"),
        (dict(fasta=shortened), chroms[-1][0]),
        (dict(regions=write_bed(str(tmp_path / "u.bed"), [("chrUn", 0, 10)])), "chrUn"),
        (dict(regions=write_bed(str(tmp_path / "e.bed"), [(chroms[0][0], 0, chroms[0][1] + 1)])), chroms[0][0]),
        (dict(regions=write_bed(str(tmp_path / "s.bed"), [(chroms[0][0], 50, 40)])), "start"),
        (dict(kmer_length=33), "33"),
        (dict(kmer_length=30), "32"),
        (dict(kmer_length=28, params=gsx.make_params(dna_bulges=2)), "32"),
        (dict(pam="NGR"), "NGR"),
    ]
    for kw, word in bad:
        out = str(tmp_path / "never")
        kw = dict(kw)
        f = kw.pop("fasta", fa)
        p = kw.pop("params", params)
        with pytest.raises(gsx.GsxError) as e:
            ix.enumerate_genome(f, out, p, **kw)
        assert e.value.code == 1, (kw, str(e.value))            # GSX_ERR_ARG
        assert word in str(e.value), (kw, str(e.value))
        assert not os.path.exists(out)                           # rejected before the output is opened


def variants():
    return json.load(open(os.path.join(GOLD, "kmers_manifest.json")))


@pytest.mark.gpu
@pytest.mark.parametrize("name", sorted(variants()))
def test_cli_kmers_matches_reference_script(gsx, tmp_path, name):
    fa = str(tmp_path / "kmers.fa")
    open(fa, "wb").write(gzip.open(os.path.join(GOLD, "kmers.fa.gz"), "rb").read())
    out = str(tmp_path / "k.csv")
    r = cli("kmers", fa, "-o", out, *variants()[name]["args"])
    assert r.returncode == 0, r.stderr
    assert open(out, "rb").read() == gzip.open(os.path.join(GOLD, "kmers.%s.csv.gz" % name), "rb").read()


@pytest.mark.gpu
@pytest.mark.parametrize("with_regions", [False, True])
def test_cli_enumerate_genome_matches_kmers_file(gsx, golden_dir, golden_index, tmp_path, with_regions):
    fa = golden_dir["g150kN"][0]
    prefix = golden_index["g150kN"]
    opts = ["-m", "2", "--format", "sam", "-a", "NAG"]
    csv = str(tmp_path / "k.csv")
    r = cli("kmers", fa, "-o", csv, "--prefix", "lib_")
    assert r.returncode == 0, r.stderr
    extra = []
    if with_regions:
        ix = gsx.Index.open(prefix, devices=[0])
        bed = head_bed(ix, 30000)
        ix.close()
        extra = ["--regions", write_bed(str(tmp_path / "r.bed"), bed)]
        text = open(csv).read()
        open(csv, "w").write(select_rows(text, bed, 20, 3, False))
    want = str(tmp_path / "want.sam")
    r = cli("enumerate", prefix, "-f", csv, "-o", want, *opts)
    assert r.returncode == 0, r.stderr
    got = str(tmp_path / "got.sam")
    r = cli("enumerate", prefix, "--genome", fa, "--prefix", "lib_", "-o", got, *opts, *extra)
    assert r.returncode == 0, r.stderr
    assert open(got, "rb").read() == open(want, "rb").read()
    assert os.path.getsize(got) > 10000
