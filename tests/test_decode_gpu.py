"""gsx_decode_database on the GPU: a SAM complete database decodes to the CSV rows enumerate prints for the same guides (sam_scoring =
1), byte for byte, with the CFD the search computed; the reference's own SAM databases decode as oracle/decode_oracle.py decodes them;
batches, concatenated runs, regions and every error case of the semantics (include/gsx.h)."""
import gzip
import json
import os

import numpy as np
import pytest

from conftest import GOLDEN

import decode_oracle as DO

pytestmark = pytest.mark.gpu

OPTION_SETS = {
    "m0": dict(mismatches=0), "m2": dict(mismatches=2), "m3": dict(mismatches=3), "m4": dict(mismatches=4),
    "m3_altNAG": dict(mismatches=3, alt_pams=("NAG",)), "m3_max1": dict(mismatches=3, max_off_targets=1),
    "m3_max2": dict(mismatches=3, max_off_targets=2),
}


@pytest.fixture(scope="module")
def gsx():
    import gsx as G
    if G.device_count() == 0:
        pytest.skip("no CUDA device")
    return G


@pytest.fixture(scope="module")
def indexes(gsx, golden_dir):
    """{case: (fasta, index, rows)}: rows = the golden guides with a PAM column, every other one on the "-" sense (SAM FLAG 16)"""
    out = {}
    for case, (fa, guides) in golden_dir.items():
        rows = [(i, s, p, k % 2 == 0) for k, (i, s, p, _) in enumerate(gsx.read_guides_csv(guides)) if p]
        out[case] = (fa, gsx.Index.build(fa, devices=[0]), rows)
    yield out
    for _, ix, _ in out.values():
        ix.close()


def enumerate_both(gsx, ix, rows, **kw):
    """(result, SAM complete text, CSV complete text) of one enumerate call with the SAM rule"""
    p = gsx.make_params(sam_scoring=True, **kw)
    r = ix.enumerate([(s, pam) for _, s, pam, _ in rows], p)
    sam = ix.header("sam") + r.format(rows, p, "sam", "complete")
    csv = ix.header("csv") + r.format(rows, p, "csv", "complete")
    return r, sam.decode(), csv.decode()


def rows_with_sam_record(csv, sam):
    ids = {l.split("\t", 1)[0] for l in sam.splitlines() if not l.startswith("@")}
    lines = csv.splitlines(True)
    return lines[0] + "".join(l for l in lines[1:] if l.split(",", 1)[0] in ids)


def decode(gsx, tmp_path, sam_text, fa, name="db", **kw):
    sam = os.path.join(tmp_path, name + ".sam")
    out = os.path.join(tmp_path, name + ".csv")
    open(sam, "w").write(sam_text)
    ng, nr = gsx.decode_database(sam, fa, out, **kw)
    text = open(out).read()
    assert nr == len(text.splitlines()) - 1
    return text


@pytest.mark.parametrize("opts", sorted(OPTION_SETS))
@pytest.mark.parametrize("case", ["g200k", "g150kN"])
def test_decode_is_enumerate_csv(gsx, indexes, tmp_path, case, opts):
    fa, ix, rows = indexes[case]
    kw = OPTION_SETS[opts]
    r, sam, csv = enumerate_both(gsx, ix, rows, **kw)
    alts = kw.get("alt_pams", ())
    want = rows_with_sam_record(csv, sam)
    assert len(want.splitlines()) > (1 if opts == "m0" else 20)
    assert decode(gsx, tmp_path, sam, fa, alt_pams=alts) == want
    succinct = decode(gsx, tmp_path, sam, fa, alt_pams=alts, mode="succinct")
    assert succinct.splitlines()[1:] == [",".join(l.split(",")[:6] + l.split(",")[9:]) for l in want.splitlines()[1:]]
    # --cfd: the column round-trips the float32 CFD of the counted hits, in their order
    with_cfd = decode(gsx, tmp_path, sam, fa, alt_pams=alts, cfd=True).splitlines()
    assert with_cfd[0] == want.splitlines()[0] + ",cfd"
    assert [l.rsplit(",", 1)[0] for l in with_cfd[1:]] == want.splitlines()[1:]
    h, g = r.hit_arrays(), r.guide_arrays()
    sam_ids = {l.split("\t", 1)[0] for l in sam.splitlines() if not l.startswith("@")}
    want_cfd = []
    for k, row in enumerate(rows):
        if row[0] in sam_ids:
            b, n = int(g["first_hit"][k]), int(g["n_hits"][k])
            want_cfd += [h["cfd"][j] for j in range(b, b + n) if h["counted"][j]]
    got_cfd = np.array([np.float32(l.rsplit(",", 1)[1]) for l in with_cfd[1:]], dtype=np.float32)
    assert np.array_equal(got_cfd.view(np.uint32), np.array(want_cfd, dtype=np.float32).view(np.uint32))


@pytest.mark.parametrize("variant,alts", [("m2_sam", ()), ("m3_altNAG_sam", ("NAG",)), ("m4_max1_sam", ())])
@pytest.mark.parametrize("case", ["g200k", "g150kN"])
def test_reference_databases_decode_as_the_oracle(gsx, golden_dir, tmp_path, case, variant, alts):
    fa = golden_dir[case][0]
    text = "".join(l for l in gzip.open(os.path.join(GOLDEN, "%s.%s.out.gz" % (case, variant)), "rt").read().splitlines(True)
                   if not l.startswith("no_pam\t"))
    path = os.path.join(tmp_path, "ref.sam")
    open(path, "w").write(text)
    want = DO.decode(path, fa, alt_pams=alts)
    assert len(want.splitlines()) > 20
    assert decode(gsx, tmp_path, text, fa, alt_pams=alts) == want
    if case == "g150kN":           # guides whose only perfect match is a sentinel: empty RNAME, decoded all the same
        assert any(l.split("\t")[2] == "" for l in text.splitlines() if not l.startswith("@"))


def test_live_genome_with_runs_of_n(gsx, tmp_path):
    import synth
    man = json.load(open(os.path.join(GOLDEN, "live_manifest.json")))
    ds = man["dataset"]
    synth.make_dataset(str(tmp_path), ds["G"], ds["n_chr"], ds["n_guides"], seed=ds["seed"], name="live", n_runs_of_N=ds["n_runs_of_N"])
    fa = os.path.join(tmp_path, "live.fa")
    rows = [(i, s, p, k % 3 != 0) for k, (i, s, p, _) in enumerate(gsx.read_guides_csv(os.path.join(tmp_path, "live.guides.csv")))]
    ix = gsx.Index.build(fa, devices=[0])
    try:
        for kw in (dict(mismatches=2), dict(mismatches=4, alt_pams=("NAG",))):
            _, sam, csv = enumerate_both(gsx, ix, rows, **kw)
            assert decode(gsx, tmp_path, sam, fa, alt_pams=kw.get("alt_pams", ())) == rows_with_sam_record(csv, sam)
    finally:
        ix.close()
    ref = gzip.open(os.path.join(GOLDEN, "live.m2_sam.out.gz"), "rt").read()
    path = os.path.join(tmp_path, "ref.sam")
    open(path, "w").write(ref)
    assert decode(gsx, tmp_path, ref, fa) == DO.decode(path, fa)


def test_concatenated_runs_and_batch_boundaries(gsx, indexes, tmp_path, monkeypatch):
    fa, ix, rows = indexes["g200k"]
    half = len(rows) // 2
    _, sam_a, csv_a = enumerate_both(gsx, ix, rows[:half], mismatches=4)
    _, sam_b, csv_b = enumerate_both(gsx, ix, rows[half:], mismatches=4)
    # the split-and-concatenate recipe: two runs' files one after the other, the second with its header
    want = rows_with_sam_record(csv_a, sam_a) + rows_with_sam_record(csv_b, sam_b).split("\n", 1)[1]
    one = decode(gsx, tmp_path, sam_a + sam_b, fa)
    assert one == want
    # batches of a few hundred bytes: lists span batch boundaries, a record longer than a batch makes its batch longer, the database
    # is dozens of batches, and a guide's second record (another perfect match) can land in the next batch
    lens = [len(l) for l in sam_a.splitlines() if not l.startswith("@")]
    assert max(lens) > 300
    for b in (150, 400, 5000):
        monkeypatch.setenv("GSX_DECODE_BATCH_BYTES", str(b))
        assert decode(gsx, tmp_path, sam_a + sam_b, fa, name="b%d" % b) == one
    # without the device turn (GSX_DEVICE_LOCK=0, INTEGRATION.md) the same text
    monkeypatch.setenv("GSX_DEVICE_LOCK", "0")
    assert decode(gsx, tmp_path, sam_a + sam_b, fa, name="nolock") == one


def test_regions(gsx, indexes, tmp_path):
    fa, ix, rows = indexes["g150kN"]
    _, sam, _ = enumerate_both(gsx, ix, rows, mismatches=3)
    path = os.path.join(tmp_path, "db.sam")
    open(path, "w").write(sam)
    names, lens, _ = DO.read_fasta(fa)
    recs = [l.split("\t") for l in sam.splitlines() if not l.startswith("@") and l.split("\t")[2]]
    chrom, pos = recs[3][2], int(recs[3][3])
    bed = [(n, 0, 40) for n in names] + [(n, l - 60, l) for n, l in zip(names, lens)] + [(chrom, pos - 1, pos - 1 + 23)]
    # (a site ending exactly at a chromosome's end, if the database has one, lies inside its last interval)
    ends = [(r[2], int(r[3])) for r in recs if int(r[3]) - 1 + 23 == dict(zip(names, lens))[r[2]]]
    bed += [(c, p - 1, p + 22) for c, p in ends]
    bf = os.path.join(tmp_path, "r.bed")
    open(bf, "w").write("".join("%s\t%d\t%d\n" % x for x in bed))
    want = DO.decode(path, fa, regions=bed)
    assert len(want.splitlines()) > 1
    got = decode(gsx, tmp_path, sam, fa, regions=bf)
    assert got == want
    assert got != decode(gsx, tmp_path, sam, fa)
    empty = os.path.join(tmp_path, "e.bed")
    open(empty, "w").write("%s\t%d\t%d\n" % (chrom, pos - 1, pos - 1 + 22))       # a base short: selects nothing
    assert decode(gsx, tmp_path, sam, fa, regions=empty) == want.splitlines(True)[0]


def expect_arg_error(gsx, tmp_path, text, fa, *words, **kw):
    path = os.path.join(tmp_path, "bad.sam")
    open(path, "w").write(text)
    with pytest.raises(gsx.GsxError) as e:
        gsx.decode_database(path, fa, os.path.join(tmp_path, "bad.csv"), **kw)
    assert e.value.code == 1, str(e.value)
    for w in words:
        assert w in str(e.value), (w, str(e.value))
    return str(e.value)


def test_errors_name_the_record(gsx, indexes, golden_dir, tmp_path):
    fa, ix, rows = indexes["g200k"]
    # a database written with bulges fails the consistency check
    _, sam, _ = enumerate_both(gsx, ix, rows, mismatches=1, rna_bulges=1)
    expect_arg_error(gsx, tmp_path, sam, fa, "at byte", "off-target")
    # another genome: @SQ lines, and without them the delimiter, and with the right length but other bases the sites
    _, sam, _ = enumerate_both(gsx, ix, rows, mismatches=2)
    expect_arg_error(gsx, tmp_path, sam, golden_dir["g150kN"][0], "@SQ line")
    body = "".join(l for l in sam.splitlines(True) if not l.startswith("@"))
    expect_arg_error(gsx, tmp_path, body, golden_dir["g150kN"][0], "-200001")
    other = os.path.join(tmp_path, "other.fa")
    names, lens, text = DO.read_fasta(fa)
    rng = np.random.default_rng(5)
    seq = "".join(rng.choice(list("ACGT"), size=len(text)))
    with open(other, "w") as f:
        at = 0
        for n, l in zip(names, lens):
            f.write(">%s\n%s\n" % (n, seq[at:at + l]))
            at += l
    expect_arg_error(gsx, tmp_path, sam, other, "off-target", "mismatches to the guide but is listed at distance")
    # a truncated of:H: in the middle of the file, and a list whose group distances are out of order
    lines = sam.splitlines(True)
    qn = [l.split("\t", 1)[0] if not l.startswith("@") else None for l in lines]
    k = [i for i in range(1, len(lines) - 1) if qn[i] and qn[i] != qn[i - 1] and qn[i] != qn[i + 1]][3]      # a guide of one record
    f = lines[k].rstrip("\n").split("\t")
    j = next(i for i, t in enumerate(f) if t.startswith("of:H:"))
    qname = f[0]
    f2 = list(f)
    f2[j] = f[j][:-7]
    expect_arg_error(gsx, tmp_path, "".join(lines[:k] + ["\t".join(f2) + "\n"] + lines[k + 1:]), fa, '"%s"' % qname, "truncated")
    vals = DO.hex_values(f[j][5:])
    d0 = vals.index(-(200000 + 1)) - 1
    f2[j] = "of:H:" + f[j][5:][:16 * d0] + (7).to_bytes(8, "little", signed=True).hex() + f[j][5:][16 * (d0 + 1):]
    expect_arg_error(gsx, tmp_path, "".join(lines[:k] + ["\t".join(f2) + "\n"] + lines[k + 1:]), fa, '"%s"' % qname, "groups")
    # a position of group 1 listed in group 0: the message names both distances
    delim = -(200000 + 1)

    def groups_of(i):
        f = lines[i].rstrip("\n").split("\t")
        j = next(c for c, t in enumerate(f) if t.startswith("of:H:"))
        return f, j, DO.groups(DO.hex_values(f[j][5:]), delim)
    one_record = [i for i in range(1, len(lines) - 1) if qn[i] and qn[i] != qn[i - 1] and qn[i] != qn[i + 1]]
    k1 = next(i for i in one_record if groups_of(i)[2][0][1] and len(groups_of(i)[2]) > 1 and groups_of(i)[2][1][1])
    f, j, g = groups_of(k1)
    g[0][1][0] = g[1][1][0]
    hexed = "".join(v.to_bytes(8, "little", signed=True).hex() for d, pos in g for v in pos + [d, delim])
    f[j] = "of:H:" + hexed
    expect_arg_error(gsx, tmp_path, "".join(lines[:k1] + ["\t".join(f) + "\n"] + lines[k1 + 1:]), fa, '"%s"' % f[0],
                     "has 1 mismatches to the guide but is listed at distance 0")
    # a delimiter that is not hex is reported as such, not as the group error it also causes
    f, j, g = groups_of(k1)
    n0 = len(g[0][1])
    v = f[j][5:]
    f[j] = "of:H:" + v[:16 * (n0 + 1)] + "zz" + v[16 * (n0 + 1) + 2:]
    msg = expect_arg_error(gsx, tmp_path, "".join(lines[:k1] + ["\t".join(f) + "\n"] + lines[k1 + 1:]), fa, '"%s"' % f[0],
                           "value %d of its of:H: list is not 16 hex digits" % (n0 + 1))
    assert "groups" not in msg
    # a succinct database
    r = ix.enumerate([(s, pam) for _, s, pam, _ in rows], gsx.make_params(mismatches=2, sam_scoring=True))
    succ = (ix.header("sam") + r.format(rows, gsx.make_params(mismatches=2, sam_scoring=True), "sam", "succinct")).decode()
    expect_arg_error(gsx, tmp_path, succ, fa, "succinct")
