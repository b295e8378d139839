"""`guidescan decode` / gsx_decode_database without a GPU: the plain-Python restatement of the decode (oracle/decode_oracle.py)
pinned to the reference's own goldens, the error cases it shares with the library, the library's checks that run before any device
work, and the command line's argument errors."""
import gzip
import os
import subprocess

import pytest

from conftest import GOLDEN, ROOT

import decode_oracle as DO

EXE = os.path.join(ROOT, "guidescan-cli_b200", "bin", "guidescan")


def golden_text(name):
    return gzip.open(os.path.join(GOLDEN, name + ".out.gz"), "rb").read().decode()


def unpack_fasta(tmp_path, case):
    fa = os.path.join(tmp_path, case + ".fa")
    open(fa, "wb").write(gzip.open(os.path.join(GOLDEN, case + ".fa.gz"), "rb").read())
    return fa


def write_sam(tmp_path, text, name="db.sam"):
    """the golden database without its PAM-less guide (a database decodes with one PAM column length)"""
    path = os.path.join(tmp_path, name)
    open(path, "w").write("".join(l for l in text.splitlines(True) if not l.startswith("no_pam\t")))
    return path


def without_specificity(lines):
    return [l.rsplit(",", 1)[0] for l in lines]


# ---- the restatement against the reference's goldens ---------------------------------------------------------------------------
@pytest.mark.parametrize("case", ["g200k", "g150kN"])
@pytest.mark.parametrize("sam,alts,csv,keep", [
    ("m2_sam", (), "m3_csv", lambda r: int(r[5]) <= 2),
    ("m3_altNAG_sam", ("NAG",), "m3_altNAG_NGA_csv", lambda r: r[6][-2:] in ("GG", "AG")),
])
def test_oracle_decodes_reference_sam_to_reference_csv(tmp_path, case, sam, alts, csv, keep):
    """m = 2 SAM against the m = 3 CSV's rows at distance <= 2, NGG + NAG SAM against the NGG + NAG + NGA CSV's xGG / xAG rows: with
    max-off-targets -1 the SAM and CSV rules keep the same hits; only the specificity differs"""
    fa = unpack_fasta(tmp_path, case)
    path = write_sam(tmp_path, golden_text("%s.%s" % (case, sam)))
    got = DO.decode(path, fa, alt_pams=alts).splitlines()
    assert got[0] == golden_text("%s.%s" % (case, csv)).splitlines()[0]
    ids = {l.split("\t")[0] for l in open(path) if not l.startswith("@")}
    want = [l for l in golden_text("%s.%s" % (case, csv)).splitlines()[1:]
            if l.split(",")[0] in ids and l.split(",")[2] != "NA" and keep(l.split(","))]
    assert len(want) > 50
    assert without_specificity(got[1:]) == without_specificity(want)
    # succinct: the same rows without the match and bulge columns
    succ = DO.decode(path, fa, alt_pams=alts, complete=False).splitlines()
    assert [l.split(",")[:6] for l in succ[1:]] == [l.split(",")[:6] for l in got[1:]]


def test_oracle_regions_select_by_on_target_site(tmp_path):
    fa = unpack_fasta(tmp_path, "g200k")
    path = write_sam(tmp_path, golden_text("g200k.m2_sam"))
    recs = [l.split("\t") for l in open(path) if not l.startswith("@")]
    chrom, pos = recs[0][2], int(recs[0][3])
    exact = DO.decode(path, fa, regions=[(chrom, pos - 1, pos - 1 + 23)]).splitlines()
    assert {l.split(",")[0] for l in exact[1:]} == {recs[0][0]}
    assert DO.decode(path, fa, regions=[(chrom, pos, pos + 23)]).splitlines()[1:] == []       # a base short at the left
    assert DO.decode(path, fa, regions=[]) == exact[0] + "\n"


# ---- malformed inputs: the restatement raises where the library returns GSX_ERR_ARG --------------------------------------------
def first_record(text):
    lines = text.splitlines(True)
    i = next(k for k, l in enumerate(lines) if not l.startswith("@"))
    return lines, i


def replace_of(line, of):
    f = line.rstrip("\n").split("\t")
    return "\t".join(t if not t.startswith("of:H:") else "of:H:" + of for t in f) + "\n"


def of_value(line):
    return next(t for t in line.rstrip("\n").split("\t") if t.startswith("of:H:"))[5:]


def test_oracle_rejects_a_broken_group(tmp_path):
    fa = unpack_fasta(tmp_path, "g200k")
    lines, i = first_record(golden_text("g200k.m2_sam"))
    of = of_value(lines[i])
    vals = DO.hex_values(of)
    j = next(k for k in range(1, len(vals)) if vals[k] == -(200000 + 1)) - 1         # the first group's distance 0 -> 1
    broken = of[:16 * j] + (1).to_bytes(8, "little", signed=True).hex() + of[16 * (j + 1):]
    lines[i] = replace_of(lines[i], broken)
    with pytest.raises(DO.DecodeError, match="group"):
        DO.decode(write_sam(tmp_path, "".join(lines)), fa)
    lines[i] = replace_of(lines[i], of[:-16])                                        # no closing delimiter
    with pytest.raises(DO.DecodeError):
        DO.decode(write_sam(tmp_path, "".join(lines)), fa)
    lines[i] = replace_of(lines[i], of[:-3])                                         # truncated inside a value
    with pytest.raises(DO.DecodeError, match="truncated"):
        DO.decode(write_sam(tmp_path, "".join(lines)), fa)


def test_oracle_rejects_succinct_and_differing_duplicates_and_another_assembly(tmp_path):
    fa = unpack_fasta(tmp_path, "g200k")
    with pytest.raises(DO.DecodeError, match="succinct"):
        DO.decode(write_sam(tmp_path, golden_text("g200k.m3_sam_succinct")), fa)
    lines, i = first_record(golden_text("g200k.m2_sam"))
    dup = replace_of(lines[i], of_value(lines[i])[:-48] + of_value(lines[i])[-32:])
    with pytest.raises(DO.DecodeError, match="same QNAME"):
        DO.decode(write_sam(tmp_path, "".join(lines[:i + 1] + [dup] + lines[i + 1:])), fa)
    with pytest.raises(DO.DecodeError, match="@SQ"):
        DO.decode(write_sam(tmp_path, golden_text("g200k.m2_sam")), unpack_fasta(tmp_path, "g150kN"))


# ---- the library's checks before any device work -------------------------------------------------------------------------------
def lib_decode(*a, **kw):
    gsx = pytest.importorskip("gsx", reason="libgsx.so not built")
    with pytest.raises(gsx.GsxError) as e:
        gsx.decode_database(*a, **kw)
    return e.value


def test_library_checks_without_a_device(tmp_path):
    if not os.path.exists(os.path.join(ROOT, "guidescan-cli_b200", "libgsx.so")):
        pytest.skip("libgsx.so not built")
    fa = unpack_fasta(tmp_path, "g200k")
    out = os.path.join(tmp_path, "o.csv")
    sam = write_sam(tmp_path, golden_text("g200k.m2_sam"))
    e = lib_decode(sam, fa, out, pam_length=0)
    assert e.code == 1 and "pam_length 0" in str(e)
    e = lib_decode(sam, fa, out, alt_pams=("NAGG",))
    assert e.code == 1 and "NAGG" in str(e)
    e = lib_decode(write_sam(tmp_path, golden_text("g200k.m3_sam_succinct"), "s.sam"), fa, out)
    assert e.code == 1 and "succinct" in str(e) and "at byte" in str(e)
    e = lib_decode(sam, unpack_fasta(tmp_path, "g150kN"), out)
    assert e.code == 1 and "@SQ line" in str(e) and "chr" in str(e)
    lines, i = first_record(golden_text("g200k.m2_sam"))
    lines[i] = replace_of(lines[i], of_value(lines[i])[:-5])
    e = lib_decode(write_sam(tmp_path, "".join(lines), "t.sam"), fa, out)
    assert e.code == 1 and '"%s"' % lines[i].split("\t")[0] in str(e) and "truncated" in str(e)
    # without @SQ lines: the delimiter of the first list names the other assembly
    body = "".join(l for l in golden_text("g200k.m2_sam").splitlines(True) if not l.startswith("@"))
    e = lib_decode(write_sam(tmp_path, body, "n.sam"), unpack_fasta(tmp_path, "g150kN"), out)
    assert e.code == 1 and "-200001" in str(e) and "-150001" in str(e)
    e = lib_decode(os.path.join(tmp_path, "missing.sam"), fa, out)
    assert e.code == 2


# ---- command line ----------------------------------------------------------------------------------------------------------------
def cli(*args):
    if not os.path.exists(EXE):
        pytest.skip("CLI not built")
    return subprocess.run([EXE, "decode"] + list(args), capture_output=True, text=True)


def test_cli_argument_errors():
    r = cli("db.sam", "-o", "out.csv")
    assert r.returncode == 106 and "--genome is required" in r.stderr
    r = cli("db.sam", "--genome", "g.fa", "-o", "out.csv", "--frobnicate")
    assert r.returncode == 109 and "--frobnicate" in r.stderr
    r = cli("db.sam", "--genome", "g.fa", "-o", "out.csv", "--pam-length", "0")
    assert r.returncode == 105 and "--pam-length" in r.stderr
    r = cli("db.sam", "--genome", "g.fa")
    assert r.returncode == 106 and "--output is required" in r.stderr
    r = cli("db.sam", "--genome", "g.fa", "-o", "out.csv", "--mode", "verbose")
    assert r.returncode == 105
    r = cli("db.sam", "--genome", "g.fa", "-o", "out.csv", "-a", "NAGG")
    assert r.returncode == 105 and "NAGG" in r.stderr
    r = subprocess.run([EXE, "--help"], capture_output=True, text=True)
    assert "decode [OPTIONS] DATABASE.sam" in r.stderr
