"""IUPAC class letters in PAMs on the GPU.  The definition the tests use: a search with class PAMs gives exactly the result of a search
with their concrete expansion (class letters replaced by their members, N kept) as the guide's PAM plus alternative PAMs -- every
hit, its order, match string, CFD, specificity, count_by_distance and threshold drop -- on every search path.  Plus: the CPU
oracle on a sample (NRRH too, which only the class form fits into one call), the option off (class letters never match, as before),
the generator, the one-pass genome enumeration and the decode round trip with "-" sense guides."""
import os
import subprocess

import numpy as np
import pytest

from conftest import ROOT
from test_decode_gpu import decode, enumerate_both, rows_with_sam_record
from test_skew_gpu import ENV_KNOBS, _run, _take
from test_split_gpu import _same

import kmers_oracle as KO
import oracle as O

pytestmark = [pytest.mark.gpu, pytest.mark.timeout(3600)]

N_GUIDES = 16384 + 37
G = 24_000_000
BIN = os.path.join(ROOT, "guidescan-cli_b200", "bin", "guidescan")
IUPAC = {"R": "AG", "Y": "CT", "S": "CG", "W": "AT", "K": "GT", "M": "AC", "B": "CGT", "D": "AGT", "H": "ACT", "V": "ACG"}


def classes(pam):
    """class letters replaced by their members, N kept (the concrete list a class PAM stands for in a search)"""
    out = [""]
    for c in pam:
        out = [s + b for s in out for b in IUPAC.get(c, c)]
    return out


def pam_set(pam):
    """kmers_oracle.pam_set with class letters expanded like N: breadth first, first expandable letter first, members in A, C, T, G order"""
    queue = [pam]
    exp = lambda p: next((i for i, c in enumerate(p) if c == "N" or c in IUPAC), None)
    while any(exp(p) is not None for p in queue):
        p = queue.pop(0)
        at = exp(p)
        if at is None:
            queue.append(p)
        else:
            queue.extend(p[:at] + c + p[at + 1:] for c in "ACTG" if c in IUPAC.get(p[at], "ACGT"))
    return queue


def generate(path, pam, **kw):
    old = KO.pam_set
    KO.pam_set = pam_set
    try:
        return KO.generate(path, pam=pam, **kw)
    finally:
        KO.pam_set = old


@pytest.fixture(scope="module")
def gsx():
    import gsx as g
    if g.device_count() < 1:
        pytest.fail("no CUDA device: the product has no CPU path")
    return g


@pytest.fixture(autouse=True)
def default_env(monkeypatch):
    for k in ENV_KNOBS + ("GSX_FUSED_PAMS",):
        monkeypatch.delenv(k, raising=False)


def _mutate(rng, s, d):
    s = list(s)
    for i in rng.choice(len(s), d, replace=False):
        s[i] = rng.choice([b for b in "ACGT" if b != s[i]])
    return "".join(s)


@pytest.fixture(scope="module")
def world(gsx, tmp_path_factory):
    """a 24 Mb genome with runs of N; 400 source guides with near-copies at distance 0..3 planted in front of (or, --start, behind)
    PAM spellings that cover every member of the classes, some non-members, and a literal N at class and at N positions"""
    import synth
    d = str(tmp_path_factory.mktemp("iupac"))
    rng = np.random.default_rng(20261022)
    g = synth.make_genome(G, 11)
    for s in rng.integers(1000, G - 10000, 40):                            # runs of N
        g[s:s + int(rng.integers(5, 3000))] = ord("N")
    text = g.tobytes().decode()
    sources = []
    variants = ["AGG", "AAG", "ACG", "ATG", "ANG", "NGG", "AGA", "CAGAAT", "CAGGGT", "CAGCAT", "CAGNAT", "NNGAGT", "AAGAAA"]
    starts = ["TTTA", "TTTC", "TTTG", "TTTT", "TTTN", "NTTA"]
    pieces, at = [], 0
    for k in range(400):
        p = int(rng.integers(20000, G - 20000))
        src = text[p:p + 20]
        if "N" in src:
            continue
        sources.append(src)
        for j in range(6):
            q = int(rng.integers(at + 100, at + 100 + (G - at) // 4000))
            if q + 40 >= G:
                break
            copy = _mutate(rng, src, int(rng.integers(0, 4)))
            site = copy + variants[int(rng.integers(len(variants)))] if j % 2 == 0 else starts[int(rng.integers(len(starts)))] + copy
            pieces.append((q, site))
            at = q + len(site)
    buf = bytearray(g.tobytes())
    for q, site in pieces:
        buf[q:q + len(site)] = site.encode()
    g = np.frombuffer(bytes(buf), dtype=np.uint8).copy()
    chroms = [("chr1", G // 2), ("chr2", G - G // 2)]
    fa = os.path.join(d, "g.fa")
    synth.write_fasta(fa, g, chroms)
    ix = gsx.Index.build(fa, devices=[0])
    ix2 = gsx.Index.build(fa, devices=[0, 0])
    yield dict(dir=d, fa=fa, ix=ix, ix2=ix2, sources=sources, rng=rng)
    ix.close()
    ix2.close()


def _guides(gsx, w, pam, start=False, n=N_GUIDES):
    """the sources plus generated guides of the class pattern (gsx.generate_kmers), as (seq, pam) pairs with the pattern as column"""
    out = os.path.join(w["dir"], "k_%s_%d.csv" % (pam, start))
    if not os.path.exists(out):
        gsx.generate_kmers(w["fa"], out, pam=pam, start=start)
    rows = open(out).read().splitlines()[1:]
    rng = np.random.default_rng(len(pam) * 7 + start)
    pick = rng.choice(len(rows), min(n - len(w["sources"]), len(rows)), replace=False)
    return [(s, pam) for s in w["sources"]] + [(rows[i].split(",")[1], pam) for i in sorted(pick)]


def _concrete(guides, alts, pam):
    """the same batch spelled concretely: column = first expansion of `pam`, alternative PAMs = the rest + the alts' expansions"""
    e = classes(pam)
    return [(s, e[0]) for s, _ in guides], e[1:] + [x for a in alts for x in classes(a)]


CASES = {            # name: (column, alternative PAMs, --start)
    "NRG": ("NRG", (), False),
    "NNGRRT": ("NNGRRT", (), False),
    "TTTV_start": ("TTTV", (), True),
    "NGG_aNRG": ("NGG", ("NRG",), False),
    "NRG_aNYG": ("NRG", ("NYG",), False),
}
PATHS = {            # name: (environment, extra parameters)
    "default": ({}, {}),
    "sweep0": ({"GSX_SWEEP": 0}, {}),
    "general": ({"GSX_FORCE_GENERAL": 1}, {}),
    "t1": ({}, {"threshold": 1}),
    "t2": ({}, {"threshold": 2}),
    "maxoff1": ({}, {"max_off_targets": 1}),
}


def _pair(gsx, ix, guides, col, alts, start, monkeypatch, env, extra, m=3):
    cg, calts = _concrete(guides, alts, col)
    a, ca = _run(gsx, ix, guides, gsx.make_params(mismatches=m, start=start, alt_pams=alts, iupac_pams=True, **extra), monkeypatch, **env)
    b, cb = _run(gsx, ix, cg, gsx.make_params(mismatches=m, start=start, alt_pams=calts, **extra), monkeypatch, **env)
    return a, ca, b, cb


@pytest.mark.parametrize("path", sorted(PATHS))
@pytest.mark.parametrize("case", sorted(CASES))
def test_class_equals_expansion(gsx, world, monkeypatch, case, path):
    col, alts, start = CASES[case]
    env, extra = PATHS[path]
    guides = _guides(gsx, world, col, start)
    if path == "general":
        guides = guides[:2000]
    a, ca, b, cb = _pair(gsx, world["ix"], guides, col, alts, start, monkeypatch, env, extra)
    _same(a, b)
    if "threshold" not in extra:
        assert a["n_hits"][:len(world["sources"])].sum() > len(world["sources"]) // 4     # the planted copies are found
    if path in ("default", "maxoff1"):
        assert ca["seeds"] > 0 and cb["seeds"] > 0                            # both on the sweep


@pytest.mark.parametrize("case", ["NRG", "NNGRRT"])
def test_class_equals_expansion_two_slots_and_bulges(gsx, world, monkeypatch, case):
    col, alts, start = CASES[case]
    guides = _guides(gsx, world, col, start)
    a, _, b, _ = _pair(gsx, world["ix2"], guides, col, alts, start, monkeypatch, {}, {})
    _same(a, b)
    one, _ = _run(gsx, world["ix"], guides, gsx.make_params(mismatches=3, alt_pams=alts, iupac_pams=True), monkeypatch)
    _same(a, one)
    sub = guides[:600]
    a, _, b, _ = _pair(gsx, world["ix"], sub, col, alts, start, monkeypatch, {}, {"rna_bulges": 1, "dna_bulges": 1}, m=2)
    _same(a, b)


def test_two_class_columns_in_one_call(gsx, world, monkeypatch):
    """NRG and NYG columns in one batch (the general kernel): each half equals its own expansion"""
    g1 = _guides(gsx, world, "NRG", False, 1500)
    g2 = [(s, "NYG") for s, _ in _guides(gsx, world, "NNGRRT", False, 1500)[400:]]
    both, _ = _run(gsx, world["ix"], g1 + g2, gsx.make_params(mismatches=3, iupac_pams=True), monkeypatch)
    for part, idx in ((g1, np.arange(len(g1))), (g2, np.arange(len(g1), len(g1) + len(g2)))):
        cg, calts = _concrete(part, (), part[0][1])
        want, _ = _run(gsx, world["ix"], cg, gsx.make_params(mismatches=3, alt_pams=calts), monkeypatch)
        _same(_take(both, idx), want)


def test_option_off_is_unchanged(gsx, world, monkeypatch):
    """without iupac_pams a class column never matches: no hits, NA rows, as before the option existed"""
    guides = _guides(gsx, world, "NRG", False, 3000)
    out, _ = _run(gsx, world["ix"], guides, gsx.make_params(mismatches=3), monkeypatch)
    assert out["n_hits"].sum() == 0 and np.all(out["specificity"] == 1.0) and not out["dropped"].any()
    out, _ = _run(gsx, world["ix"], guides, gsx.make_params(mismatches=3, alt_pams=("NYG",)), monkeypatch)
    assert out["n_hits"].sum() == 0


@pytest.mark.parametrize("col,start", [("NRG", False), ("NNGRRT", False), ("TTTV", True), ("NRRH", False)])
def test_against_cpu_oracle(gsx, world, monkeypatch, col, start):
    """a sample of about 200 guides against the CPU oracle given the concrete list (NRRH: 12 PAMs in one oracle call)"""
    guides = _guides(gsx, world, col, start, 600)[::3][:200]
    if col == "NRRH":
        guides = [(s, col) for s, _ in guides]
    out, _ = _run(gsx, world["ix"], guides, gsx.make_params(mismatches=2, start=start, iupac_pams=True), monkeypatch)
    e = classes(col)
    assert len(e) <= 17
    oix = O.Index(world["fa"])
    opts = O.make_opts(mismatches=2, start=start, alt_pams=e[1:])
    n_hits = 0
    for i, (s, _) in enumerate(guides):
        hits, spec, dropped = oix.hits(opts, s, e[0])
        f, n = int(out["first_hit"][i]), int(out["n_hits"][i])
        got = sorted(zip(out["abs_pos"][f:f + n].tolist(), out["distance"][f:f + n].tolist(), out["index_id"][f:f + n].tolist()))
        assert got == sorted((h[0], h[2], h[5]) for h in hits), (i, s)
        assert abs(float(out["specificity"][i]) - spec) <= 1e-6 * max(1.0, spec)
        n_hits += n
    assert n_hits > len(guides) // 2


@pytest.mark.parametrize("pam,start", [("NRG", False), ("NNGRRT", False), ("TTTV", True)])
def test_generator(gsx, world, tmp_path, pam, start):
    """kmers --pam with class letters: the restatement (kmers_oracle.generate with classes expanded like N)"""
    small = os.path.join(str(tmp_path), "s.fa")
    with open(world["fa"]) as f, open(small, "w") as o:
        lines = f.read().splitlines()
        o.write("\n".join(lines[:20000] + [">chr9"] + lines[50000:60000]) + "\n")
    out = os.path.join(str(tmp_path), "k.csv")
    n = gsx.generate_kmers(small, out, pam=pam, start=start)
    want = generate(small, pam, start=start)
    assert open(out).read() == want
    assert n == len(want.splitlines()) - 1


@pytest.mark.parametrize("devices", ["0", "0,0"])
def test_one_pass_cli(gsx, world, tmp_path, devices):
    """`enumerate --genome --pam NNGRRT` (class semantics set by itself) equals `kmers` + `enumerate -f --iupac-pam`, byte for byte"""
    small = os.path.join(str(tmp_path), "s.fa")
    with open(world["fa"]) as f, open(small, "w") as o:
        o.write("\n".join(f.read().splitlines()[:30000]) + "\n")
    idx = os.path.join(str(tmp_path), "s")
    subprocess.check_call([BIN, "index", "--index", idx, small], stdout=subprocess.DEVNULL)
    k = os.path.join(str(tmp_path), "k.csv")
    subprocess.check_call([BIN, "kmers", "--pam", "NNGRRT", "-o", k, small], stdout=subprocess.DEVNULL)
    a, b = os.path.join(str(tmp_path), "a.csv"), os.path.join(str(tmp_path), "b.csv")
    subprocess.check_call([BIN, "enumerate", idx, "--genome", small, "--pam", "NNGRRT", "-m", "2", "-o", a, "--devices", devices],
                          stdout=subprocess.DEVNULL)
    subprocess.check_call([BIN, "enumerate", idx, "-f", k, "--iupac-pam", "-m", "2", "-o", b, "--devices", devices], stdout=subprocess.DEVNULL)
    ta, tb = open(a, "rb").read(), open(b, "rb").read()
    assert ta == tb and ta.count(b"\n") > 100
    r = subprocess.run([BIN, "enumerate", idx, "-f", k, "-m", "2", "-o", b], capture_output=True)
    assert r.returncode == 0 and open(b, "rb").read() != ta                  # without --iupac-pam: NA rows only


def test_decode_round_trip(gsx, world, tmp_path):
    """a class-column SAM complete database with "-" sense guides decodes to enumerate's CSV rows; "-" SEQ carries the IUPAC complement"""
    guides = _guides(gsx, world, "NRG", False, 1200)
    rows = [("g%d" % i, s, p, i % 2 == 0) for i, (s, p) in enumerate(guides)]
    r, sam, csv = enumerate_both(gsx, world["ix"], rows, mismatches=2, iupac_pams=True)
    r.close()
    minus = [l.split("\t") for l in sam.splitlines() if not l.startswith("@") and l.split("\t")[1] == "16"]
    assert minus and all(f[9].startswith("CYN") for f in minus)
    got = decode(gsx, str(tmp_path), sam, world["fa"], pam_length=3)
    assert got == rows_with_sam_record(csv, sam)
    r, sam2, csv2 = enumerate_both(gsx, world["ix"], [(i, s, "NGG", pos) for i, s, _, pos in rows], mismatches=2, alt_pams=("NRG",),
                                   iupac_pams=True)
    r.close()
    assert decode(gsx, str(tmp_path), sam2, world["fa"], name="alt", pam_length=3, alt_pams=("NRG",)) == rows_with_sam_record(csv2, sam2)
