"""Two-part sweep (sweep_split_kernel: distal half with at most one substitution, or the guide read PAM-first in the other strand's
index with at most one substitution in its proximal half, re-anchored afterwards): the same result arrays as the plain sweep
(GSX_SPLIT=0), field by field, and the same text as the CPU oracle."""
import os

import numpy as np
import pytest

pytestmark = [pytest.mark.gpu, pytest.mark.timeout(900)]


@pytest.fixture(scope="module")
def gsx():
    import gsx as g
    if g.device_count() < 1:
        pytest.fail("no CUDA device: the product has no CPU path")
    return g


def _build(gsx, fa, devices=(0,)):
    """an index whose jump table holds both capped halves of the two-part sweep (L = 13; genomes of a few Mb get 9)"""
    old = os.environ.get("GSX_FTAB")
    os.environ["GSX_FTAB"] = "13"
    try:
        return gsx.Index.build(fa, devices=list(devices))
    finally:
        if old is None:
            os.environ.pop("GSX_FTAB")
        else:
            os.environ["GSX_FTAB"] = old


def _guides_of_csv(path):
    rows = open(path).read().splitlines()[1:]
    return [(r.split(",")[1], r.split(",")[2]) for r in rows]


def _run(gsx, ix, guides, m, monkeypatch, split, sweep_min="1"):
    monkeypatch.setenv("GSX_SPLIT", split)
    monkeypatch.setenv("GSX_SWEEP_MIN", sweep_min)
    r = ix.enumerate(guides, gsx.make_params(mismatches=m))
    out = {k: np.array(v, copy=True) for k, v in r.guide_arrays().items()}
    out.update({k: np.array(v, copy=True) for k, v in r.hit_arrays().items()})
    out["match"] = np.array([r.match_sequence(h) for h in range(r.n_hits)], dtype=object)
    ctr = r.counters()
    r.close()
    return out, ctr


def _same(a, b):
    assert a.keys() == b.keys()
    for k in a:
        assert a[k].shape == b[k].shape, k
        assert np.array_equal(a[k], b[k]), k


def _check_split(gsx, ix, guides, m, monkeypatch, sweep_min="1"):
    old, c0 = _run(gsx, ix, guides, m, monkeypatch, "0", sweep_min)
    new, c1 = _run(gsx, ix, guides, m, monkeypatch, "1", sweep_min)
    _same(old, new)
    assert c0["seeds"] > 0 and c1["seeds"] > 0
    assert c1["launches"] > c0["launches"]                 # the two-part path really ran ...
    if m >= 2:
        assert c1["sectors"] < c0["sectors"]               # ... and requested fewer summary sectors (at m <= 1 the free PAM wildcard of form 1 costs more)
    assert (c1["matches"], c1["hits"]) == (c0["matches"], c0["hits"])
    return new, c1


@pytest.fixture(scope="module")
def seeded(gsx, tmp_path_factory):
    import synth
    d = str(tmp_path_factory.mktemp("split"))
    synth.make_dataset(d, 2_000_000, 5, 300, seed=31, name="s")
    fa, gcsv = os.path.join(d, "s.fa"), os.path.join(d, "s.guides.csv")
    ix = _build(gsx, fa)
    yield d, fa, gcsv, ix
    ix.close()


@pytest.mark.parametrize("m", [0, 1, 2, 3])
def test_split_matches_plain_sweep_and_oracle(gsx, seeded, monkeypatch, m):
    import oracle as O
    d, fa, gcsv, ix = seeded
    _check_split(gsx, ix, _guides_of_csv(gcsv), m, monkeypatch)
    want = os.path.join(d, "o%d.csv" % m)
    O.Index(fa).enumerate_file(O.make_opts(mismatches=m), gcsv, want, nthreads=8)
    monkeypatch.setenv("GSX_SPLIT", "1")
    out = os.path.join(d, "g%d.csv" % m)
    ix.enumerate_file(gcsv, out, gsx.make_params(mismatches=m))
    assert open(out, "rb").read() == open(want, "rb").read()


# mismatch positions of planted copies (0 = the PAM-distal end): both sides of the split after the tenth character, at g10 / g11
PLANTS = [(9,), (10,), (9, 10), (8, 9), (10, 11), (0, 5), (12, 18), (0, 5, 9), (10, 15, 19), (9, 10, 11), (3, 9, 12), (1, 14, 17),
          (0, 19), (2, 7, 11), (4, 6), (13, 16, 19)]


def _planted_dataset(d, G, n_guides, seed, repeats):
    import synth
    rng = np.random.default_rng(seed)
    g = synth.make_genome(G, seed)
    pos, kmers = synth.sample_guides(g, n_guides, seed)
    at = 1000
    step = (G - 4000) // (n_guides * (len(PLANTS) + repeats) + 1)
    comp = {ord("A"): ord("T"), ord("C"): ord("G"), ord("G"): ord("C"), ord("T"): ord("A")}
    for i in range(n_guides):
        copies = [(w, int(rng.integers(0, 2))) for w in PLANTS]
        if i < 3:                                           # a repeat family: 40 copies of one site with two distal mismatches
            copies += [((2, 7), 0)] * repeats
        for k, (where, rc) in enumerate(copies):
            c = kmers[i].copy()
            for w in where:
                c[w] = [b for b in b"ACGT" if b != c[w]][(i + w) % 3]
            c[20] = ord("A") if k >= len(PLANTS) else b"ACGT"[int(rng.integers(0, 4))]
            if rc:
                c = np.array([comp[b] for b in c[::-1]], dtype=np.uint8)
            g[at:at + 23] = c
            at += step
    chroms = synth.chromosome_table(G, 3)
    synth.write_fasta(os.path.join(d, "p.fa"), g, chroms)
    synth.write_guides_csv(os.path.join(d, "p.guides.csv"), pos, kmers, chroms)
    return os.path.join(d, "p.fa"), os.path.join(d, "p.guides.csv")


def test_planted_copies_on_both_sides_of_the_split(gsx, tmp_path, monkeypatch):
    """2 and 3 mismatches on either side of the split and at g10 / g11, on both strands, and repeat families whose PAM-first
    intervals hold more than 32 rows (the tree search takes those unexamined)"""
    import oracle as O
    d = str(tmp_path)
    fa, gcsv = _planted_dataset(d, 2_500_000, 60, 5, repeats=40)
    ix = _build(gsx, fa)
    try:
        new, _ = _check_split(gsx, ix, _guides_of_csv(gcsv), 3, monkeypatch)
        assert (new["distance"] == 3).sum() >= 60 * 6 and (new["distance"] == 2).sum() >= 60 * 7
        want = os.path.join(d, "o.csv")
        O.Index(fa).enumerate_file(O.make_opts(mismatches=3), gcsv, want, nthreads=8)
        out = os.path.join(d, "g.csv")
        monkeypatch.setenv("GSX_SPLIT", "1")
        ix.enumerate_file(gcsv, out, gsx.make_params(mismatches=3))
        assert open(out, "rb").read() == open(want, "rb").read()
    finally:
        ix.close()


@pytest.mark.parametrize("n_guides", [8192, 8192 + 37])
def test_default_sized_and_uneven_batches(gsx, tmp_path, monkeypatch, n_guides):
    """batches at and above the sweep's default minimum, one of them not a multiple of 32 guides"""
    import synth
    d = str(tmp_path)
    synth.make_dataset(d, 2_000_000, 4, n_guides, seed=41, name="b")
    ix = _build(gsx, os.path.join(d, "b.fa"))
    try:
        _check_split(gsx, ix, _guides_of_csv(os.path.join(d, "b.guides.csv")), 3, monkeypatch, sweep_min="8192")
    finally:
        ix.close()


def test_two_job_slots(gsx, seeded, monkeypatch):
    d, fa, gcsv, ix = seeded
    guides = _guides_of_csv(gcsv)
    one, _ = _run(gsx, ix, guides, 3, monkeypatch, "0")
    ix2 = _build(gsx, fa, devices=(0, 0))
    try:
        two, _ = _run(gsx, ix2, guides, 3, monkeypatch, "1")
    finally:
        ix2.close()
    _same(one, two)


def test_genome_with_n_keeps_the_plain_sweep(gsx, tmp_path, monkeypatch):
    """an index with N rows is not eligible: GSX_SPLIT changes nothing there"""
    import synth
    d = str(tmp_path)
    synth.make_dataset(d, 2_000_000, 4, 200, seed=43, name="n", n_runs_of_N=30)
    ix = _build(gsx, os.path.join(d, "n.fa"))
    try:
        guides = _guides_of_csv(os.path.join(d, "n.guides.csv"))
        old, c0 = _run(gsx, ix, guides, 3, monkeypatch, "0")
        new, c1 = _run(gsx, ix, guides, 3, monkeypatch, "1")
        _same(old, new)
        assert c1["launches"] == c0["launches"] and c1["sectors"] == c0["sectors"]
    finally:
        ix.close()
