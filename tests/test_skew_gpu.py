"""The default search path on skewed genomes (synth.add_skew, what `bench.py --skew` runs): Zipf repeat families of 10..3000
near-copies and low-complexity tracts, 1 % of the guides drawn from each.  Uniform genomes almost never reach what these guides do:
table entries of more than 32 rows (passed to the tree search unexamined) and of 17..32 rows (parked and drained), the PAM-first form of
the two-part sweep over GG-rich text, queue and arena growth, the radix ordering and the warp-per-guide specificity chosen from the
data, thousands of hits per guide through locate, --max-off-targets, SAM and decode.  Everything against the CPU oracle or, field
by field, against every other search path."""
import ctypes as C
import os
import time

import numpy as np
import pytest

from conftest import canonical_blocks
from test_decode_gpu import decode, enumerate_both, rows_with_sam_record
from test_split_gpu import _build, _same

pytestmark = [pytest.mark.gpu, pytest.mark.timeout(1800)]

N_GUIDES = 16384 + 37                  # above the sweep's default minimum batch (GSX_SWEEP_MIN), and not a multiple of 32
SAM_BYTES_PER_GUIDE = 1_000_000        # SAM complete repeats a guide's of:H: list once per perfect match: keep each guide's text bounded
GUIDE_KEYS = ("dropped", "first_hit", "n_hits", "specificity", "perfect_match", "count_by_distance")
ENV_KNOBS = ("GSX_SPLIT", "GSX_SWEEP", "GSX_SWEEP_MIN", "GSX_SWEEP_VARIANT", "GSX_FORCE_GENERAL", "GSX_ORDER", "GSX_ORDER_CTA",
             "GSX_SPEC_WARP", "GSX_QUEUE_CAP", "GSX_MATCH_CAP", "GSX_SPILL_CAP", "GSX_FTAB")


@pytest.fixture(scope="module")
def gsx():
    import gsx as g
    if g.device_count() < 1:
        pytest.fail("no CUDA device: the product has no CPU path")
    return g


@pytest.fixture(autouse=True)
def default_env(monkeypatch):
    """every test starts from the default path: no search knob set"""
    for k in ENV_KNOBS:
        monkeypatch.delenv(k, raising=False)


def _write_csv(path, lines, keep):
    with open(path, "w") as f:
        f.write("\n".join([lines[0]] + [lines[1 + i] for i in keep]) + "\n")
    return path


def _arrays(gsx, r):
    out = {k: np.array(v, copy=True) for k, v in r.guide_arrays().items()}
    out.update({k: np.array(v, copy=True) for k, v in r.hit_arrays().items()})
    buf, f = C.create_string_buffer(64), gsx._L.gsx_result_match_sequence
    seqs = []
    for h in range(r.n_hits):
        if f(r.h, h, buf, 64) != 0:
            raise gsx.GsxError(1, "gsx_result_match_sequence")
        seqs.append(buf.value)
    out["match"] = np.array(seqs, dtype=object)
    return out


def _run(gsx, ix, guides, params, monkeypatch, **env):
    """result arrays (with every hit's match sequence) and counters of one enumerate call under the GSX_* settings `env`"""
    with monkeypatch.context() as mp:
        for k, v in env.items():
            mp.setenv(k, str(v))
        t0 = time.time()
        r = ix.enumerate(guides, params)
        try:
            out, ctr = _arrays(gsx, r), r.counters()
        finally:
            r.close()
    ctr["seconds"] = time.time() - t0
    return out, ctr


def _take(out, idx):
    """the result of the guides `idx` (ascending) cut out of a whole-batch result, with first_hit rebased"""
    first, nh = out["first_hit"].astype(np.int64), out["n_hits"].astype(np.int64)
    hits = np.concatenate([np.arange(first[i], first[i] + nh[i]) for i in idx]) if len(idx) else np.zeros(0, np.int64)
    res = {k: v[idx] if k in GUIDE_KEYS else v[hits] for k, v in out.items()}
    res["first_hit"] = np.concatenate([[0], np.cumsum(nh[idx])[:-1]]).astype(out["first_hit"].dtype)
    return res


@pytest.fixture(scope="module")
def skewed(gsx, tmp_path_factory):
    """24 Mb, 4 chromosomes, bench.make_workload's recipe with add_skew: 164 repeat families and 164 low-complexity guides"""
    import oracle as O
    import synth
    d = str(tmp_path_factory.mktemp("skew"))
    G, seed = 24_000_000, 1
    g = synth.make_genome(G, seed)
    pos, kmers = synth.sample_guides(g, N_GUIDES, seed)
    synth.plant(g, kmers[:2000], seed)
    kmers, fam, low = synth.add_skew(g, kmers, seed, frac=0.01, lowc_mb=1.0, max_copies=3000)
    chroms = synth.chromosome_table(G, 4)
    fa, gcsv = os.path.join(d, "k.fa"), os.path.join(d, "k.guides.csv")
    synth.write_fasta(fa, g, chroms)
    synth.write_guides_csv(gcsv, pos, kmers, chroms)
    lines = open(gcsv).read().splitlines()
    guides = [(l.split(",")[1], "NGG") for l in lines[1:]]
    ix = _build(gsx, fa)                      # GSX_FTAB=13: a 24 Mb genome gets a depth-9 table, the two-part sweep needs 13
    oix = O.Index(fa)
    # the skew is really there, measured on the oracle's m = 3 text (test_default_path_matches_oracle compares the GPU's with it)
    oix.enumerate_file(O.make_opts(mismatches=3), gcsv, os.path.join(d, "o_m3"), nthreads=os.cpu_count() or 8)
    row = {("g%d" % i): i for i in range(N_GUIDES)}
    nh, perfect = np.zeros(N_GUIDES, np.int64), np.zeros(N_GUIDES, np.int64)
    with open(os.path.join(d, "o_m3")) as f:
        next(f)
        for line in f:
            t = line.split(",", 6)
            nh[row[t[0]]] += 1
            perfect[row[t[0]]] += t[5] == "0"
    assert nh.max() > 2048                    # ... some guide has thousands of hits
    assert nh.mean() > 64                     # ... the job picks the warp-per-guide specificity kernel by itself (gsx_api.cpp specificity())
    # every family guide has its site plus 10..3000 near-copies; a later family's copy or a tract overwrites a copy now and then
    # (about 5 % of them at this density), so a family of 10 may keep 8
    assert nh[fam].min() >= 8 and (nh[fam] >= 10).mean() >= 0.9
    rest = np.setdiff1d(np.arange(N_GUIDES), np.concatenate([fam, low]))
    others = np.sort(np.random.default_rng(0).choice(rest, 2000, replace=False))
    sample = np.unique(np.concatenate([fam, low, others]))
    # guides whose SAM complete text stays small: max(1, perfect matches) x hits x 16 hex digits
    light = np.nonzero(np.maximum(perfect, 1) * nh * 16 <= SAM_BYTES_PER_GUIDE)[0]
    mp = pytest.MonkeyPatch()
    for k in ENV_KNOBS:
        mp.delenv(k, raising=False)
    base3, c3 = _run(gsx, ix, guides, gsx.make_params(mismatches=3), mp)
    mp.undo()
    print("\nskew fixture: hits per guide max %d mean %.1f; family guides min %d median %d max %d; low-complexity guides min %d max %d; "
          "m=3 default: seeds %d launches %d matches %d hits %d, %.1f s; %d guides with bounded SAM text"
          % (nh.max(), nh.mean(), nh[fam].min(), np.median(nh[fam]), nh[fam].max(), nh[low].min(), nh[low].max(),
             c3["seeds"], c3["launches"], c3["matches"], c3["hits"], c3["seconds"], len(light)))
    yield dict(d=d, fa=fa, gcsv=gcsv, lines=lines, guides=guides, ix=ix, oix=oix, fam=np.sort(fam), low=np.sort(low), sample=sample,
               light=light, nh=nh, base3=base3, c3=c3)
    oix.close()
    ix.close()


CASES = {"m0": (dict(mismatches=0), "csv", False), "m1": (dict(mismatches=1), "csv", False), "m2": (dict(mismatches=2), "csv", False),
         "m3": (dict(mismatches=3), "csv", False), "m3_sam": (dict(mismatches=3), "sam", True),
         "m3_max5": (dict(mismatches=3, max_off_targets=5), "csv", False)}


@pytest.mark.parametrize("case", sorted(CASES))
def test_default_path_matches_oracle(gsx, skewed, monkeypatch, case):
    """the whole batch (for SAM complete: the guides whose text stays bounded, still more than the sweep's minimum) through the
    default path with no knob, byte for byte against the oracle; the counters show that the two-part sweep ran"""
    import oracle as O
    kw, fmt, light = CASES[case]
    d = skewed["d"]
    gcsv = skewed["gcsv"]
    if light:
        assert len(skewed["light"]) >= 8192 and np.isin(skewed["low"], skewed["light"]).sum() >= 8
        gcsv = _write_csv(os.path.join(d, "light.csv"), skewed["lines"], skewed["light"])
    want = os.path.join(d, "o_%s" % case)
    if case != "m3":                          # (the fixture's)
        skewed["oix"].enumerate_file(O.make_opts(fmt=fmt, **kw), gcsv, want, nthreads=os.cpu_count() or 8)
    p = gsx.make_params(**kw)
    got = os.path.join(d, "g_%s" % case)
    _, c1 = skewed["ix"].enumerate_file(gcsv, got, p, fmt=fmt)
    want_b = open(want, "rb").read()
    assert open(got, "rb").read() == want_b
    monkeypatch.setenv("GSX_SPLIT", "0")
    _, c0 = skewed["ix"].enumerate_file(gcsv, got, p, fmt=fmt)
    assert open(got, "rb").read() == want_b
    assert c1["seeds"] > 0 and c1["launches"] > c0["launches"], (c1, c0)
    if kw["mismatches"] >= 2:
        assert c1["sectors"] < c0["sectors"]
    if case == "m3":
        print("\nm=3 seeds: default %d, GSX_SPLIT=0 %d; launches %d / %d" % (c1["seeds"], c0["seeds"], c1["launches"], c0["launches"]))


@pytest.mark.parametrize("m", [0, 1, 2, 3])
def test_every_search_path_gives_the_same_arrays(gsx, skewed, monkeypatch, m):
    """two-part sweep (default), lean sweep, sweep_kernel, tree search from the jump table, search_kernel: the same arrays, field by
    field; at m = 3 also every match ordering and both specificity kernels"""
    ix, guides = skewed["ix"], skewed["guides"]
    p = gsx.make_params(mismatches=m)
    base = skewed["base3"] if m == 3 else _run(gsx, ix, guides, p, monkeypatch)[0]
    for env in (dict(GSX_SPLIT=0), dict(GSX_SWEEP_VARIANT=2), dict(GSX_SWEEP=0)):
        _same(base, _run(gsx, ix, guides, p, monkeypatch, **env)[0])
    # search_kernel (the general path) on the family and low-complexity guides and 2 000 others, against the same guides' part of
    # the default whole-batch result
    sample = skewed["sample"]
    general, _ = _run(gsx, ix, [guides[i] for i in sample], p, monkeypatch, GSX_FORCE_GENERAL=1)
    _same(_take(base, sample), general)
    if m == 3:
        launches = {}
        for env in (dict(GSX_ORDER=0), dict(GSX_ORDER=1), dict(GSX_ORDER=2), dict(GSX_SPEC_WARP=0), dict(GSX_SPEC_WARP=1)):
            out, ctr = _run(gsx, ix, guides, p, monkeypatch, **env)
            _same(base, out)
            launches[tuple(env.items())] = ctr["launches"]
        # the default chose the radix ordering by itself: as many launches as GSX_ORDER=2 (+1: the probe of the largest match count)
        c3 = skewed["c3"]
        print("\nlaunches: default %d, %s" % (c3["launches"], launches))
        assert c3["launches"] in (launches[(("GSX_ORDER", 2),)], launches[(("GSX_ORDER", 2),)] + 1)


def _m4_batch(skewed):
    """the guides whose SAM complete text stays bounded (at m = 3), minus those with more than 20 000 hits at m = 3"""
    nh = skewed["nh"]
    return np.array([i for i in skewed["light"] if nh[i] <= 20000])


def test_m4_nag_sam_against_oracle(gsx, skewed):
    """m = 4 with NAG: fused PAMs and the lean sweep variant 11 (xor table in global memory); SAM complete, per-guide blocks of the
    whole batch against the oracle's text of the family / low-complexity guides and 2 000 others"""
    import oracle as O
    d, lines = skewed["d"], skewed["lines"]
    batch = _m4_batch(skewed)
    assert len(batch) >= 8192
    gcsv = _write_csv(os.path.join(d, "m4.csv"), lines, batch)
    sub = np.intersect1d(batch, skewed["sample"])
    assert np.isin(skewed["fam"], sub).sum() >= 100 and np.isin(skewed["low"], sub).sum() >= 2
    scsv = _write_csv(os.path.join(d, "m4_sub.csv"), lines, sub)
    want = os.path.join(d, "o_m4.sam")
    skewed["oix"].enumerate_file(O.make_opts(mismatches=4, alt_pams=("NAG",), fmt="sam"), scsv, want, nthreads=os.cpu_count() or 8)
    got = os.path.join(d, "g_m4.sam")
    skewed["ix"].enumerate_file(gcsv, got, gsx.make_params(mismatches=4, alt_pams=("NAG",)), fmt="sam")
    hw, bw = canonical_blocks(open(want).read(), "sam")
    hg, bg = canonical_blocks(open(got).read(), "sam")
    assert hw == hg
    ids = ["g%d" % i for i in sub]
    assert sum(1 for i in ids if i in bw) > len(ids) // 2
    for i in ids:
        assert bg.get(i) == bw.get(i), i


def test_retries_under_skew(gsx, skewed, monkeypatch):
    """tiny first sizes of both seed queues, the match arena, the re-anchor arena and the spill stack: grown and retried, same arrays"""
    ix, guides = skewed["ix"], skewed["guides"]
    caps = dict(GSX_QUEUE_CAP=4096, GSX_MATCH_CAP=1024, GSX_SPILL_CAP=64)
    small, _ = _run(gsx, ix, guides, gsx.make_params(mismatches=3), monkeypatch, **caps)
    _same(skewed["base3"], small)
    batch = [guides[i] for i in _m4_batch(skewed)]
    p4 = gsx.make_params(mismatches=4, alt_pams=("NAG",))
    _same(_run(gsx, ix, batch, p4, monkeypatch)[0], _run(gsx, ix, batch, p4, monkeypatch, **caps)[0])


def test_bulges_through_edited_guides(gsx, skewed):
    """m = 1, R = D = 1 on 64 family guides and the 4 lightest low-complexity guides: thousands of matches per guide.  (Bulge output
    grows fast on this text: the next lightest low-complexity guides print about 80 MB of CSV each.)"""
    import oracle as O
    d, lines = skewed["d"], skewed["lines"]
    nh, low = skewed["nh"], skewed["low"]
    pick = np.sort(np.concatenate([np.random.default_rng(1).choice(skewed["fam"], 64, replace=False),
                                   low[np.argsort(nh[low], kind="stable")[:4]]]))
    gcsv = _write_csv(os.path.join(d, "bulge.csv"), lines, pick)
    kw = dict(mismatches=1, rna_bulges=1, dna_bulges=1)
    want, got = os.path.join(d, "o_bulge.csv"), os.path.join(d, "g_bulge.csv")
    skewed["oix"].enumerate_file(O.make_opts(**kw), gcsv, want, nthreads=os.cpu_count() or 8)
    skewed["ix"].enumerate_file(gcsv, got, gsx.make_params(**kw))
    w = open(want, "rb").read()
    assert w.count(b"\n") > 68 * 50
    assert open(got, "rb").read() == w


def test_two_job_slots(gsx, skewed, monkeypatch):
    """an index on [0, 0]: each slot runs its own shard of the batch, one of them with the heavy guides"""
    ix2 = _build(gsx, skewed["fa"], devices=(0, 0))
    try:
        two, _ = _run(gsx, ix2, skewed["guides"], gsx.make_params(mismatches=3), monkeypatch)
    finally:
        ix2.close()
    _same(skewed["base3"], two)


def test_decode_round_trip(gsx, skewed, tmp_path, monkeypatch):
    """the SAM complete database of the bounded-text guides at m = 3 decodes to enumerate's CSV rows, with batches smaller than its
    longest record (an of:H: list of more than 10^4 entries)"""
    rows = [r for k, r in enumerate(gsx.read_guides_csv(skewed["gcsv"])) if k in set(skewed["light"].tolist())]
    _, sam, csv = enumerate_both(gsx, skewed["ix"], rows, mismatches=3)
    longest = max(len(l) for l in sam.splitlines() if not l.startswith("@"))
    assert longest > 16 * 10_000
    monkeypatch.setenv("GSX_DECODE_BATCH_BYTES", str(longest // 3))
    want = rows_with_sam_record(csv, sam)
    assert len(want.splitlines()) > 100_000
    assert decode(gsx, str(tmp_path), sam, skewed["fa"]) == want


COMP = np.zeros(256, dtype=np.uint8)
for _a, _b in zip(b"ACGTN", b"TGCAN"):
    COMP[_a] = _b


def _format_guide(gsx, r, p, k, gid, seq):
    row = (gsx.GuideRow * 1)(gsx.GuideRow(gid.encode(), seq.encode(), b"NGG", 1))
    buf, ln = C.c_void_p(), C.c_size_t()
    gsx._ck(gsx._L.gsx_format_rows(r.index.h, r.h, row, k, k + 1, C.byref(p), 0, 1, C.byref(buf), C.byref(ln)), "gsx_format_rows")
    out = C.string_at(buf, ln.value).decode()
    gsx._L.gsx_free(buf)
    return out


@pytest.mark.timeout(1500)
def test_realistic_density_depth_14(gsx, monkeypatch):
    """1.1 Gb (n >= 4^15: the default jump table has depth 14, as at 3.1 Gb), 50 000 guides with bench.py --skew's defaults, no knob:
    the same arrays as the lean sweep, every hit re-verified against the text, the float32 specificity of every family and
    low-complexity guide recomputed in hit order, and 200 guides against the oracle over the exported BWT"""
    import oracle as O
    import synth
    for k in ENV_KNOBS:
        monkeypatch.delenv(k, raising=False)
    G, n, seed = 1_100_000_000, 50_000, 5
    t0 = time.time()
    g = synth.make_genome(G, seed)
    pos, kmers = synth.sample_guides(g, n, seed)
    synth.plant(g, kmers[:2000], seed)
    kmers, fam, low = synth.add_skew(g, kmers, seed, frac=0.01, lowc_mb=2.0, max_copies=10000)
    chroms = synth.chromosome_table(G, 8)
    ix = gsx.Index.build_from_text(g, chroms, sa_shift=6, devices=[0])
    t_build = time.time() - t0
    p = gsx.make_params(mismatches=3)
    arr = (gsx.Guide * n)()
    keep = [kmers[i, :20].tobytes() for i in range(n)]
    for i, sq in enumerate(keep):
        arr[i] = gsx.Guide(sq, b"NGG")

    def run(**env):
        with monkeypatch.context() as mp:
            for k, v in env.items():
                mp.setenv(k, str(v))
            r = ix.enumerate_raw(arr, n, p)
        out = {k: np.array(v, copy=True) for k, v in r.guide_arrays().items()}
        out.update({k: np.array(v, copy=True) for k, v in r.hit_arrays().items()})
        return r, out, r.counters()
    try:
        r0, lean, cl = run(GSX_SPLIT=0)
        r0.close()
        r, ref, c = run()
        _same(lean, ref)
        del lean, ref
        assert c["seeds"] > 0 and c["launches"] > cl["launches"]
        ga, ha = r.guide_arrays(), r.hit_arrays()
        nhit = ga["n_hits"].astype(np.int64)
        first = ga["first_hit"].astype(np.int64)
        assert nhit.max() > 2048 and nhit.mean() > 64
        hit_guide = np.repeat(np.arange(n), nhit)
        # every hit is a true site: guide orientation at the reported position, `distance` mismatches, xGG
        ab = ha["abs_pos"]
        for s in range(0, len(ab), 1 << 21):
            a = ab[s:s + (1 << 21)]
            minus = a < 0
            start = np.where(minus, -a, a - 22)
            assert np.all((start >= 0) & (start + 23 <= G))
            txt = g[start[:, None] + np.arange(23)[None, :]]
            txt[minus] = COMP[txt[minus][:, ::-1]]
            gk = kmers[hit_guide[s:s + (1 << 21)]]
            mism = (txt[:, :20] != gk[:, :20]).sum(axis=1)
            assert np.array_equal(mism, ha["distance"][s:s + (1 << 21)].astype(np.int64))
            assert np.all(txt[:, 21] == ord("G")) and np.all(txt[:, 22] == ord("G"))
        # float32 specificity in hit order (printer.hpp): 1 / (sum of the counted CFDs, +1 without a perfect match)
        cfd, counted, spec = ha["cfd"], ha["counted"], ga["specificity"]
        for gi in np.concatenate([fam, low]):
            b, k = int(first[gi]), int(nhit[gi])
            if k == 0:
                assert spec[gi] == np.float32(1.0)
                continue
            v = cfd[b:b + k][counted[b:b + k] != 0]
            ssum = np.add.accumulate(v, dtype=np.float32)[-1] if len(v) else np.float32(0.0)
            if not ga["perfect_match"][gi]:
                ssum = np.float32(ssum + np.float32(1.0))
            assert spec[gi] == (np.float32(1.0) / ssum if ssum > 0 else np.float32(0.0)), gi
        # 200 guides through the oracle over the exported BWT: the 50 largest families, 50 low-complexity guides, 100 others
        big = fam[np.argsort(nhit[fam], kind="stable")[::-1][:50]]
        lows = np.random.default_rng(0).choice(low, 50, replace=False)
        rest = np.setdiff1d(np.arange(n), np.concatenate([fam, low]))
        pick = np.sort(np.concatenate([big, lows, np.random.default_rng(1).choice(rest, 100, replace=False)]))
        oix = O.Index.from_bwt(ix.export_bwt(0), ix.export_sa_samples(0)[0], ix.export_bwt(1), ix.export_sa_samples(1)[0], chroms)
        import tempfile
        with tempfile.TemporaryDirectory() as d:
            gcsv = os.path.join(d, "s.csv")
            with open(gcsv, "w") as f:
                f.write("id,sequence,pam,chromosome,position,sense\n")
                for i in pick:
                    f.write("g%d,%s,NGG,chr1,1,+\n" % (i, kmers[i, :20].tobytes().decode()))
            want = os.path.join(d, "o.csv")
            oix.enumerate_file(O.make_opts(mismatches=3), gcsv, want, nthreads=os.cpu_count() or 8)
            _, bw = canonical_blocks(open(want).read(), "csv")
        oix.close()
        for i in pick:
            got = _format_guide(gsx, r, p, int(i), "g%d" % i, kmers[i, :20].tobytes().decode())
            assert got.splitlines() == bw.get("g%d" % i), i
        print("\n1.1 Gb: built in %.0f s; hits per guide max %d mean %.1f; seeds %d (GSX_SPLIT=0: %d); %d hits; %.0f s in all"
              % (t_build, nhit.max(), nhit.mean(), c["seeds"], cl["seeds"], len(ab), time.time() - t0))
        r.close()
    finally:
        ix.close()
