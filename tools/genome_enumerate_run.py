#!/usr/bin/env python
"""`guidescan enumerate --genome` (generation and enumeration in one pass) against the two-step path it replaces
(`guidescan kmers` -> guides CSV -> `guidescan enumerate -f`), on the 3.1 Gb synthetic genome of bench.py (sa_shift = 2, as
tools/config5_run.py builds it), configs[4] options: m = 4, -a NAG, SAM complete, on N GPUs of one box.

  equality   the first --check-mb Mb of chr1 as a BED region, both paths written to files: byte-identical?
  rate       chr1 whole to /dev/null: (a) kmers over a chr1-only FASTA, then enumerate -f; (b) enumerate --genome over the full
             FASTA with a BED covering chr1 (the same guides).  Wall, guides/s, the GSX_FILE_TIMING line, peak RSS of each process,
             device ms per batch.
  --whole-genome  every guide of the genome through (b) without regions, to /dev/null.

  python tools/genome_enumerate_run.py --gpus 8 [--whole-genome] --out profiles/r03a_genome_enumerate_8gpu.json
"""
import argparse
import hashlib
import json
import os
import re
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "guidescan-cli_b200"))
EXE = os.path.join(ROOT, "guidescan-cli_b200", "bin", "guidescan")
# runs one command and reports its own peak RSS: RUSAGE_CHILDREN of a process whose only child is that command
RSS_WRAPPER = ("import resource, subprocess, sys\n"
               "r = subprocess.run(sys.argv[1:])\n"
               "sys.stderr.write('\\npeak_rss_kb %d\\n' % resource.getrusage(resource.RUSAGE_CHILDREN).ru_maxrss)\n"
               "sys.exit(r.returncode)\n")


def log(*a):
    print(*a, file=sys.stderr, flush=True)


def run_cli(args, env):
    t0 = time.time()
    r = subprocess.run([sys.executable, "-c", RSS_WRAPPER, EXE] + args, capture_output=True, text=True,
                       env={**os.environ, "GSX_FILE_TIMING": "1", **env})
    dt = time.time() - t0
    if r.returncode:
        raise RuntimeError("guidescan %s failed: %s" % (" ".join(args), r.stderr[-800:]))
    out = {"args": args, "wall_s": dt, "peak_rss_gb": int(re.search(r"peak_rss_kb (\d+)", r.stderr).group(1)) / 1e6}
    m = re.search(r"Processed (\d+) kmers in \d+ seconds. \(([\d.]+) s, ([\d.]+) kmers/s; device ([\d.]+) ms", r.stdout)
    if m:
        out.update(guides=int(m.group(1)), enumerate_s=float(m.group(2)), guides_per_s_in_call=float(m.group(3)), device_ms_sum=float(m.group(4)))
    timing = [l for l in r.stderr.splitlines() if l.startswith("gsx file job:")]
    if timing:
        out["file_job_timing"] = timing[-1]
        t = re.search(r"(\d+) guides in batches of (\d+).*calls: device ([\d.]+) s", timing[-1])
        n, b, dev = int(t.group(1)), int(t.group(2)), float(t.group(3))
        out["batches"] = -(-n // b)
        out["device_ms_per_batch"] = 1e3 * dev / max(1, out["batches"])
        s = re.search(r"PAM scan ([\d.]+) s over (\d+) chromosome\(s\) \(\+ ([\d.]+) s waiting", timing[-1])
        if s:
            out.update(scan_s=float(s.group(1)), scan_chromosomes=int(s.group(2)), scan_wait_s=float(s.group(3)))
    o = re.search(r"files ([\d.]+) s, device layout ([\d.]+) s, replication ([\d.]+) s", r.stdout)
    if o:
        out["index_open_s"] = sum(float(o.group(i)) for i in (1, 2, 3))
    return out


def sha256(path):
    h = hashlib.sha256()
    with open(path, "rb") as f:
        for b in iter(lambda: f.read(1 << 24), b""):
            h.update(b)
    return h.hexdigest()


def select_csv(src, dst, chrom, lo, hi, k=20, plen=3):
    """rows of a generated (NGG, PAM at the end) guides CSV whose k-mer lies in [lo, hi) of chrom"""
    with open(src) as f, open(dst, "w") as o:
        o.write(f.readline())
        for line in f:
            _, _, _, c, pos, sense = line.rstrip("\n").split(",")
            a = int(pos) - 1 + (0 if sense == "+" else plen)
            if c == chrom and lo <= a and a + k <= hi:
                o.write(line)


def gpu_identity():
    r = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"], capture_output=True, text=True)
    return r.stdout.strip().splitlines()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=0, help="0: every visible device")
    ap.add_argument("--genome-mb", type=float, default=3100)
    ap.add_argument("--check-mb", type=float, default=8)
    ap.add_argument("--file-batch", type=int, default=50000, help="guides per device and batch (GSX_FILE_BATCH), as tools/config5_run.py")
    ap.add_argument("--whole-genome", action="store_true")
    ap.add_argument("--workdir", default="/tmp/gsx_genome_enum")
    ap.add_argument("--out", required=True, help="JSON result file, e.g. profiles/<tag>_genome_enumerate.json")
    a = ap.parse_args()
    import bench
    import gsx
    import synth
    n_gpus = a.gpus or gsx.device_count()
    os.makedirs(a.workdir, exist_ok=True)
    os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)

    def save():                                                             # after every part: a cut-short run keeps what it measured
        json.dump(res, open(a.out, "w"), indent=1)
    res = {"gpu": gpu_identity(), "n_gpus": n_gpus, "genome_mb": a.genome_mb, "host_cores": os.cpu_count(), "file_batch_per_device": a.file_batch}
    log("gpu:", res["gpu"])
    b = bench.parse_args([])
    b.genome_mb = a.genome_mb
    b.n_chr = 24 if a.genome_mb >= 1000 else 8
    g, chroms, _, _ = bench.make_workload(b, 1)
    prefix = os.path.join(a.workdir, "genome")
    t0 = time.time()
    ix = gsx.Index.build_from_text(g, chroms, sa_shift=2, devices=[0], save_prefix=prefix)
    ix.close()
    res["index_build_s"] = time.time() - t0
    fa = os.path.join(a.workdir, "genome.fa")
    t0 = time.time()
    synth.write_fasta(fa, g, chroms)
    c1, l1 = chroms[0][0], int(chroms[0][1])
    fa1 = os.path.join(a.workdir, "chr1.fa")
    synth.write_fasta(fa1, g[:l1], [(c1, l1)])
    res["fasta_write_s"] = time.time() - t0
    log("index + FASTA:", res["index_build_s"], res["fasta_write_s"])
    env = {"GSX_FILE_BATCH": str(a.file_batch)} if a.file_batch else {}
    cfg4 = ["-m", "4", "-a", "NAG", "--format", "sam", "--mode", "complete", "--gpus", str(n_gpus)]

    # ---- equality at size: the first check_mb of chr1 ----
    hi = int(min(a.check_mb * 1e6, l1))
    bed = os.path.join(a.workdir, "head.bed")
    open(bed, "w").write("%s\t0\t%d\n" % (c1, hi))
    fa_head = os.path.join(a.workdir, "chr1_head.fa")                        # (k-mers inside [0, hi) need at most a PAM beyond it)
    synth.write_fasta(fa_head, g[:hi + 64], [(c1, hi + 64)])
    kall, ksel = os.path.join(a.workdir, "head_all.csv"), os.path.join(a.workdir, "head.csv")
    subprocess.check_call([EXE, "kmers", fa_head, "-o", kall], stdout=subprocess.DEVNULL)
    select_csv(kall, ksel, c1, 0, hi)
    eq = {"region": [c1, 0, hi]}
    for name, args in (("csv_path", ["-f", ksel]), ("fused", ["--genome", fa, "--regions", bed])):
        out = os.path.join(a.workdir, name + ".sam")
        eq[name] = run_cli(["enumerate", prefix] + cfg4 + args + ["-o", out], env)
        eq[name]["bytes"] = os.path.getsize(out)
        eq[name]["sha256"] = sha256(out)
        os.remove(out)
        log("equality", name, eq[name])
    eq["identical"] = eq["csv_path"]["sha256"] == eq["fused"]["sha256"] and eq["csv_path"]["guides"] == eq["fused"]["guides"]
    res["equality"] = eq
    save()

    # ---- rate: chromosome 1 whole, to /dev/null ----
    kcsv = os.path.join(a.workdir, "chr1.csv")
    ka = run_cli(["kmers", fa1, "-o", kcsv], {})
    ka["csv_bytes"] = os.path.getsize(kcsv)
    ea = run_cli(["enumerate", prefix] + cfg4 + ["-f", kcsv, "-o", "/dev/null"], env)
    os.remove(kcsv)
    res["chr1_two_step"] = {"kmers": ka, "enumerate": ea, "wall_s": ka["wall_s"] + ea["wall_s"],
                            "guides_per_s": ea["guides"] / (ka["wall_s"] + ea["wall_s"]), "peak_rss_gb": max(ka["peak_rss_gb"], ea["peak_rss_gb"])}
    log("chr1 two-step:", res["chr1_two_step"])
    bed1 = os.path.join(a.workdir, "chr1.bed")
    open(bed1, "w").write("%s\t0\t%d\n" % (c1, l1))
    eb = run_cli(["enumerate", prefix] + cfg4 + ["--genome", fa, "--regions", bed1, "-o", "/dev/null"], env)
    res["chr1_fused"] = {**eb, "guides_per_s": eb["guides"] / eb["wall_s"]}
    res["chr1_same_guides"] = eb["guides"] == ea["guides"]
    log("chr1 fused:", res["chr1_fused"])
    save()

    if a.whole_genome:
        ew = run_cli(["enumerate", prefix] + cfg4 + ["--genome", fa, "-o", "/dev/null"], env)
        res["whole_genome_fused"] = {**ew, "guides_per_s": ew["guides"] / ew["wall_s"]}
        log("whole genome:", res["whole_genome_fused"])
    else:
        res["whole_genome_fused"] = "not measured"
    save()
    print(json.dumps(res))


if __name__ == "__main__":
    main()
