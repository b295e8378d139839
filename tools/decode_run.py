#!/usr/bin/env python
"""`guidescan decode` at genome scale: on the synthetic genome of bench.py (3.1 Gb by default), a configs[4]-shaped database --
200 k guides, m = 4, NGG + NAG, SAM complete -- written by `guidescan enumerate`, then decoded back into CSV complete.  For
comparison the same guides through `enumerate --format csv --mode complete` (the same rows, from the search), and a diff of the
two texts on a sample of guides.  One JSON line per run is appended to --out (profiles/ by default).

  python tools/decode_run.py --out profiles/r04a_decode_3100mb_200k.jsonl
"""
import argparse
import json
import os
import random
import re
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "guidescan-cli_b200"))
EXE = os.path.join(ROOT, "guidescan-cli_b200", "bin", "guidescan")


def log(*a):
    print(*a, file=sys.stderr, flush=True)


def run(args, env=None):
    t0 = time.time()
    r = subprocess.run([EXE] + args, capture_output=True, text=True, env={**os.environ, "GSX_FILE_TIMING": "1", **(env or {})})
    dt = time.time() - t0
    if r.returncode:
        raise RuntimeError("guidescan %s failed: %s" % (" ".join(args), r.stderr[-800:]))
    return dt, r.stdout, r.stderr


def gpu_identity():
    r = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"], capture_output=True, text=True)
    return r.stdout.strip().splitlines()


def rows_by_guide(path, ids):
    out = {}
    with open(path) as f:
        next(f)
        for line in f:
            gid = line.split(",", 1)[0]
            if gid in ids:
                out.setdefault(gid, []).append(line)
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--genome-mb", type=float, default=3100)
    ap.add_argument("--guides", type=int, default=200000)
    ap.add_argument("--sample", type=int, default=2000, help="guides whose decoded rows are diffed against enumerate's CSV")
    ap.add_argument("--workdir", default="/tmp/gsx_decode_run")
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "decode_run.jsonl"))
    a = ap.parse_args()
    import bench
    import gsx
    import synth
    os.makedirs(a.workdir, exist_ok=True)
    os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
    res = {"gpu": gpu_identity(), "genome_mb": a.genome_mb, "guides": a.guides, "host_cores": os.cpu_count(),
           "options": "-m 4 -a NAG (configs[4])"}
    log("gpu:", res["gpu"])
    b = bench.parse_args([])
    b.genome_mb, b.guides_per_step, b.steps, b.warmup = a.genome_mb, a.guides, 1, 0
    b.n_chr = 24 if a.genome_mb >= 1000 else 8
    g, chroms, pos, kmers = bench.make_workload(b, 1)
    prefix, fa, guides = (os.path.join(a.workdir, x) for x in ("genome", "genome.fa", "guides.csv"))
    t0 = time.time()
    ix = gsx.Index.build_from_text(g, chroms, sa_shift=2, devices=[0], save_prefix=prefix)
    ix.close()
    synth.write_fasta(fa, g, chroms)
    synth.write_guides_csv(guides, pos[:a.guides], kmers[:a.guides], chroms)
    res["setup_s"] = time.time() - t0
    del g
    cfg4 = ["-m", "4", "-a", "NAG", "--mode", "complete"]
    sam, dec, csv = (os.path.join(a.workdir, x) for x in ("db.sam", "decoded.csv", "enumerate.csv"))
    dt, _, err = run(["enumerate", prefix, "-f", guides, "--format", "sam", "-o", sam] + cfg4)
    res["enumerate_sam"] = {"wall_s": dt, "bytes": os.path.getsize(sam), "timing": [l for l in err.splitlines() if l.startswith("gsx file job")]}
    log("enumerate sam:", res["enumerate_sam"])
    dt, out, err = run(["decode", sam, "--genome", fa, "-o", dec, "-a", "NAG"])
    line = [l for l in err.splitlines() if l.startswith("gsx decode:")][-1]
    m = re.search(r"(\d+) SAM bytes, (\d+) guides decoded, (\d+) rows, (\d+) batch.*FASTA read ([\d.]+) s .*genome upload ([\d.]+) s; read/split ([\d.]+) s; "
                  r"device ([\d.]+) s \(events ([\d.]+) ms, ([\d.]+) ms per batch\); format ([\d.]+) s; write ([\d.]+) s", line)
    sam_bytes, guides_dec, rows, batches = (int(m.group(i)) for i in range(1, 5))
    res["decode"] = {"wall_s": dt, "timing": line, "sam_bytes": sam_bytes, "guides_decoded": guides_dec, "rows": rows, "batches": batches,
                     "fasta_read_s": float(m.group(5)), "genome_upload_s": float(m.group(6)), "read_split_s": float(m.group(7)),
                     "device_s": float(m.group(8)), "device_event_ms": float(m.group(9)), "device_ms_per_batch": float(m.group(10)),
                     "format_s": float(m.group(11)), "write_s": float(m.group(12)), "out_bytes": os.path.getsize(dec),
                     "sam_bytes_per_s": sam_bytes / dt, "rows_per_s": rows / dt}
    job = float(re.search(r"gsx decode: ([\d.]+) s wall", line).group(1))
    res["decode"]["job_wall_s"] = job                                        # after the FASTA read, genome upload included
    res["decode"]["rows_per_s_after_upload"] = rows / (job - res["decode"]["genome_upload_s"])
    log("decode:", res["decode"])
    dt, _, err = run(["enumerate", prefix, "-f", guides, "--format", "csv", "-o", csv] + cfg4)
    res["enumerate_csv"] = {"wall_s": dt, "bytes": os.path.getsize(csv), "timing": [l for l in err.splitlines() if l.startswith("gsx file job")]}
    log("enumerate csv:", res["enumerate_csv"])
    # the sample: decoded rows against enumerate's CSV rows (the CSV rule's specificity differs from the SAM rule's: compared without it)
    ids = set(random.Random(7).sample(sorted({l.split("\t", 1)[0] for l in open(sam) if not l.startswith("@")}), a.sample))
    got, want = rows_by_guide(dec, ids), rows_by_guide(csv, ids)
    strip = lambda v: [l.rsplit(",", 1)[0] for l in v]
    diff = [k for k in ids if strip(got.get(k, [])) != strip(want.get(k, []))]
    res["sample"] = {"guides": len(ids), "rows": sum(len(v) for v in got.values()), "guides_differing_without_specificity": len(diff)}
    log("sample:", res["sample"])
    for p in (sam, dec, csv):
        os.remove(p)
    with open(a.out, "a") as f:
        f.write(json.dumps(res) + "\n")
    print(json.dumps(res))


if __name__ == "__main__":
    main()
