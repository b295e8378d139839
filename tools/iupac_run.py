#!/usr/bin/env python
"""IUPAC class PAMs against their concrete expansions on the bench workload (3.1 Gb, 200 k 20-mers per step, m = 3): one genome and
index build, then, alternated over the same steps `--rounds` times, column NRG against NAG + NGG and NNGRRT against its 4-PAM
expansion.  Per run: device and end-to-end guides/s, ms_sweep, seeds, matches and summary sectors per guide; per step: whether
every result array of the class form equals the expansion's, field by field.  One JSON line per run to <out>/<tag>.jsonl, the
first one with the card's name and power limit.

  python tools/iupac_run.py --tag iupac_run [--out profiles] [--genome-mb 3100] [--rounds 2] [--steps 3]
"""
import argparse
import json
import os
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, os.path.join(ROOT, "tools"))

PAIRS = {"NRG": ("NRG", ["NAG", "NGG"]), "NNGRRT": ("NNGRRT", ["NNGAAT", "NNGAGT", "NNGGAT", "NNGGGT"])}


def arrays(r):
    out = dict(r.guide_arrays())
    out.update(r.hit_arrays())
    return {k: np.array(v, copy=True) for k, v in out.items()}


def guide_arrays(gsx, kmers, per, steps, pam):
    arrs = []
    for i in range(steps):
        arr = (gsx.Guide * per)()
        for j in range(per):
            arr[j] = gsx.Guide(kmers[i * per + j, :20].tobytes(), pam.encode())
        arrs.append(arr)
    return arrs


def run(ix, arrs, per, params):
    ix.enumerate_raw(arrs[0], per, params).close()                 # warm-up of this configuration
    ctrs, outs, walls = [], [], []
    for a in arrs:
        t0 = time.perf_counter()
        r = ix.enumerate_raw(a, per, params)
        walls.append(time.perf_counter() - t0)
        ctrs.append(r.counters()); outs.append(arrays(r)); r.close()
    return ctrs, outs, walls


def summary(name, ctrs, walls, per):
    n = len(ctrs)
    d = {"name": name, "steps": n, "guides_per_step": per}
    d["ms_sweep"] = [c["ms_sweep"] for c in ctrs]
    d["ms_total_device"] = [c["ms_total_device"] for c in ctrs]
    d["guides_per_s_device"] = per * n / (sum(d["ms_total_device"]) * 1e-3)
    d["guides_per_s_e2e"] = per * n / sum(walls)
    for k in ("seeds", "matches", "sectors"):
        d[k + "_per_guide"] = sum(c[k] for c in ctrs) / (per * n)
    d["launches"] = ctrs[0]["launches"]
    return d


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--tag", required=True)
    ap.add_argument("--genome-mb", type=float, default=3100)
    ap.add_argument("--seed", type=int, default=3)
    ap.add_argument("--guides", type=int, default=200000)
    ap.add_argument("--steps", type=int, default=3)
    ap.add_argument("--rounds", type=int, default=2)
    ap.add_argument("--workdir", default="/tmp/gsx_iupac_run")
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles"), help="directory of the JSON lines file")
    args = ap.parse_args()
    import gpu_session
    import gsx
    os.makedirs(args.workdir, exist_ok=True)
    os.makedirs(args.out, exist_ok=True)
    path = os.path.join(args.out, args.tag + ".jsonl")
    card = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                          capture_output=True, text=True).stdout.strip().splitlines()
    s = gpu_session.Session(args, {"devices": [0]})
    per = args.guides
    with open(path, "a") as f:
        def emit(d):
            f.write(json.dumps(d) + "\n"); f.flush()
            print(json.dumps(d)[:700], flush=True)
        emit({"name": "_index", "card": card[0] if card else None, "index_wall_s": s.index_s, "genome_mb": args.genome_mb,
              "mismatches": 3})
        for rnd in range(args.rounds):
            for name, (cls, concrete) in PAIRS.items():
                a_cls = guide_arrays(gsx, s.kmers, per, args.steps, cls)
                a_con = guide_arrays(gsx, s.kmers, per, args.steps, concrete[0])
                c0, o0, w0 = run(s.ix, a_cls, per, gsx.make_params(mismatches=3, iupac_pams=True))
                c1, o1, w1 = run(s.ix, a_con, per, gsx.make_params(mismatches=3, alt_pams=concrete[1:]))
                eq = [all(a[k].shape == b[k].shape and np.array_equal(a[k], b[k]) for k in a) for a, b in zip(o0, o1)]
                emit(dict(summary(name + "_class", c0, w0, per), round=rnd, pams=[cls]))
                emit(dict(summary(name + "_expansion", c1, w1, per), round=rnd, pams=concrete, equal_per_step=eq, all_equal=all(eq)))
    s.close()


if __name__ == "__main__":
    main()
