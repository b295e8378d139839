#!/usr/bin/env python
"""A/B of the two-part sweep (sweep_split_kernel) against the plain one on the bench workload (3.1 Gb, 200 k NGG 20-mers per
step, m = 3): one genome and index build, then GSX_SPLIT=0 / 1 alternated over the same steps, `--rounds` times each.  Per run:
device ms per stage, summary sectors and seeds per guide; per step: whether every result array of the two paths is equal, field
by field.  Then the two-part path at other slice widths / CTAs per SM (`--variants`).  One JSON line per run to <out>/<tag>.jsonl.

  python tools/split_ab.py --tag split_ab [--out profiles] [--genome-mb 3100] [--rounds 3] [--steps 3] [--variants sb4,sb3,c5]
"""
import argparse
import json
import os
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, os.path.join(ROOT, "tools"))

STAGES = ("ms_sweep", "ms_search", "ms_arrange", "ms_locate", "ms_score", "ms_total_device")


def arrays(r):
    out = dict(r.guide_arrays())
    out.update(r.hit_arrays())
    return {k: np.array(v, copy=True) for k, v in out.items()}


def run(s, arrs, per, params, env):
    for k, v in env.items():
        os.environ[k] = str(v)
    try:
        s.ix.enumerate_raw(arrs[0][0], per, params).close()          # warm-up of this configuration
        ctrs, outs = [], []
        for a in arrs:
            r = s.ix.enumerate_raw(a[0], per, params)
            ctrs.append(r.counters()); outs.append(arrays(r)); r.close()
    finally:
        for k in env:
            os.environ.pop(k, None)
    return ctrs, outs


def summary(name, env, ctrs, per):
    n = len(ctrs)
    d = {"name": name, "env": env, "steps": n, "guides_per_step": per}
    for k in STAGES:
        d[k] = [c[k] for c in ctrs]
    d["guides_per_s_device"] = per * n / (sum(d["ms_total_device"]) * 1e-3)
    d["sectors_per_guide"] = sum(c["sectors"] for c in ctrs) / (per * n)
    d["seeds_per_guide"] = sum(c["seeds"] for c in ctrs) / (per * n)
    d["matches_per_guide"] = sum(c["matches"] for c in ctrs) / (per * n)
    d["launches"] = ctrs[0]["launches"]
    return d


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--tag", required=True)
    ap.add_argument("--genome-mb", type=float, default=3100)
    ap.add_argument("--seed", type=int, default=3)
    ap.add_argument("--guides", type=int, default=200000)
    ap.add_argument("--steps", type=int, default=3)
    ap.add_argument("--rounds", type=int, default=3)
    ap.add_argument("--variants", default="")
    ap.add_argument("--workdir", default="/tmp/gsx_split_ab")
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles"), help="directory of the JSON lines file")
    args = ap.parse_args()
    import gpu_session
    import gsx
    os.makedirs(args.workdir, exist_ok=True)
    os.makedirs(args.out, exist_ok=True)
    path = os.path.join(args.out, args.tag + ".jsonl")
    s = gpu_session.Session(args, {"devices": [0]})
    per, params = args.guides, gsx.make_params(mismatches=3)
    arrs = [s.guide_array(i * per, per) for i in range(args.steps)]
    with open(path, "a") as f:
        def emit(d):
            f.write(json.dumps(d) + "\n"); f.flush()
            print(json.dumps({k: v for k, v in d.items()})[:700], flush=True)
        emit({"name": "_index", "index_wall_s": s.index_s, "genome_mb": args.genome_mb})
        for rnd in range(args.rounds):
            c0, o0 = run(s, arrs, per, params, {"GSX_SPLIT": "0"})
            c1, o1 = run(s, arrs, per, params, {"GSX_SPLIT": "1"})
            eq = []
            for a, b in zip(o0, o1):
                eq.append({k: bool(a[k].shape == b[k].shape and np.array_equal(a[k], b[k])) for k in a})
            emit(dict(summary("plain", {"GSX_SPLIT": "0"}, c0, per), round=rnd))
            emit(dict(summary("split", {"GSX_SPLIT": "1"}, c1, per), round=rnd, equal_per_step=eq,
                      all_equal=all(all(e.values()) for e in eq)))
        for v in [x for x in args.variants.split(",") if x]:
            env = {"GSX_SPLIT": "1"}
            if v.startswith("sb"):
                env["GSX_SPLIT_SB"] = v[2:]
            elif v.startswith("c"):
                env["GSX_SPLIT_CTAS"] = v[1:]
            c1, o1 = run(s, arrs, per, params, env)
            eq = all(all(a[k].shape == b[k].shape and np.array_equal(a[k], b[k]) for k in a) for a, b in zip(o0, o1))
            emit(dict(summary("split_" + v, env, c1, per), all_equal=eq))
    s.close()


if __name__ == "__main__":
    main()
