#!/usr/bin/env python
"""Fill / walk time of every K (columns per lane) and recurrence form on the wavefront workloads, in ONE process
(GX_K / GX_CHAIN1 are read per plan).  Results: one JSON line per run in the --out file.

    python tools/sweep_kr.py [--workloads brca2_global,brca2_local,corona45,corona6,nw200k,nw1m] [--k 4,8,16] [--steps 5]
"""
import argparse
import json
import os
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))

import genomics_rs_b200 as gx  # noqa: E402
from genomics_rs_b200 import _lib, workloads as wl  # noqa: E402

SCORES = wl.CONFIG_TOML
ALL = [4, 8, 16]


def workload(name):
    """-> (pairs as (blob, off1, len1, off2, len2), is_local, traceback)"""
    if name.startswith("corona"):
        seqs, jobs = wl.corona_pairs()
        shard = {"corona6": 8, "corona11": 4, "corona23": 2}.get(name)
        if shard:                 # rank 0's shard of the 8 / 4 / 2-GPU run
            costs = [(len(seqs[a]) + 1) * (len(seqs[b]) + 1) for a, b in jobs]
            jobs = [jobs[k] for k in wl.lpt_shards(costs, shard)[0]]
        elif name == "corona1":
            jobs = jobs[:1]
        return gx.pack_pairs([(seqs[a], seqs[b]) for a, b in jobs]), False, True
    if name in ("brca2_global", "brca2_local"):
        a, b = wl.brca2_pair()
        return gx.pack_pairs([(a, b)]), name.endswith("local"), True
    if name.startswith("nw"):
        n = {"nw200k": 200_000, "nw1m": 1_000_000, "nw50k": 50_000}[name]
        a, b = wl.long_pair(n)
        return gx.pack_pairs([(a, b)]), False, False
    raise SystemExit(name)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--workloads", default="brca2_global,brca2_local,corona6,corona45,nw200k")
    ap.add_argument("--k", default="", help="comma list of K values to force (default: 4,8,16)")
    ap.add_argument("--chain", default="0,1")
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--auto-only", action="store_true", help="only the configuration the library picks itself")
    ap.add_argument("--out", default=os.path.join(ROOT, "gpurun_out", "sweep_kr.jsonl"))
    args = ap.parse_args()
    if not os.path.dirname(args.out):   # a bare file name goes next to the default output file
        args.out = os.path.join(os.path.dirname(ap.get_default("out")), args.out)
    ks = [int(k) for k in args.k.split(",") if k] or ALL
    chains = [int(c) for c in args.chain.split(",")]
    _lib.ensure_init(0)
    os.makedirs(os.path.dirname(args.out), exist_ok=True)
    fh = open(args.out, "a")
    for name in args.workloads.split(","):
        (blob, off1, len1, off2, len2), is_local, tb = workload(name)
        cells = int(((len1 + 1) * (len2 + 1)).sum())
        ref = None
        for k in [0] + ([] if args.auto_only else ks):
            for c in ([-1] if k == 0 else chains):
                for var in ("GX_K", "GX_CHAIN1"):
                    os.environ.pop(var, None)
                if k:
                    os.environ["GX_K"], os.environ["GX_CHAIN1"] = str(k), str(c)
                try:
                    plan = gx.Plan(len1, len2, SCORES, is_local, traceback=tb)
                    plan.upload(blob, off1, off2)
                    for _ in range(2):
                        plan.execute()
                    fills, walks = [], []
                    t0 = time.perf_counter()
                    for _ in range(args.steps):
                        plan.execute()
                        fills.append(plan.fill_ms)
                        walks.append(plan.walk_ms)
                    wall = (time.perf_counter() - t0) / args.steps * 1e3
                    scores = plan.fetch_scores().tolist() if not tb else plan.fetch()[0]["score"].tolist()
                    rec = dict(workload=name, K=int(plan.stat(15)), chain1=int(plan.stat(17)), forced=bool(k),
                               batch=int(plan.stat(22)), resident=int(plan.stat(21)),
                               fill_ms=float(np.median(fills)), fill_min=float(min(fills)), walk_ms=float(np.median(walks)), wall_ms=wall,
                               gcups_fill=cells / (np.median(fills) * 1e-3) / 1e9, cells=cells)
                    if ref is None:
                        ref = scores
                    rec["scores_agree"] = scores == ref
                    plan.close()
                except Exception as e:   # keep sweeping: one broken tile shape must not hide the others
                    rec = dict(workload=name, K=k, chain1=c, error=str(e)[:300])
                print(json.dumps(rec), flush=True)
                fh.write(json.dumps(rec) + "\n")
                fh.flush()


if __name__ == "__main__":
    main()
