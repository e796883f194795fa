#!/usr/bin/env python
"""Start cells from the short-read kernels on BASELINE config 4 (10 M x 150 bp, local, CONFIG_TOML): one JSON line.

  kernels   fill_ms of three resident 10 M-pair plans, warmed up, then alternated over --repeats rounds:
            score only (s16x2), start cells (s16x2), start cells with GX_READS32=1 (32-bit kernel)
  e2e       gx_score_batch against gx_score_batch_cells on the same pairs from pinned host memory, alternated
  wavefront the first 2^18 pairs through the wavefront start-cell path (plans of 1023 pairs: fill + walk ms summed)
            against one read plan with start cells (fill ms)
  checks    every score of the start-cell calls equals the score-only call; a seeded 2^16-pair sample of start cells
            equals the oracle (score_linear)

TCUPS count (m+1)(n+1) = 151 x 151 cells per pair, as bench.py does.  Needs a B200; there is no CPU fallback.

    python tools/reads_start_cells.py [--pairs N] [--repeats R] [--out FILE]
"""
import argparse
import ctypes as C
import json
import os
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.dont_write_bytecode = True

import genomics_rs_b200 as gx  # noqa: E402
from genomics_rs_b200 import _lib, workloads as wl  # noqa: E402
from oracle import gxo  # noqa: E402

SCORES = wl.CONFIG_TOML


def device_info():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True, timeout=60)
    name, power, clock = [x.strip() for x in q.stdout.splitlines()[0].split(",")]
    return {"name": name, "power_limit": power, "max_sm_clock": clock}


def pinned(arr):
    import torch
    t = torch.empty(arr.size, dtype=torch.uint8, pin_memory=True)
    v = t.numpy()
    v[:] = arr.view(np.uint8).reshape(-1)
    return t, v


def make_plan(packed, start_cell, reads32):
    if reads32:
        os.environ["GX_READS32"] = "1"       # read once, when the plan is created
    else:
        os.environ.pop("GX_READS32", None)
    blob, off1, len1, off2, len2 = packed
    plan = gx.Plan(len1, len2, SCORES, True, traceback=False, start_cell=start_cell)
    plan.upload(blob, off1, off2)
    os.environ.pop("GX_READS32", None)
    return plan


def compact(packed, lo, hi):
    """pairs lo..hi-1 with only their own bytes: a plan uploads the whole blob it is given"""
    blob, off1, len1, off2, len2 = packed
    o1, l1, o2, l2 = off1[lo:hi], len1[lo:hi], off2[lo:hi], len2[lo:hi]
    b0 = int(min(o1.min(), o2.min()))
    b1 = int(max((o1 + l1).max(), (o2 + l2).max()))
    return blob[b0:b1], o1 - np.uint64(b0), l1, o2 - np.uint64(b0), l2


def stats(xs):
    xs = np.asarray(xs, np.float64)
    return {"median": float(np.median(xs)), "min": float(xs.min()), "max": float(xs.max()), "n": int(xs.size)}


def oracle_sample(packed, idx):
    lib = gxo.lib()
    blob, off1, len1, off2, len2 = packed
    base = blob.ctypes.data
    out = np.zeros((idx.size, 3), np.int64)
    v, i, j = C.c_int64(), C.c_uint64(), C.c_uint64()
    for r, q in enumerate(idx):
        rc = lib.gxo_score_linear(base + int(off1[q]), int(len1[q]), base + int(off2[q]), int(len2[q]), *SCORES, 1,
                                  C.byref(v), C.byref(i), C.byref(j))
        assert rc == 0
        out[r] = (v.value, i.value, j.value)
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--pairs", type=int, default=10_000_000)
    ap.add_argument("--repeats", type=int, default=7)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    _lib.ensure_init(0)
    dev = device_info()
    n = args.pairs
    t0 = time.perf_counter()
    blob, off1, len1, off2, len2 = wl.reads150(0, n)
    pin_t, pblob = pinned(blob)
    del blob
    packed = (pblob, off1, len1, off2, len2)
    gen_s = time.perf_counter() - t0
    cells = n * 151 * 151
    out = {"tool": "reads_start_cells", "device": dev, "pairs": n, "cells": cells, "scores": list(SCORES),
           "repeats": args.repeats, "input_gen_s": round(gen_s, 1)}

    # ---- kernels only: three resident plans, alternated
    variants = {"score_s16": (False, False), "cells_s16": (True, False), "cells_32": (True, True)}
    plans = {k: make_plan(packed, *v) for k, v in variants.items()}
    for p in plans.values():
        for _ in range(3):
            p.execute()
    ms = {k: [] for k in plans}
    for _ in range(args.repeats):
        for k, p in plans.items():
            p.execute()
            ms[k].append(p.fill_ms)
    out["kernels"] = {k: {"fill_ms": stats(ms[k]), "lane_bits": int(plans[k].stat(26)), "family": int(plans[k].stat(9)),
                          "tcups": round(cells / (np.median(ms[k]) * 1e-3) / 1e12, 3)} for k in plans}
    scores_plan = plans["score_s16"].fetch_scores()
    res16, _, _ = plans["cells_s16"].fetch()
    res32, _, _ = plans["cells_32"].fetch()
    for p in plans.values():
        p.close()
    del plans

    # ---- end to end from pinned host buffers
    sc_only = np.zeros(n, np.int64)
    sc_cells = np.zeros(n, np.int64)
    si, sj = np.zeros(n, np.uint64), np.zeros(n, np.uint64)
    lib = _lib.load()
    gs = _lib.GxScores(*SCORES)

    def call_scores():
        _lib.check(lib.gx_score_batch(pblob.ctypes.data, pblob.size, off1.ctypes.data, len1.ctypes.data, off2.ctypes.data,
                                      len2.ctypes.data, n, gs, 1, sc_only.ctypes.data))

    def call_cells():
        _lib.check(lib.gx_score_batch_cells(pblob.ctypes.data, pblob.size, off1.ctypes.data, len1.ctypes.data,
                                            off2.ctypes.data, len2.ctypes.data, n, gs, 1, sc_cells.ctypes.data,
                                            si.ctypes.data, sj.ctypes.data))
    calls = {"gx_score_batch": call_scores, "gx_score_batch_cells": call_cells}
    for f in calls.values():
        f()
    e2e = {k: [] for k in calls}
    for _ in range(max(3, args.repeats // 2)):
        for k, f in calls.items():
            t = time.perf_counter()
            f()
            e2e[k].append((time.perf_counter() - t) * 1e3)
    out["e2e"] = {k: {"ms": stats(v), "tcups": round(cells / (np.median(v) * 1e-3) / 1e12, 3)} for k, v in e2e.items()}

    # ---- the first 2^18 pairs: wavefront start-cell plans of 1023 pairs against one read plan
    m18 = min(n, 1 << 18)
    rp = make_plan(compact(packed, 0, m18), True, False)
    rp.execute()
    read_ms = []
    for _ in range(args.repeats):
        rp.execute()
        read_ms.append(rp.fill_ms)
    read_res, _, _ = rp.fetch()
    read_family = int(rp.stat(9))
    rp.close()
    wave_plans = []
    for lo in range(0, m18, 1023):
        wave_plans.append(make_plan(compact(packed, lo, min(m18, lo + 1023)), True, False))
    for p in wave_plans:
        p.execute()
    wave_ms = []
    for _ in range(max(2, args.repeats // 3)):
        tot = 0.0
        for p in wave_plans:
            p.execute()
            tot += p.fill_ms + p.walk_ms
        wave_ms.append(tot)
    wave_res = np.concatenate([p.fetch()[0] for p in wave_plans])
    wave_family = {int(p.stat(9)) for p in wave_plans}
    for p in wave_plans:
        p.close()
    c18 = m18 * 151 * 151
    out["first_2e18"] = {
        "pairs": m18,
        "read_plan": {"family": read_family, "ms": stats(read_ms), "tcups": round(c18 / (np.median(read_ms) * 1e-3) / 1e12, 3)},
        "wavefront_plans": {"family": sorted(wave_family), "plans": len(wave_plans), "ms": stats(wave_ms),
                            "tcups": round(c18 / (np.median(wave_ms) * 1e-3) / 1e12, 3)},
        "speedup": round(float(np.median(wave_ms) / np.median(read_ms)), 2),
        "same_results": bool(all(np.array_equal(read_res[f], wave_res[f]) for f in ("score", "start_i", "start_j", "end_i", "end_j"))),
    }

    # ---- output checks
    idx = np.sort(np.random.default_rng(2026).choice(n, min(n, 1 << 16), replace=False))
    ora = oracle_sample(packed, idx)
    out["checks"] = {
        "scores_cells_e2e_equal_score_only": bool(np.array_equal(sc_cells, sc_only)),
        "scores_plans_equal_score_only": bool(np.array_equal(res16["score"], scores_plan) and np.array_equal(res32["score"], scores_plan)
                                              and np.array_equal(sc_only, scores_plan)),
        "cells_s16_equal_cells_32": bool(np.array_equal(res16["start_i"], res32["start_i"]) and
                                         np.array_equal(res16["start_j"], res32["start_j"])),
        "cells_e2e_equal_plan": bool(np.array_equal(si, res16["start_i"]) and np.array_equal(sj, res16["start_j"])),
        "sample_pairs": int(idx.size),
        "sample_equals_oracle": bool(np.array_equal(ora[:, 0], sc_cells[idx]) and np.array_equal(ora[:, 1], si[idx].astype(np.int64))
                                     and np.array_equal(ora[:, 2], sj[idx].astype(np.int64))),
    }
    line = json.dumps(out)
    print(line)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            f.write(line + "\n")


if __name__ == "__main__":
    main()
