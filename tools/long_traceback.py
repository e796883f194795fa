"""Global traceback of the BASELINE config-5 pair (1 Mbp x 1 Mbp) on one GPU, with compact code storage (DESIGN.md section 2).

Reports, in one run, with the GPU's name and power limit:
  full      fill / walk ms of a traceback plan, end-to-end gx_align_pair ms, code and device bytes, repeats (stat 24)
  score     the score-only fill of the same pair, for comparison
  prefix    compact (GX_CODE_COMPACT=1) against dense code storage at the 262144 x 262144 prefix, alternated
Every result is checked against the pure diagonal (tests/test_long_traceback.py).  Writes one JSON file (--out).

    python tools/long_traceback.py [--reps 3] [--out profiles/long_traceback.json]
"""
import argparse
import ctypes as C
import json
import os
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))

import numpy as np  # noqa: E402

import genomics_rs_b200 as gx  # noqa: E402
from genomics_rs_b200 import _lib, workloads as wl  # noqa: E402
from genomics_rs_b200.alignment import _scores_struct  # noqa: E402
from test_long_traceback import _diagonal  # noqa: E402

SCORES = (1, -2, -1, -5)   # config.toml
FULL, PREFIX = 1_000_000, 262144


def gpu_info():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True, timeout=60)
    name, power, clk = [x.strip() for x in q.stdout.splitlines()[0].split(",")]
    return {"name": name, "power_limit": power, "max_sm_clock": clk}


def plan_run(a, b, traceback):
    blob, off1, len1, off2, len2 = gx.pack_pairs([(a, b)])
    plan = gx.Plan(len1, len2, SCORES, False, traceback=traceback)
    plan.upload(blob, off1, off2)
    plan.execute()
    if traceback:
        res, ops, _ = plan.fetch()
        ops = ops[:int(res["n_ops"][0])].copy()
    else:
        res, ops = None, None
        plan.fetch_scores()
    st = {"fill_ms": plan.fill_ms, "walk_ms": plan.walk_ms, "code_bytes": plan.stat(4), "device_bytes": plan.stat(5),
          "code_storage": plan.stat(27), "code_halfwidth": plan.stat(28), "repeats": plan.stat(24), "K": plan.stat(15)}
    plan.close()
    return st, res, ops


def check(res, ops, d):
    ok = int(res["score"][0]) == d["score"] and np.array_equal(ops, d["ops"])
    ok = ok and (int(res["matches"][0]), int(res["mismatches"][0]), int(res["gap_extensions"][0]), int(res["opening_gaps"][0])) == (
        d["matches"], d["mismatches"], 0, 0)
    return bool(ok and (int(res["end_i"][0]), int(res["end_j"][0])) == (1, 1))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=3)
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "long_traceback.json"))
    args = ap.parse_args()
    lib = _lib.ensure_init(0)
    out = {"gpu": gpu_info(), "scores": SCORES, "reps": args.reps}
    a, b = wl.long_pair(FULL)
    d = _diagonal(a, b, FULL)

    # ---- full pair: end to end through gx_align_pair (the first call creates the plan the later ones reuse)
    ops = np.zeros(2 * FULL + 1, np.uint8)
    e2e = []
    for it in range(args.reps + 1):
        r = _lib.GxResult()
        t0 = time.perf_counter()
        rc = lib.gx_align_pair(a.ctypes.data, FULL, b.ctypes.data, FULL, _scores_struct(SCORES), 0, _lib.GX_FLAG_TRACEBACK,
                               C.byref(r), ops.ctypes.data, ops.size)
        t1 = time.perf_counter()
        assert rc == 0, (rc, lib.gx_last_error().decode())
        assert r.score == d["score"] and np.array_equal(ops[:r.n_ops], d["ops"])
        if it:
            e2e.append({"e2e_ms": (t1 - t0) * 1e3, "fill_ms": r.fill_ms, "walk_ms": r.walk_ms})
    full = [plan_run(a, b, True) for _ in range(args.reps)]
    assert all(check(res, o, d) for _, res, o in full)
    out["full"] = {"gx_align_pair": e2e, "plan": [s for s, _, _ in full], "matches_diagonal": True}

    # ---- score-only fill of the same pair
    out["score_only"] = [plan_run(a, b, False)[0] for _ in range(args.reps)]

    # ---- compact (forced) against dense storage at the 262144 x 262144 prefix, alternated
    pa, pb = a[:PREFIX], b[:PREFIX]
    dp = _diagonal(a, b, PREFIX)
    rows = []
    for it in range(args.reps + 1):
        for compact in (True, False):
            if compact:
                os.environ["GX_CODE_COMPACT"] = "1"
            else:
                os.environ.pop("GX_CODE_COMPACT", None)
            st, res, o = plan_run(pa, pb, True)
            assert check(res, o, dp), compact
            if it:
                rows.append(dict(st, compact=compact))
    os.environ.pop("GX_CODE_COMPACT", None)
    out["prefix_262144"] = rows

    def med(xs, k):
        return float(np.median([x[k] for x in xs]))
    out["summary"] = {
        "full_fill_ms": med(out["full"]["plan"], "fill_ms"), "full_walk_ms": med(out["full"]["plan"], "walk_ms"),
        "full_e2e_ms": med(e2e, "e2e_ms"), "full_code_bytes": out["full"]["plan"][0]["code_bytes"],
        "full_device_bytes": out["full"]["plan"][0]["device_bytes"], "score_only_fill_ms": med(out["score_only"], "fill_ms"),
        "prefix_compact_fill_ms": med([r for r in rows if r["compact"]], "fill_ms"),
        "prefix_dense_fill_ms": med([r for r in rows if not r["compact"]], "fill_ms"),
        "prefix_compact_walk_ms": med([r for r in rows if r["compact"]], "walk_ms"),
        "prefix_dense_walk_ms": med([r for r in rows if not r["compact"]], "walk_ms"),
        "prefix_compact_code_bytes": rows[0]["code_bytes"], "prefix_dense_code_bytes": rows[1]["code_bytes"],
    }
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "w") as f:
        json.dump(out, f, indent=1)
    print(json.dumps({"gpu": out["gpu"], **out["summary"]}))


if __name__ == "__main__":
    main()
