"""Local traceback of the BASELINE config-5 pair (1 Mbp x 1 Mbp) on one GPU, with compact code storage: a score-only pass
finds the start cell, then codes are kept only for the band around the slope-1 line that ends there (DESIGN.md section 2).

Reports, in one run, with the GPU's name and power limit:
  full      end-to-end gx_align_pair ms; start-cell pass, traceback fill and walk ms of a local traceback plan; code and
            device bytes, repeats (stat 24)
  score     the score-only start-cell plan (GX_FLAG_START_CELL) of the same pair, for comparison
  prefix    compact (GX_CODE_COMPACT=1) against dense code storage at the 262144 x 262144 prefix, alternated
  partial   a 1 Mbp pair homologous only in its middle half: rounds, final half-width and code bytes, or the
            GX_ERR_NOMEM it returns (reported, not checked: its run-on tail crosses 250 kb of unrelated sequence)
Results of the first three are checked against the diagonal construction (tests/test_long_local_traceback.py).  Writes one
JSON file (--out).

    python tools/long_local_traceback.py [--reps 3] [--out profiles/long_local_traceback.json]
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
from test_long_local_traceback import _local_diagonal  # noqa: E402

SCORES = (1, -2, -1, -5)   # config.toml
FULL, PREFIX = 1_000_000, 262144


def gpu_info():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True, timeout=60)
    name, power, clk = [x.strip() for x in q.stdout.splitlines()[0].split(",")]
    return {"name": name, "power_limit": power, "max_sm_clock": clk}


def plan_run(a, b, traceback):
    blob, off1, len1, off2, len2 = gx.pack_pairs([(a, b)])
    plan = gx.Plan(len1, len2, SCORES, True, traceback=traceback, start_cell=not traceback)
    plan.upload(blob, off1, off2)
    plan.execute()
    res, ops, _ = plan.fetch()
    if traceback:
        ops = ops[:int(res["n_ops"][0])].copy()
    st = {"fill_ms": plan.fill_ms, "start_pass_ms": plan.stat(29), "walk_ms": plan.walk_ms, "code_bytes": plan.stat(4),
          "device_bytes": plan.stat(5), "code_storage": plan.stat(27), "code_halfwidth": plan.stat(28),
          "repeats": plan.stat(24), "K": plan.stat(15), "score": int(res["score"][0]),
          "start": [int(res["start_i"][0]), int(res["start_j"][0])]}
    st["traceback_fill_ms"] = st["fill_ms"] - st["start_pass_ms"]
    plan.close()
    return st, res, ops


def check(res, ops, d):
    ok = int(res["score"][0]) == d["score"] and np.array_equal(ops, d["ops"])
    ok = ok and (int(res["start_i"][0]), int(res["start_j"][0])) == d["start"]
    ok = ok and (int(res["matches"][0]), int(res["mismatches"][0]), int(res["gap_extensions"][0]), int(res["opening_gaps"][0])) == (
        d["matches"], d["mismatches"], 0, 0)
    return bool(ok and (int(res["end_i"][0]), int(res["end_j"][0])) == (1, 1))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=3)
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "long_local_traceback.json"))
    args = ap.parse_args()
    lib = _lib.ensure_init(0)
    out = {"gpu": gpu_info(), "scores": SCORES, "reps": args.reps}
    a, b = wl.long_pair(FULL)
    d = _local_diagonal(a, b)

    # ---- full pair: end to end through gx_align_pair (the first call creates the plan the later ones reuse)
    ops = np.zeros(2 * FULL + 1, np.uint8)
    e2e = []
    for it in range(args.reps + 1):
        r = _lib.GxResult()
        t0 = time.perf_counter()
        rc = lib.gx_align_pair(a.ctypes.data, FULL, b.ctypes.data, FULL, _scores_struct(SCORES), 1, _lib.GX_FLAG_TRACEBACK,
                               C.byref(r), ops.ctypes.data, ops.size)
        t1 = time.perf_counter()
        assert rc == 0, (rc, lib.gx_last_error().decode())
        assert r.score == d["score"] and (r.start_i, r.start_j) == d["start"] and np.array_equal(ops[:r.n_ops], d["ops"])
        if it:
            e2e.append({"e2e_ms": (t1 - t0) * 1e3, "fill_ms": r.fill_ms, "walk_ms": r.walk_ms})
    full = [plan_run(a, b, True) for _ in range(args.reps)]
    assert all(check(res, o, d) for _, res, o in full)
    out["full"] = {"gx_align_pair": e2e, "plan": [s for s, _, _ in full], "matches_diagonal": True}

    # ---- score-only start-cell plan of the same pair
    out["score_only"] = [plan_run(a, b, False)[0] for _ in range(args.reps)]
    assert all(s["score"] == d["score"] and tuple(s["start"]) == d["start"] for s in out["score_only"])

    # ---- compact (forced) against dense storage at the 262144 x 262144 prefix, alternated
    pa, pb = a[:PREFIX], b[:PREFIX]
    dp = _local_diagonal(pa, pb)
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

    # ---- homologous middle half: unrelated flanks of 250 kb on both sides
    rng = np.random.default_rng(2026)
    lut = np.frombuffer(b"ACGT", np.uint8)
    q = FULL // 4
    pa = np.concatenate([lut[rng.integers(0, 4, size=q)], a[q:3 * q], lut[rng.integers(0, 4, size=q)]])
    pb = np.concatenate([lut[rng.integers(0, 4, size=q)], b[q:3 * q], lut[rng.integers(0, 4, size=q)]])
    blob, off1, len1, off2, len2 = gx.pack_pairs([(pa, pb)])
    plan = gx.Plan(len1, len2, SCORES, True, traceback=True)
    plan.upload(blob, off1, off2)
    t0 = time.perf_counter()
    try:
        plan.execute()
        res, _, _ = plan.fetch()
        part = {"status": 0, "score": int(res["score"][0]), "start": [int(res["start_i"][0]), int(res["start_j"][0])],
                "end": [int(res["end_i"][0]), int(res["end_j"][0])], "n_ops": int(res["n_ops"][0])}
    except _lib.GxError as e:
        part = {"status": e.status, "error": str(e)}
    part.update({"execute_ms": (time.perf_counter() - t0) * 1e3, "rounds": plan.stat(24), "halfwidth": plan.stat(28),
                 "code_bytes": plan.stat(4), "device_bytes": plan.stat(5), "fill_ms": plan.fill_ms,
                 "start_pass_ms": plan.stat(29), "walk_ms": plan.walk_ms})
    plan.close()
    out["partial_homology"] = part

    def med(xs, k):
        return float(np.median([x[k] for x in xs]))
    pc, pd_ = [r for r in rows if r["compact"]], [r for r in rows if not r["compact"]]
    out["summary"] = {
        "full_e2e_ms": med(e2e, "e2e_ms"), "full_fill_ms": med(out["full"]["plan"], "fill_ms"),
        "full_start_pass_ms": med(out["full"]["plan"], "start_pass_ms"),
        "full_traceback_fill_ms": med(out["full"]["plan"], "traceback_fill_ms"),
        "full_walk_ms": med(out["full"]["plan"], "walk_ms"), "full_repeats": out["full"]["plan"][0]["repeats"],
        "full_code_bytes": out["full"]["plan"][0]["code_bytes"], "full_device_bytes": out["full"]["plan"][0]["device_bytes"],
        "score_only_fill_ms": med(out["score_only"], "fill_ms"),
        "prefix_compact_fill_ms": med(pc, "fill_ms"), "prefix_dense_fill_ms": med(pd_, "fill_ms"),
        "prefix_compact_start_pass_ms": med(pc, "start_pass_ms"),
        "prefix_compact_walk_ms": med(pc, "walk_ms"), "prefix_dense_walk_ms": med(pd_, "walk_ms"),
        "prefix_compact_code_bytes": pc[0]["code_bytes"], "prefix_dense_code_bytes": pd_[0]["code_bytes"],
        "partial_status": part["status"], "partial_rounds": part["rounds"], "partial_halfwidth": part["halfwidth"],
        "partial_code_bytes": part["code_bytes"],
    }
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "w") as f:
        json.dump(out, f, indent=1)
    print(json.dumps({"gpu": out["gpu"], **out["summary"]}))


if __name__ == "__main__":
    main()
