"""Traceback for short-read sets (gx_align_reads) on the config-4 workload, in one run, with the GPU's name and power limit.

  kernels   the first 2^18 pairs of the config-4 generator (workloads.reads150), local and global, variants alternated,
            medians of --reps: gx_align_reads kernel time (its fill_ms: CUDA events around the read kernel), a wavefront
            traceback Plan on the same pairs (fill + walk), and the start-cell read plan (GX_FLAG_START_CELL; the default
            lane width and the 32-bit kernel), which is what traceback costs on top of the score
  parity    gx_align_reads results and op bytes equal the wavefront plan's on those pairs, both modes
  memory    device bytes in use after gx_align_reads on 2^20 pairs and after 10 M pairs (same process, nothing else ran)
  e2e       --pairs (10 M) x 150 bp local through gx_align_reads against gx_score_batch_cells, from the same pinned
            buffers, alternated; and what gx_align_batch with GX_FLAG_TRACEBACK does on the same pairs (time or status)
  bench     with --parent DIR: `bench.py --gpus 1` all-configs lines of DIR (the parent commit's tree, built) and of this
            tree, alternated

    python tools/read_traceback.py [--reps 5] [--pairs 10000000] [--parent DIR] [--out profiles/read_traceback.json]
"""
import argparse
import json
import os
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

import numpy as np  # noqa: E402

import genomics_rs_b200 as gx  # noqa: E402
from genomics_rs_b200 import _lib, workloads as wl  # noqa: E402

SCORES = (1, -2, -1, -5)   # config.toml
CHUNK = 1 << 18
FIELDS = ("score", "start_i", "start_j", "end_i", "end_j", "n_ops", "matches", "mismatches", "gap_extensions",
          "opening_gaps", "lcs_at_first_max")


def gpu_info():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True, timeout=60)
    name, power, clk = [x.strip() for x in q.stdout.splitlines()[0].split(",")]
    return {"name": name, "power_limit": power, "max_sm_clock": clk}


def device_used_bytes():
    import torch
    free, total = torch.cuda.mem_get_info()
    return int(total - free)


def pinned_like(arr):
    import torch
    t = torch.empty(arr.nbytes, dtype=torch.uint8, pin_memory=True)
    v = t.numpy().view(arr.dtype)
    v[:] = arr.reshape(-1)
    return t, v


def med(xs):
    return float(np.median(np.asarray(xs, np.float64)))


def same(got, gops, goff, exp, eops, eoff):
    for f in FIELDS:
        if not np.array_equal(got[f], exp[f]):
            return False
    n = got["n_ops"].astype(np.int64)
    for q in range(len(got)):
        a, b = int(goff[q]), int(eoff[q])
        if not np.array_equal(gops[a:a + n[q]], eops[b:b + n[q]]):
            return False
    return True


def kernels(packed, is_local, reps):
    blob, off1, len1, off2, len2 = packed
    cells = float(((len1 + 1) * (len2 + 1)).sum())
    wave = gx.Plan(len1, len2, SCORES, is_local, traceback=True)
    wave.upload(blob, off1, off2)
    reads = {}
    for bits in ("default", "32"):
        if bits == "32":
            os.environ["GX_READS32"] = "1"
        p = gx.Plan(len1, len2, SCORES, is_local, traceback=False, start_cell=True)
        os.environ.pop("GX_READS32", None)
        p.upload(blob, off1, off2)
        reads[bits] = p
    t = {"align_reads": [], "wave_fill": [], "wave_walk": [], "cells_default": [], "cells_32": []}
    got = None
    for r in range(reps + 1):     # the first round warms every variant up and is not counted
        res, ops, ops_off = gx.align_reads(blob, off1, len1, off2, len2, SCORES, is_local)
        wave.execute()
        for bits, p in reads.items():
            p.execute()
        if r == 0:
            got = (res, ops, ops_off)
            continue
        t["align_reads"].append(float(res["fill_ms"][0]))
        t["wave_fill"].append(wave.fill_ms)
        t["wave_walk"].append(wave.walk_ms)
        t["cells_default"].append(reads["default"].fill_ms)
        t["cells_32"].append(reads["32"].fill_ms)
    exp, eops, eoff = wave.fetch()
    parity = same(got[0], got[1], got[2], exp, eops, eoff)
    out = {k: med(v) for k, v in t.items()}
    out["wave_fill_plus_walk"] = out["wave_fill"] + out["wave_walk"]
    out["cells_default_lane_bits"] = reads["default"].stat(26)
    out["wave_code_bytes"] = wave.stat(4)
    out["speedup_vs_wavefront"] = out["wave_fill_plus_walk"] / out["align_reads"]
    out["traceback_over_start_cells_32"] = out["align_reads"] / out["cells_32"]
    out["align_reads_tcups"] = cells / (out["align_reads"] * 1e-3) / 1e12
    out["cells"] = cells
    out["samples"] = t
    out["parity_with_wavefront_plan"] = bool(parity)
    for p in [wave] + list(reads.values()):
        p.close()
    return out


def e2e(n_pairs, reps):
    t0 = time.perf_counter()
    blob, off1, len1, off2, len2 = wl.reads150(0, n_pairs)
    gen_s = time.perf_counter() - t0
    _keep, pblob = pinned_like(blob)
    del blob
    ops_off = np.zeros(n_pairs + 1, np.uint64)
    np.cumsum(len1 + len2 + np.uint64(1), out=ops_off[1:])
    _k2, ops = pinned_like(np.zeros(int(ops_off[-1]), np.uint8))
    res = np.zeros(n_pairs, gx.RESULT_DTYPE)
    out = {"pairs": n_pairs, "generate_s": gen_s, "wire_bytes_per_pair_d2h": 20 + 301, "wire_bytes_per_pair_h2d": 16 + 4 + 300}
    lib = _lib.ensure_init()
    from genomics_rs_b200.alignment import _scores_struct
    sc = np.empty(n_pairs, np.int64)
    si, sj = np.empty(n_pairs, np.uint64), np.empty(n_pairs, np.uint64)
    ta, tc, fill = [], [], []
    for r in range(reps + 1):
        t0 = time.perf_counter()
        _lib.check(lib.gx_align_reads(pblob.ctypes.data, pblob.size, off1.ctypes.data, len1.ctypes.data, off2.ctypes.data,
                                      len2.ctypes.data, n_pairs, _scores_struct(SCORES), 1, res.ctypes.data, ops.ctypes.data,
                                      ops_off.ctypes.data))
        a = time.perf_counter() - t0
        if r == 0:
            out["device_used_after_first_call"] = device_used_bytes()
        t0 = time.perf_counter()
        _lib.check(lib.gx_score_batch_cells(pblob.ctypes.data, pblob.size, off1.ctypes.data, len1.ctypes.data,
                                            off2.ctypes.data, len2.ctypes.data, n_pairs, _scores_struct(SCORES), 1,
                                            sc.ctypes.data, si.ctypes.data, sj.ctypes.data))
        c = time.perf_counter() - t0
        if r:
            ta.append(a * 1e3)
            tc.append(c * 1e3)
            fill.append(float(res["fill_ms"][0]))
    out["align_reads_ms"] = med(ta)
    out["align_reads_kernel_ms"] = med(fill)
    out["score_batch_cells_ms"] = med(tc)
    out["samples"] = {"align_reads_ms": ta, "score_batch_cells_ms": tc, "align_reads_kernel_ms": fill}
    out["align_reads_e2e_tcups"] = n_pairs * 151 * 151 / (out["align_reads_ms"] * 1e-3) / 1e12
    out["scores_equal_score_batch_cells"] = bool(np.array_equal(res["score"], sc))
    out["start_cells_equal"] = bool(np.array_equal(res["start_i"], si) and np.array_equal(res["start_j"], sj))
    # gx_align_batch with traceback on the same pairs: one wavefront plan (dense codes for every pair)
    t0 = time.perf_counter()
    rc = lib.gx_align_batch(pblob.ctypes.data, pblob.size, off1.ctypes.data, len1.ctypes.data, off2.ctypes.data,
                            len2.ctypes.data, n_pairs, _scores_struct(SCORES), 1, _lib.GX_FLAG_TRACEBACK, res.ctypes.data,
                            ops.ctypes.data, ops_off.ctypes.data)
    dt = time.perf_counter() - t0
    out["align_batch_traceback"] = {"status": int(rc), "ms": dt * 1e3,
                                    "detail": lib.gx_last_error().decode() if rc else "",
                                    "fill_ms": float(res["fill_ms"][0]) if rc == 0 else None,
                                    "walk_ms": float(res["walk_ms"][0]) if rc == 0 else None}
    return out


def bench_ab(parent, reps):
    def line(tree):
        p = subprocess.run([sys.executable, os.path.join(tree, "bench.py"), "--gpus", "1", "--steps", "10", "--warmup", "3",
                            "--no-cpu-baseline", "--no-k0"], capture_output=True, text=True, timeout=1800, cwd=tree)
        js = [x for x in p.stdout.splitlines() if x.startswith("{")]
        if p.returncode or not js:
            return {"error": (p.stderr or p.stdout)[-600:]}
        d = json.loads(js[-1])
        row = {"corona45": d["value"], "parity_ok": d.get("all_parity_ok", d.get("parity_ok"))}
        for k, v in d.get("configs", {}).items():
            row[k] = v.get("value")
            row[k + "_parity_ok"] = v.get("parity_ok")
        return row
    out = {"parent": [], "this": []}
    parent = os.path.abspath(parent)
    for _ in range(reps):
        out["parent"].append(line(parent))
        out["this"].append(line(ROOT))
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--pairs", type=int, default=10_000_000)
    ap.add_argument("--parent", default=None, help="the parent commit's tree (built): bench.py lines alternated with this one")
    ap.add_argument("--bench-reps", type=int, default=2)
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "read_traceback.json"))
    args = ap.parse_args()
    _lib.ensure_init(0)
    rec = {"gpu": gpu_info(), "scores": SCORES, "reps": args.reps, "chunk_pairs": CHUNK}
    # device bytes in use (this process's CUDA context included): after 4 chunks every lane has held a chunk
    rec["memory"] = {"before": device_used_bytes()}
    gx.align_reads(*wl.reads150(0, 4 * CHUNK), SCORES, True)
    rec["memory"]["after_%d_pairs" % (4 * CHUNK)] = device_used_bytes()
    small = wl.reads150(0, CHUNK)
    rec["e2e"] = e2e(args.pairs, max(1, args.reps // 2))
    rec["memory"]["after_%d_pairs" % args.pairs] = rec["e2e"].pop("device_used_after_first_call")
    for is_local in (True, False):
        rec["kernels_local" if is_local else "kernels_global"] = kernels(small, is_local, args.reps)
    if args.parent:
        rec["bench"] = bench_ab(args.parent, args.bench_reps)
    kl, kg = rec["kernels_local"], rec["kernels_global"]
    rec["summary"] = {
        "local_align_reads_ms": kl["align_reads"], "local_wavefront_fill_plus_walk_ms": kl["wave_fill_plus_walk"],
        "global_align_reads_ms": kg["align_reads"], "global_wavefront_fill_plus_walk_ms": kg["wave_fill_plus_walk"],
        "parity": kl["parity_with_wavefront_plan"] and kg["parity_with_wavefront_plan"],
        "e2e_10m_align_reads_ms": rec["e2e"]["align_reads_ms"], "e2e_10m_score_batch_cells_ms": rec["e2e"]["score_batch_cells_ms"],
    }
    os.makedirs(os.path.dirname(args.out), exist_ok=True)
    with open(args.out, "w") as f:
        json.dump(rec, f, indent=1)
    print(json.dumps(rec["summary"]))


if __name__ == "__main__":
    main()
