#!/usr/bin/env python
"""bench.py -- GCUPS of the affine-gap NW/SW hot path on B200, one process per GPU.

    python bench.py [--gpus N] [--steps K] [--warmup W]          # headline (config 3) + every other BASELINE config
    python bench.py --workload corona45|brca2_global|brca2_local|reads150|nw1m ...      # one workload only
    python -m torch.distributed.run --nproc-per-node N ... bench.py --gpus N ...
    python bench.py --impl reference ...      # the reference's CPU algorithm (oracle port) on the host cores
    python bench.py ... --dump-outputs DIR    # also write what the kernels computed in the last timed step as DIR/*.npy

A "step" is one pass of the hot path over the workload's batch of pairs:
  value      kernels only, sequences resident in HBM (gx_plan_execute / gx_band_execute), device-timed with CUDA events
  e2e        the public host-buffer call (gx_align_batch / gx_score_batch / gx_nw_score_banded): H2D + kernels + D2H, wall clock
Metric: GCUPS = sum (m+1)(n+1) / seconds / 1e9 (cells of the reference's table, algo.rs:172).

The JSON line's top level is the headline workload (BASELINE config 3, the metric's configuration); `configs` carries the
other four BASELINE configs (value, e2e, roofline, parity_ok each), so that every named shape is measured at every N.
Parity inside the bench uses only committed fixtures (tests/golden): no oracle code runs outside the `cpu_baseline` leg.
torch is used for process-group plumbing (rendezvous, barrier, max over ranks) and pinned host buffers only.
"""
from __future__ import annotations

import argparse
import atexit
import json
import os
import subprocess
import sys
import tempfile
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
sys.dont_write_bytecode = True      # the benchmark writes nothing into the tree (which may be read-only)

from genomics_rs_b200 import workloads as wl  # noqa: E402

SCORES = wl.CONFIG_TOML
GOLDEN = os.path.join(ROOT, "tests", "golden")

# ALU-pipe instructions per cell of the fill kernels, read off the SASS of the unmasked inner loops
# (tools/sass_loops.py; DESIGN.md 4): VIADDMNMX x2 + VIMNMX3 = 3 for the classic score-only cell, +1 VIMNMX for the running
# local maximum, +2 ISETP with traceback codes; the latency-optimised form (CHAIN1) trades the VIMNMX3 for two VIADDMNMX (+1).
# The adds (S, E) and the code accumulation are IMAD on the FMA pipe.  s16x2 read kernel: 6 ALU instructions per TWO cells.
ALU_PER_CELL = {"global_score": 3, "local_score": 4, "traceback": 5, "traceback_local": 6, "reads16": 3.0, "reads32": 4}
INSTR_PER_CELL = {"global_score": 5, "local_score": 6, "traceback": 9, "traceback_local": 10}     # ALU + FMA pipe, no glue


def measured_peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        d = json.load(open(p))
        return dict(hbm_gbs=float(d.get("hbm_gbs", 6650.0)), sm_max_mhz=float(d.get("sm_max_mhz", 1965.0)), source="measured")
    return dict(hbm_gbs=6650.0, sm_max_mhz=1965.0, source="fallback")


def ncu_traffic(workload: str):
    """DRAM bytes (read + write) of one launch of the dominant kernel from the committed ncu capture of the same command
    (profiles/*_traffic.json, written from `ncu --set full`); None when no capture exists for this workload."""
    for name in ("r2_traffic.json", "r1d_traffic.json"):
        p = os.path.join(ROOT, "profiles", name)
        if not os.path.exists(p):
            continue
        d = json.load(open(p)).get({"corona45": "prof_fill_corona45"}.get(workload, workload))
        if d:
            return d["dram_read_bytes"] + d["dram_write_bytes"], d.get("source", "profiles/" + name) + " (ncu --set full, one launch of the fill kernel)"
    return None, None


class ClockSampler:
    """nvidia-smi clocks / throttle reasons sampled every 200 ms during the timed region."""
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu: int):
        self.gpu = gpu
        self.proc = None
        self.lines = []

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.gpu), f"--query-gpu={self.Q}", "--format=csv,noheader,nounits",
                                          "-lms", "200"], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            atexit.register(self.proc.kill)     # a run that fails before stop() must not leave the sampler running
            self.th = threading.Thread(target=self._pump, daemon=True)
            self.th.start()
        except OSError:
            self.proc = None

    def _pump(self):
        for line in self.proc.stdout:
            self.lines.append(line.strip())

    def stop(self):
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.25)
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except Exception:
            self.proc.kill()
        sm, mx, reasons, power = [], [], set(), []
        for ln in self.lines:
            f = [x.strip() for x in ln.split(",")]
            if len(f) < 9:
                continue
            try:
                sm.append(float(f[1])); mx.append(float(f[2])); power.append(float(f[3]))
            except ValueError:
                continue
            for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), f[5:9]):
                if v.lower().startswith("active"):
                    reasons.add(name)
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "power_w_max": max(power) if power else None, "samples": len(sm), "reasons": sorted(reasons)}


# ----------------------------------------------------------------------------------------------------
def fnv_ops(ops: np.ndarray, start) -> str:
    """op-hash of SURVEY.md 8c: FNV-1a-64 fed, per op in walk order, with the 8 little-endian bytes of
    code*1000003 + i*10007 + j.  (Restated here so that the bench's parity check runs no oracle code.)"""
    i, j = int(start[0]), int(start[1])
    h = 1469598103934665603
    M = (1 << 64) - 1
    for c in ops.tolist():
        v = (c * 1000003 + i * 10007 + j) & M
        for _ in range(8):
            h = ((h ^ (v & 0xFF)) * 1099511628211) & M
            v >>= 8
        if c in (0, 1):
            i, j = max(i - 1, 0), max(j - 1, 0)
        elif c in (2, 4):
            j = max(j - 1, 0)
        else:
            i = max(i - 1, 0)
    return "%016x" % h


def build_workload(name: str, rank: int, world: int, n_pairs: int):
    """-> dict(blob, off1, len1, off2, len2, is_local, traceback, cells, desc, scaling, mode, gold)"""
    if name == "corona45":
        seqs, jobs = wl.corona_pairs()
        costs = [(len(seqs[a]) + 1) * (len(seqs[b]) + 1) for a, b in jobs]
        mine = wl.lpt_shards(costs, world)[rank]
        off, pos = [], 0
        for s in seqs:
            off.append(pos); pos += len(s)
        blob = np.frombuffer(b"".join(seqs), np.uint8).copy()
        off1 = np.array([off[jobs[k][0]] for k in mine], np.uint64)
        off2 = np.array([off[jobs[k][1]] for k in mine], np.uint64)
        len1 = np.array([len(seqs[jobs[k][0]]) for k in mine], np.uint64)
        len2 = np.array([len(seqs[jobs[k][1]]) for k in mine], np.uint64)
        g = json.load(open(os.path.join(GOLDEN, "oracle_goldens.json")))
        gold = {tuple(c["pair"]): c for c in g["corona"]}
        return dict(blob=blob, off1=off1, len1=len1, off2=off2, len2=len2, is_local=False, traceback=True,
                    cells=int(sum(costs[k] for k in mine)), scaling="strong", mode="traceback", gold=[gold[jobs[k]] for k in mine],
                    desc=CORONA_WHAT)
    if name in ("brca2_global", "brca2_local"):
        a, b = wl.brca2_pair()
        blob = np.frombuffer(a + b, np.uint8).copy()
        is_local = name.endswith("local")
        g = json.load(open(os.path.join(GOLDEN, "oracle_goldens.json")))
        gold = [next(p for p in g["pairs"] if p["fixture"] == "Human-Mouse-BRCA2-cds" and p["is_local"] == is_local)]
        return dict(blob=blob, off1=np.array([0], np.uint64), len1=np.array([len(a)], np.uint64),
                    off2=np.array([len(a)], np.uint64), len2=np.array([len(b)], np.uint64), is_local=is_local, traceback=True,
                    cells=(len(a) + 1) * (len(b) + 1), scaling="replicas", mode="traceback_local" if is_local else "traceback", gold=gold,
                    desc=f"config {'2' if is_local else '1'}: {'local SW' if is_local else 'global NW'} of "
                         "Human-Mouse-BRCA2-cds (11382 x 10346), score + traceback; one pair, one replica per rank")
    if name == "reads150":
        per = n_pairs // world
        first = rank * per
        blob, off1, len1, off2, len2 = wl.reads150(first, per)
        return dict(blob=blob, off1=off1, len1=len1, off2=off2, len2=len2, is_local=True, traceback=False,
                    cells=per * 151 * 151, scaling="strong", mode="local_score", gold=None, first=first,
                    desc=f"config 4: {n_pairs} synthetic 150 bp pairs (splitmix64), local SW score only, contiguous ranges per rank")
    raise SystemExit(f"unknown workload {name}")


def pinned_like(arr: np.ndarray):
    """copy into page-locked host memory (torch owns the allocation; numpy view for ctypes)"""
    import torch
    t = torch.empty(arr.size, dtype=torch.uint8, pin_memory=torch.cuda.is_available())
    v = t.numpy()
    v[:] = arr.view(np.uint8).reshape(-1)
    return t, v


def cpu_baseline_sample(march_native: bool = True, rows: int = 12000, threads: int = 1):
    """The reference's algorithm as written (oracle faithful variant: 48 B cells, F-order table, i-outer/j-inner)
    on a bounded sample of the workload: the first `rows` x `rows` bases of corona pair (0,1), global + retrace."""
    from oracle import gxo
    seqs, jobs = wl.corona_pairs()
    a, b = seqs[0][:rows], seqs[1][:rows]
    cells = (len(a) + 1) * (len(b) + 1)
    with tempfile.TemporaryDirectory() as tmp:      # the host-tuned oracle is compiled outside the tree
        so = gxo.build(march="native", out_dir=tmp) if march_native else None
        t0 = time.perf_counter()
        r = gxo.align_faithful(a, b, SCORES, False, so=so)
        dt = time.perf_counter() - t0
    out = dict(value=cells / dt / 1e9, unit="GCUPS", cores=threads, kind="port",
               sample=f"oracle faithful variant (48 B cells, column-major, single thread like algo.rs), global NW + retrace of the "
                      f"first {rows}x{rows} bases of corona pair (Covid_Australia, Covid_Brazil): {cells} cells in {dt:.2f} s "
                      f"(fill {r.fill_ms / 1e3:.2f} s)",
               seconds=dt)
    full = os.path.join(ROOT, "profiles", "r2_cpu_full_pair.json")
    if os.path.exists(full):   # one FULL 30 kb pair (43 GB table) run once on a GPU box's host: tools/full_pair_oracle.py
        out["full_pair"] = json.load(open(full))
    return out


def workload_config(name: str, what: str, cells_per_step: float) -> dict:
    """`config` of the JSON line: the workload, identical in our arm and in the --impl reference arm"""
    return {"workload": name, "what": what, "scores": dict(zip(("s_match", "s_mismatch", "g", "h"), SCORES)),
            "cells_per_step": float(cells_per_step)}


CORONA_WHAT = ("config 3: all-vs-all global NW of the 10 comparison_data coronavirus genomes (45 pairs, ~30 kb each), "
               "score + traceback, pairs dealt LPT over ranks")


def mem_available_gb() -> float:
    try:
        for line in open("/proc/meminfo"):
            if line.startswith("MemAvailable:"):
                return int(line.split()[1]) / 1e6
    except OSError:
        pass
    return 0.0


def run_reference(args):
    """--impl reference: the reference's CPU implementation of the path (oracle port; the Rust crate cannot be built
    here) on the host cores.  The reference aligns ONE pair on ONE thread (no rayon in algo.rs); to use the host
    it is run as T independent single-threaded aligners, one bounded-sample pair each, per step."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    from concurrent.futures import ThreadPoolExecutor
    from oracle import gxo
    tmp = tempfile.TemporaryDirectory()      # the host-tuned oracle is compiled outside the tree (removed on return)
    so = gxo.build(march="native", out_dir=tmp.name)
    ncpu = os.cpu_count() or 1
    threads = max(1, min(ncpu, 32))
    # the largest prefix whose 48 B/cell tables fit a third of the free host memory with one aligner per thread
    # (a full 30 kb pair is 43 GB and 42 s on one thread: profiles/r2_cpu_full_pair.json)
    rows = 4000
    for cand in (12000, 8000, 6000):
        if threads * (cand + 1) ** 2 * 48 / 1e9 <= mem_available_gb() / 3:
            rows = cand
            break
    seqs, jobs = wl.corona_pairs()
    work = [(seqs[a][:rows], seqs[b][:rows]) for a, b in jobs]
    work = (work * ((threads + len(work) - 1) // len(work)))[:threads]
    cells = sum((len(a) + 1) * (len(b) + 1) for a, b in work)

    def one(ab):
        return gxo.align_faithful(ab[0], ab[1], SCORES, False, so=so).score   # ctypes releases the GIL

    def step():
        with ThreadPoolExecutor(threads) as ex:
            list(ex.map(one, work))

    for _ in range(min(args.warmup, 1)):
        step()
    t0 = time.perf_counter()
    for _ in range(args.steps):
        step()
    dt = (time.perf_counter() - t0) / args.steps
    val = cells / dt / 1e9
    sample = (f"{threads} concurrent single-threaded aligners (reference algorithm as written, 48 B cells), each the first "
              f"{rows}x{rows} bases of a corona pair, global NW + retrace; {cells} cells per step")
    print(json.dumps({
        "impl": "reference", "metric": "GCUPS (affine NW/SW, score+traceback)", "value": val, "unit": "GCUPS",
        "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup, "ms_per_step": dt * 1e3, "higher_is_better": True,
        "scaling": "strong", "vs_baseline": None, "dtype": "int64", "data": "reference fixtures (comparison_data genomes, prefixes)",
        "config": workload_config("corona45", CORONA_WHAT, sum((len(seqs[a]) + 1) * (len(seqs[b]) + 1) for a, b in jobs)),
        "cpu_baseline": {"value": val, "unit": "GCUPS", "cores": threads, "kind": "port", "sample": sample},
        "e2e": {"value": val, "unit": "GCUPS", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0}))


# ----------------------------------------------------------------------------------------------------
class Env:
    """process-group plumbing shared by the workloads"""

    def __init__(self, args):
        import torch
        import torch.distributed as dist
        self.torch, self.dist = torch, dist
        self.rank = int(os.environ.get("RANK", "0"))
        self.world = int(os.environ.get("WORLD_SIZE", "1"))
        self.local_rank = int(os.environ.get("LOCAL_RANK", "0"))
        if self.world != args.gpus and self.world > 1:
            raise SystemExit(f"--gpus {args.gpus} but WORLD_SIZE={self.world}")
        if not torch.cuda.is_available():
            raise SystemExit("bench.py needs a B200: libgxalign has no CPU path (use --impl reference for the CPU arm)")
        torch.cuda.set_device(self.local_rank)
        if self.world > 1:
            os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
            dist.init_process_group("nccl", device_id=torch.device("cuda", self.local_rank))
        self.peaks = measured_peaks()
        self.k0 = None

    def sync_all(self):
        if self.world > 1:
            self.dist.barrier()
        self.torch.cuda.synchronize()

    def reduce(self, values, op="max"):
        t = self.torch.tensor([float(v) for v in values], dtype=self.torch.float64, device="cuda")
        if self.world > 1:
            self.dist.all_reduce(t, op={"max": self.dist.ReduceOp.MAX, "sum": self.dist.ReduceOp.SUM, "min": self.dist.ReduceOp.MIN}[op])
        return [float(x) for x in t.tolist()]


def alu_roofline(env, kind: str, alu_per_cell: float, cells: float, kernel_ms: float, kernel: str, extra=None):
    """Per-pipe accounting (VERDICT r1): the fill is bound by the INT32 ALU pipe (VIADDMNMX / VIMNMX3 / ISETP issue there;
    the adds and the code accumulation are IMAD on the FMA pipe).  achieved = cells x ALU-pipe instructions per cell (from
    the SASS) / kernel time; peak = the ALU pipe's issue rate measured on THIS GPU in this run (gx_k0_measure: VIADDMNMX,
    CUDA-event timed, dependency-free) x SMs x the SM clock seen by the probe.  frac <= 1 by construction."""
    k0 = env.k0 or {}
    sms = int(k0.get("sm_count", 148))
    ghz = float(k0.get("sm_ghz", env.peaks["sm_max_mhz"] / 1e3))
    alu_rate = float(k0.get("viaddmnmx", 2.0))        # warp-instructions / clk / SM
    peak = sms * alu_rate * 32.0 * ghz * 1e9 / 1e12
    achieved = cells * alu_per_cell / (kernel_ms * 1e-3) / 1e12
    cells_clk_sm = cells / (kernel_ms * 1e-3) / (sms * ghz * 1e9)
    out = {"bound": "int32-alu-pipe", "kernel": kernel, "achieved": achieved, "peak": peak, "unit": "T ALU-pipe lane-instr/s",
           "frac": achieved / peak, "alu_instr_per_cell": alu_per_cell, "cells_per_clk_per_sm": cells_clk_sm,
           "peak_basis": f"{sms} SMs x {alu_rate:.3f} warp-instr/clk/SM (VIADDMNMX, event-timed by gx_k0_measure"
                         f"{'' if env.k0 else ' -- probe skipped, nominal 2.0'}) x 32 lanes x {ghz:.3f} GHz",
           "gcups_kernel": cells / (kernel_ms * 1e-3) / 1e9, "traffic": None}
    mix = {"global_score": "score_cell", "local_score": "score_cell", "traceback": "traceback_cell", "traceback_local": "traceback_cell"}.get(kind)
    if mix and k0.get(mix):
        # what the SM issues for the cell's own instruction mix with NO dependencies and NO glue (5 / 9 instructions per cell)
        ceil = float(k0[mix]) * 32.0 / INSTR_PER_CELL["global_score" if mix == "score_cell" else "traceback"]
        out["mix_ceiling_cells_per_clk_per_sm"] = ceil
        out["frac_of_mix_ceiling"] = cells_clk_sm / ceil
    if extra:
        out.update(extra)
    return out


def check_gold(w, res, ops, ops_off) -> bool:
    """results of this rank's pairs against the committed goldens (score, start/end cell, op count, counters, op-hash of
    the first pair)"""
    ok = True
    for q, g in enumerate(w["gold"]):
        r = res[q]
        ok &= int(r["score"]) == g["score"] and int(r["n_ops"]) == g["n_ops"]
        ok &= [int(r["start_i"]), int(r["start_j"])] == g["start"] and [int(r["end_i"]), int(r["end_j"])] == g["end"]
        ok &= (int(r["matches"]), int(r["mismatches"]), int(r["gap_extensions"]), int(r["opening_gaps"])) == (
            g["matches"], g["mismatches"], g["gap_extensions"], g["opening_gaps"])
        if q == 0 and ops is not None:
            o = int(ops_off[q])
            ok &= fnv_ops(ops[o:o + int(r["n_ops"])], (int(r["start_i"]), int(r["start_j"]))) == g["op_hash"]
    return bool(ok)


RESULT_FIELDS = ("score", "start_i", "start_j", "end_i", "end_j", "n_ops", "matches", "mismatches", "gap_extensions",
                 "opening_gaps")
SCORE_SAMPLE = 1 << 20      # score-only batches with more pairs are dumped as this many pairs, a fixed seeded sample


def dump_outputs(args, env, workload: str, arrays: dict) -> None:
    """--dump-outputs DIR: what this rank's last timed step computed, as DIR/<workload>_<array>.npy (float64; the op
    codes float32).  With several ranks every rank writes its own shard, the file names ending in _rank<r>."""
    os.makedirs(args.dump_outputs, exist_ok=True)
    tag = f"_rank{env.rank}" if env.world > 1 else ""
    for key, v in arrays.items():
        np.save(os.path.join(args.dump_outputs, f"{workload}_{key}{tag}.npy"), np.asarray(v, np.float32 if key == "ops" else np.float64))


def traceback_outputs(res, ops, ops_off) -> dict:
    """per-pair results, and the op codes of every pair in walk order, concatenated (ops_off holds capacities)"""
    out = {f: res[f] for f in RESULT_FIELDS}
    out["ops"] = np.concatenate([ops[int(o):int(o) + int(k)] for o, k in zip(ops_off[:-1], res["n_ops"])])
    return out


def run_plan_workload(env, args, name: str, steps: int, warmup: int, headline: bool):
    """corona45 / brca2_* / reads150 through a resident plan (kernels only) and the public host-buffer call (e2e)."""
    import genomics_rs_b200 as gx
    from genomics_rs_b200 import _lib
    torch = env.torch
    w = build_workload(name, env.rank, env.world, args.pairs)
    pin_t, blob = pinned_like(w["blob"])
    plan = gx.Plan(w["len1"], w["len2"], SCORES, w["is_local"], traceback=w["traceback"])
    plan.upload(blob, w["off1"], w["off2"])
    for _ in range(warmup):
        plan.execute()
    # timing rule: inputs larger than L2, or flush it.  A workload whose per-step working set (codes + boundary buffers +
    # sequences) is below 2x the 126 MB L2 gets a 512 MB buffer rewritten between the timed steps (outside the CUDA-event
    # span inside gx_plan_execute, so the flush itself is not timed).
    flush = None
    if plan.stat(5) < 2.5e8:
        flush = torch.empty(512 << 20, dtype=torch.uint8, device="cuda")
    sampler = ClockSampler(env.local_rank) if headline else None
    env.sync_all()
    if sampler:
        sampler.start()
    fill_ms, walk_ms, launches = 0.0, 0.0, 0
    t0 = time.perf_counter()
    for it in range(steps):
        if flush is not None:
            flush.fill_(it & 0xFF)
            torch.cuda.synchronize()
        plan.execute()
        fill_ms += plan.fill_ms
        walk_ms += plan.walk_ms
        launches += plan.launches
    env.sync_all()
    wall_ms = (time.perf_counter() - t0) * 1e3
    clocks = sampler.stop() if sampler else None
    dev_ms = fill_ms + walk_ms
    n = int(w["len1"].size)
    parity = {}
    # ---- parity of the resident plan against the committed goldens
    if w["traceback"]:
        res, ops, ops_off = plan.fetch()
        parity["goldens"] = check_gold(w, res, ops, ops_off)
        if args.dump_outputs:
            dump_outputs(args, env, name, traceback_outputs(res, ops, ops_off))
    elif args.dump_outputs:
        scores = plan.fetch_scores()
        pick = np.arange(n) if n <= SCORE_SAMPLE else np.sort(np.random.default_rng(0).choice(n, SCORE_SAMPLE, replace=False))
        dump_outputs(args, env, name, {"pair": w["first"] + pick, "score": scores[pick]})
    # ---- end to end: host buffers in, host buffers out, through the public batch call
    if w["traceback"]:
        res = np.zeros(n, dtype=gx.RESULT_DTYPE)
        ops_off = np.zeros(n + 1, np.uint64)
        np.cumsum(w["len1"] + w["len2"] + np.uint64(1), out=ops_off[1:])
        ops_t = torch.empty(int(ops_off[-1]), dtype=torch.uint8, pin_memory=True)
        ops = ops_t.numpy()
        lib = _lib.load()
        sc = _lib.GxScores(*SCORES)

        def e2e_step():
            _lib.check(lib.gx_align_batch(blob.ctypes.data, blob.size, w["off1"].ctypes.data, w["len1"].ctypes.data,
                                          w["off2"].ctypes.data, w["len2"].ctypes.data, n, sc, int(w["is_local"]),
                                          _lib.GX_FLAG_TRACEBACK, res.ctypes.data, ops.ctypes.data, ops_off.ctypes.data))
        d2h = n * gx.RESULT_DTYPE.itemsize + int((w["len1"] + w["len2"] + np.uint64(1)).sum())
        h2d = int(blob.size) + n * 104
    else:
        scores_out = np.zeros(n, np.int64)

        def e2e_step():
            gx.score_batch(blob, w["off1"], w["len1"], w["off2"], w["len2"], SCORES, w["is_local"], out=scores_out)
        d2h = n * 4
        h2d = int(blob.size) + n * 16
    for _ in range(min(warmup, 2)):
        e2e_step()
    env.sync_all()
    t0 = time.perf_counter()
    for _ in range(steps):
        e2e_step()
    env.sync_all()
    e2e_ms = (time.perf_counter() - t0) * 1e3 / steps
    if w["traceback"]:
        parity["e2e_goldens"] = check_gold(w, res, ops, ops_off)
    else:
        # the streamed host-buffer call and the resident plan must agree pair for pair ...
        parity["streamed_equals_plan"] = bool(np.array_equal(scores_out, plan.fetch_scores()))
        # ... and SURVEY 8d's parity sets (every score of the first 100 000 mutated pairs + a strided 1 % of the throughput
        # set) must equal the frozen oracle scores (tests/golden/config4_scores.npz); rank 0 runs them
        if env.rank == 0:
            gold = np.load(os.path.join(GOLDEN, "config4_scores.npz"))
            pb = wl.reads150(0, wl.CONFIG4_PARITY_PAIRS, parity_set=True)
            got = gx.score_batch(pb[0], pb[1], pb[2], pb[3], pb[4], SCORES, True)
            parity["parity_set_100k"] = bool(np.array_equal(got, gold["parity"].astype(np.int64)))
            per, first = n, w["first"]
            idx = np.arange(0, args.pairs, wl.CONFIG4_STRIDE, dtype=np.int64)
            sel = idx[(idx >= first) & (idx < first + per)]
            parity["strided_1pct"] = bool(sel.size > 0 and np.array_equal(scores_out[sel - first],
                                                                           gold["strided"][sel // wl.CONFIG4_STRIDE].astype(np.int64))) \
                if args.pairs == 10_000_000 else None
    kind = int(plan.stat(9))
    K, chain1 = int(plan.stat(15)), int(plan.stat(17))
    code_bytes = float(plan.stat(4))
    code_frac = plan.stat(23) if plan.stat(23) > 0 else 1.0     # share of the cells whose tile writes direction codes (code band)
    band_fallbacks = int(max(plan.stat(24), 0))
    plan.close()
    del pin_t, flush

    # ---- max over ranks, totals over ranks
    ms_step, wall_step, e2e_step_ms, fill_step, walk_step = env.reduce(
        [dev_ms / steps, wall_ms / steps, e2e_ms, fill_ms / steps, walk_ms / steps], "max")
    cells, launches_all, h2d_all, d2h_all, code_all = env.reduce([w["cells"], launches, h2d, d2h, code_bytes], "sum")
    par_ok = env.reduce([1.0 if all(v is not False for v in parity.values()) else 0.0], "min")[0] == 1.0
    replicas = w["scaling"] == "replicas"
    if replicas:
        cells = float(w["cells"]) * env.world      # every rank aligned its own copy of the pair
    out = None
    if env.rank == 0:
        value = cells / (ms_step * 1e-3) / 1e9
        e2e_val = cells / (e2e_step_ms * 1e-3) / 1e9
        my_cells, my_fill = float(w["cells"]), fill_ms / steps
        if kind == 1:
            roof = alu_roofline(env, "reads16", ALU_PER_CELL["reads16"], my_cells, my_fill, "gx_reads16_kernel",
                                {"note": "s16x2: two pairs per register, 6 ALU-pipe instructions per two cells"})
        else:
            alu = ALU_PER_CELL[w["mode"]] + (1 if chain1 else 0)
            extra = {"K": K, "chain1": bool(chain1)}
            if w["traceback"] and code_frac < 1.0:
                # code band: only tiles near the table's diagonal run the 5-ALU traceback cell, the rest the 3-ALU score cell
                alu = ALU_PER_CELL["global_score"] + (1 if chain1 else 0) + 2.0 * code_frac
                extra.update({"code_cell_frac": code_frac, "band_fallbacks": band_fallbacks,
                              "note": "ALU instructions per cell = 3 + 2 x the share of cells in code-writing tiles"})
            roof = alu_roofline(env, w["mode"] if code_frac >= 1.0 else "mixed", alu, my_cells, my_fill, "gx_fill_kernel", extra)
        hbm = None
        if w["traceback"]:
            if env.world == 1:
                roof["traffic"], roof["traffic_source"] = ncu_traffic(name)
            roof["algorithmic_bytes"] = code_bytes * code_frac    # 2-bit codes written once per cell of a code-writing tile
            roof["traffic_note"] = ("DRAM traffic also holds the strip-boundary hand-off (8 B per row per strip boundary, written once and "
                                    "polled through L2): ~1.25 GB per step for the 45 pairs at K=8")
            gbs = code_bytes * code_frac / (my_fill * 1e-3) / 1e9
            hbm = {"bound": "hbm", "achieved": gbs, "peak": env.peaks["hbm_gbs"], "unit": "GB/s", "frac": gbs / env.peaks["hbm_gbs"],
                   "what": "traceback codes written once per cell (0.25 B/cell)", "peak_source": env.peaks["source"]}
        out = {
            "metric": "GCUPS (affine NW/SW, score+traceback)" if w["traceback"] else "GCUPS (affine SW, score only)",
            "value": value, "unit": "GCUPS", "n_gpus": env.world, "steps": steps, "warmup": warmup,
            "ms_per_step": ms_step, "higher_is_better": True, "scaling": w["scaling"], "vs_baseline": None,
            "dtype": "int32" if kind == 0 else "int16x2",
            "data": "reference fixtures (tests/golden/fasta, gz copies of comparison_data/test_data)"
            if name != "reads150" else "synthetic (splitmix64 reads, SURVEY 8d)",
            "config": workload_config(name, w["desc"], cells),
            "plan": {"K": K, "chain1": bool(chain1),
                     "l2": ("each step rewrites %.2f GB of traceback codes + boundary buffers, far above the 126 MB L2, so no "
                            "step sees a warm cache" % (code_all / 1e9)) if code_all > 2e8 else
                           ("inputs (%.2f GB) exceed L2" % (blob.size * env.world / 1e9)) if blob.size * env.world > 2e8 else
                           "working set below L2: a 512 MB buffer is rewritten between the timed steps (L2 flush, outside the timed span)"},
            "wall_ms_per_step": wall_step, "fill_ms_per_step": fill_step, "walk_ms_per_step": walk_step,
            "e2e": {"value": e2e_val, "unit": "GCUPS", "ms_per_step": e2e_step_ms, "h2d_bytes_per_step": h2d_all,
                    "d2h_bytes_per_step": d2h_all, "api": "gx_align_batch" if w["traceback"] else "gx_score_batch"},
            "gpu_launches": int(launches_all), "parity_ok": par_ok, "parity": parity,
            "roofline": roof, "roofline_hbm": hbm,
        }
        if clocks is not None:
            out["clocks"] = clocks
    return out


def run_banded(env, args, steps: int, warmup: int, headline: bool = False):
    """config 5: ONE synthetic 1 Mbp x 1 Mbp pair (splitmix64, SURVEY 8d), global NW score only, column-banded over
    the ranks (one band per GPU; boundary columns stored into the neighbour's HBM over NVLink by the fill kernel)."""
    import genomics_rs_b200 as gx
    from genomics_rs_b200 import banded
    torch, dist, rank, world = env.torch, env.dist, env.rank, env.world
    n = args.length
    a, b = wl.long_pair(n)
    gold_all = json.load(open(os.path.join(GOLDEN, "config5_scores.json")))["prefix_scores"]
    gold = gold_all.get(str(n))
    pin_a, av = pinned_like(a)
    pin_b, bv = pinned_like(b)
    cells = (n + 1) * (n + 1)

    # ---- parity of the SAME multi-GPU banded path on prefixes the CPU oracle froze (SURVEY 8d config 5 (i))
    band_parity = {}
    for pre in (65536, 262144):
        if pre >= n or str(pre) not in gold_all:
            continue
        if world == 1:
            sc = gx.nw_score_banded_local(av[:pre], bv[:pre], SCORES, 1)
        else:
            sc, bd = banded.nw_score_banded(av[:pre], bv[:pre], SCORES)
            bd.close()
        band_parity[str(pre)] = bool(sc == gold_all[str(pre)])

    band = gx.Band(n, n, world, rank, rank + 1, SCORES)
    if world > 1:
        banded.connect_ring(band)
    band.upload(av, bv)
    for _ in range(warmup):
        band.execute()
    sampler = ClockSampler(env.local_rank) if headline else None
    env.sync_all()
    if sampler:
        sampler.start()
    t0 = time.perf_counter()
    fill_ms = 0.0
    for _ in range(steps):
        band.execute()              # synchronous on this rank; ranks pipeline against each other (ack flow control)
        fill_ms += band.fill_ms
    env.sync_all()
    wall_ms = (time.perf_counter() - t0) * 1e3 / steps
    clocks = sampler.stop() if sampler else None
    score = band.score()
    launches = int(band.stat(2)) * steps
    my_cells = float(band.stat(3))
    K = int(band.stat(15))
    chain1 = int(band.stat(17))
    dev_bytes = band.stat(5)
    band.close()

    # ---- end to end: host sequences in, score out, through the public entry point (create + H2D + kernels + D2H)
    # (both entry points keep the band object of the previous call with the same shape: the first call, untimed, creates it)
    def e2e_step():
        if world == 1:
            return gx.nw_score_banded_local(av, bv, SCORES, 1)
        return banded.nw_score_banded(av, bv, SCORES, cache=True)[0]
    e2e_step()
    env.sync_all()
    t0 = time.perf_counter()
    for _ in range(steps):
        e2e_score = e2e_step()
    env.sync_all()
    e2e_ms = (time.perf_counter() - t0) * 1e3 / steps

    banded.clear_cache()
    ms_step, e2e_step_ms, fill_max = env.reduce([wall_ms, e2e_ms, fill_ms / steps], "max")
    per_rank = [0.0] * world
    per_rank[rank] = fill_ms / steps
    per_rank = env.reduce(per_rank, "sum")
    launches_all, final_score = env.reduce([launches, score if score is not None else 0], "sum")
    out = None
    if rank == 0:
        final_score = int(final_score)
        if args.dump_outputs:
            dump_outputs(args, env, "nw1m", {"score": [final_score]})
        full_ok = (gold is None) or (final_score == gold and e2e_score == gold)
        par = dict(band_parity)
        par[str(n)] = bool(full_ok)
        alu = ALU_PER_CELL["global_score"] + (1 if chain1 else 0)
        roof = alu_roofline(env, "global_score", alu, my_cells, per_rank[0], "gx_fill_kernel",
                            {"K": K, "chain1": bool(chain1),
                             "note": "rank 0's band (never waits for a neighbour); every rank's kernel ms is in config.band_fill_ms"})
        link = None
        if world > 1:
            link = {"bound": "nvlink", "bytes_per_step_per_edge": 8 * n, "edges": world - 1,
                    "achieved_GBs_per_edge": 8 * n / (ms_step * 1e-3) / 1e9, "peak_GBs": 770.0,
                    "what": "8 B per row per band edge, stored by the fill kernel into the neighbour's HBM (st.relaxed.sys.u64)"}
        out = {
            "metric": "GCUPS (affine NW, score only, one 1 Mbp x 1 Mbp pair column-banded over the GPUs)",
            "value": cells / (ms_step * 1e-3) / 1e9, "unit": "GCUPS", "n_gpus": world, "steps": steps, "warmup": warmup,
            "ms_per_step": ms_step, "higher_is_better": True, "scaling": "strong", "vs_baseline": None, "dtype": "int32",
            "data": "synthetic (splitmix64 pair, SURVEY 8d: s2 = s1 with 1/32 substitutions)",
            "config": workload_config("nw1m", f"config 5: one {n} x {n} global NW, score only; one column band per GPU; boundary columns "
                                      "handed over by peer stores inside the fill kernel (no collective on the data path)", cells),
            "plan": {"K": K, "chain1": bool(chain1), "bands": world, "band_fill_ms": per_rank, "score": final_score,
                     "score_matches_frozen_oracle": bool(full_ok),
                     "l2": "each step streams %.1f GB of strip-boundary buffers (8 B per row per strip), far above the 126 MB L2"
                           % (dev_bytes / 1e9)},
            "wall_ms_per_step": ms_step, "fill_ms_per_step": fill_max,
            "e2e": {"value": cells / (e2e_step_ms * 1e-3) / 1e9, "unit": "GCUPS", "ms_per_step": e2e_step_ms,
                    "h2d_bytes_per_step": float(2 * n + 104 * 1), "d2h_bytes_per_step": float(104 * world),
                    "api": "gx_nw_score_banded" if world == 1 else "gx_band_create/export/connect/upload/execute/score (nw_score_banded)"},
            "gpu_launches": int(launches_all), "parity_ok": bool(all(par.values())), "band_parity": bool(all(par.values())),
            "parity": {"frozen_oracle_scores_through_this_banded_path": par},
            "roofline": roof, "roofline_link": link}
        if clocks is not None:
            out["clocks"] = clocks
    del pin_a, pin_b
    return out


SECONDARY = ("brca2_global", "brca2_local", "reads150", "nw1m")
CONFIG_KEY = {"brca2_global": "brca2_global", "brca2_local": "brca2_local", "reads150": "reads10m", "nw1m": "nw1m", "corona45": "corona45"}


def slim(rec):
    """what a secondary config contributes to the headline line"""
    keep = ("metric", "value", "unit", "ms_per_step", "fill_ms_per_step", "walk_ms_per_step", "scaling", "steps", "warmup", "dtype", "e2e",
            "gpu_launches", "parity_ok", "band_parity", "parity", "roofline", "roofline_hbm", "roofline_link")
    out = {k: rec[k] for k in keep if k in rec and rec[k] is not None}
    out["what"] = rec["config"]["what"]
    out["cells_per_step"] = rec["config"]["cells_per_step"]
    out.update({k: v for k, v in rec.get("plan", {}).items()})
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--workload", default="all", help="all (headline corona45 + the other BASELINE configs) or one workload")
    ap.add_argument("--only-headline", action="store_true", help="with --workload all: skip the secondary configs")
    ap.add_argument("--pairs", type=int, default=10_000_000, help="reads150: total pairs")
    ap.add_argument("--length", type=int, default=1_000_000, help="nw1m: bases per sequence")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-k0", action="store_true")
    ap.add_argument("--dump-outputs", metavar="DIR", help="write the results of every workload's last timed step as DIR/*.npy")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.impl == "reference":
        run_reference(args)
        return
    if args.warmup < 3:
        print(f"note: --warmup {args.warmup} < 3 (timing rules want >= 3 warm-up steps)", file=sys.stderr)
    env = Env(args)
    import genomics_rs_b200 as gx
    from genomics_rs_b200 import _lib
    _lib.ensure_init(env.local_rank)
    if env.rank == 0 and not args.no_k0:
        env.k0 = gx.k0_measure()

    head_name = "corona45" if args.workload == "all" else args.workload
    if head_name == "nw1m":
        line = run_banded(env, args, args.steps, args.warmup, headline=True)
    else:
        line = run_plan_workload(env, args, head_name, args.steps, args.warmup, headline=True)
    if args.workload == "all" and not args.only_headline:
        configs = {}
        sec_warm = max(3, min(args.warmup, 3))
        for name in SECONDARY:
            t0 = time.perf_counter()
            try:
                rec = run_banded(env, args, args.steps, sec_warm) if name == "nw1m" else \
                    run_plan_workload(env, args, name, args.steps, sec_warm, headline=False)
                if env.rank == 0:
                    configs[CONFIG_KEY[name]] = slim(rec)
                    configs[CONFIG_KEY[name]]["bench_seconds"] = time.perf_counter() - t0
            except Exception as e:      # a secondary config must not take the headline number down with it -- but it is reported
                if env.world > 1:
                    raise
                configs[CONFIG_KEY[name]] = {"error": str(e)[:400], "parity_ok": False}
        if env.rank == 0:
            line["configs"] = configs
            line["all_parity_ok"] = bool(line.get("parity_ok")) and all(c.get("parity_ok") for c in configs.values())
    if env.rank == 0:
        if head_name == "corona45" and not args.no_cpu_baseline and env.world == 1:
            line["cpu_baseline"] = cpu_baseline_sample()
        else:
            line["cpu_baseline"] = None
        line["k0"] = env.k0
        print(json.dumps(line))
    if env.world > 1:
        env.dist.destroy_process_group()


if __name__ == "__main__":
    main()
