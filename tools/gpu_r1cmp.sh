#!/bin/bash
# A/B of the round-1 library (built from commit 11bb267) against the current one on the single-pair and shard workloads
mkdir -p gpurun_out
for tag in r1 ""; do
  lib=genomics_rs_b200/libgxalign${tag:+_$tag}.so
  out=gpurun_out/sweep_r1cmp_${tag:-cur}.jsonl; rm -f $out
  GX_LIB_PATH=$PWD/$lib timeout 600 python tools/sweep_kr.py --workloads brca2_global,brca2_local,corona1,corona6,corona11,corona23,corona45,nw200k --k 4 --chain 0,1 --steps 5 --out $out > ${out%.jsonl}.log 2>&1
  echo "== ${tag:-current}"; python - $out <<'PY'
import json, sys
for l in open(sys.argv[1]):
    r = json.loads(l)
    if 'error' in r: print(r); continue
    print(f"{r['workload']:13s} K={r['K']:2d} B={r.get('batch')} res={r.get('resident')} c1={r['chain1']} forced={int(r['forced'])} fill {r['fill_ms']:9.3f} walk {r['walk_ms']:6.3f} gcups {r['gcups_fill']:8.1f}")
PY
done
