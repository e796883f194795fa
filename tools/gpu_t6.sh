#!/bin/bash
rm -f gpurun_out/sweep_t6.jsonl
GX_TICKETS=1 python tools/sweep_kr.py --workloads corona6,corona11 --k 4,8 --chain 0 --steps 4 --out sweep_t6.jsonl > /dev/null 2>&1
python - <<'PY'
import json
for l in open('gpurun_out/sweep_t6.jsonl'):
    r = json.loads(l)
    if 'error' in r: print(r); continue
    print(f"{r['workload']:13s} K={r['K']:2d} B={r.get('batch')} res={r.get('resident')} c1={r['chain1']} forced={int(r['forced'])} fill {r['fill_ms']:9.3f} walk {r['walk_ms']:6.3f} gcups {r['gcups_fill']:8.1f}")
PY
