#!/bin/bash
for band in 0 ""; do
  echo "== GX_CODE_BAND=${band:-default}"
  if [ -n "$band" ]; then export GX_CODE_BAND=$band; else unset GX_CODE_BAND; fi
  python tools/mode_probe.py brca2 | grep "local=0 traceback=1"
  python tools/mode_probe.py corona1 | grep "local=0 traceback=1"
  rm -f gpurun_out/sweep_band.jsonl
  python tools/sweep_kr.py --workloads corona6,corona11,corona23 --k 4,8 --chain 0 --steps 4 --out sweep_band.jsonl > /dev/null 2>&1
  python - <<'PY'
import json
for l in open('gpurun_out/sweep_band.jsonl'):
    r = json.loads(l)
    if 'error' in r: print(r); continue
    print(f"{r['workload']:13s} K={r['K']:2d} B={r.get('batch')} res={r.get('resident')} c1={r['chain1']} forced={int(r['forced'])} fill {r['fill_ms']:9.3f} walk {r['walk_ms']:6.3f} gcups {r['gcups_fill']:8.1f}")
PY
done
