#!/bin/bash
# walk kernel iteration: traceback parity tests first (short timeout: the walk has spin loops), then the full GPU suite and the wavefront workloads
mkdir -p gpurun_out
timeout 300 python -m pytest tests -m gpu -x -q -k "traceback or band or walk or golden or local" 2>&1 | tail -4 | tee gpurun_out/pytest_walk.log
timeout 900 python -m pytest tests -m gpu -x -q 2>&1 | tail -4 | tee gpurun_out/pytest_gpu.log
for w in corona45 brca2_global brca2_local; do
  timeout 300 python bench.py --workload $w --steps 20 --warmup 5 --no-cpu-baseline --no-k0 > gpurun_out/bench_walk_$w.json 2> gpurun_out/bench_walk_$w.err
  python tools/show_bench.py gpurun_out/bench_walk_$w.json | head -2
done
