#!/bin/bash
# final tree of round 2 (turned pass at 8 CTAs per SM, gated sweeps with the early exit): full GPU suite, smoke,
# the default bench line
mkdir -p gpurun_out
python -m pytest tests -m gpu -q > gpurun_out/pytest_gpu.log 2>&1; echo "pytest rc=$?"; tail -3 gpurun_out/pytest_gpu.log
python __graft_entry__.py smoke > gpurun_out/smoke.log 2>&1; echo "smoke rc=$?"; tail -1 gpurun_out/smoke.log
python bench.py > gpurun_out/r2t_bench_n1.json 2> gpurun_out/r2t_bench_n1.err; echo "bench rc=$?"
python - <<PY
import json
d = json.load(open('gpurun_out/r2t_bench_n1.json'))
print('cfg2 %.1f Gpx/s (%.4f ms) sustained %.1f kernel %.4f ms frac %.3f e2e %.2f' % (d['value'], d['ms_per_step'], d['sustained']['value'], d['roofline']['kernel_ms'], d['roofline']['frac'], d['e2e']['value']))
for c in d.get('configs') or []:
    print('  %-60s %.1f Gpx/s  %.4f ms  kernel %.4f ms frac %.3f' % (c['workload'][:60], c['value'], c['ms_per_step'], c['roofline']['kernel_ms'], c['roofline']['frac']))
PY
