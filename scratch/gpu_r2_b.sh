#!/bin/bash
# Round 2, GPU call B: radix-64 column kernel on hardware -- tests, bench, ncu.
cd "$(dirname "$0")/.."
mkdir -p gpurun_out/parity
export SB_PARITY_DIR=gpurun_out/parity
( time timeout 1500 python -m pytest tests -m gpu -q ) > gpurun_out/b_tests.log 2>&1
echo "tests rc=$?" >> gpurun_out/b_tests.log
timeout 600 python bench.py --steps 3 --warmup 3 --no-cpu-baseline > gpurun_out/b_bench_c3_r64.json 2> gpurun_out/b_bench_c3_r64.err
timeout 1200 ncu --set full --clock-control none --import-source on -k regex:'k_conv_cols_r' -s 20 -c 1 \
  -o /tmp/b_prof -f python bench.py --steps 1 --warmup 1 --e2e-steps 1 --no-cpu-baseline --no-dropin > gpurun_out/b_ncu.log 2>&1
ncu -i /tmp/b_prof.ncu-rep --page raw --csv > gpurun_out/b_prof_raw.csv 2>/dev/null
ncu -i /tmp/b_prof.ncu-rep --page source --csv --print-source sass > gpurun_out/b_prof_source.csv 2>/dev/null
gzip -f gpurun_out/b_prof_source.csv
du -sh gpurun_out
tail -8 gpurun_out/b_tests.log
for f in gpurun_out/b_bench_*.json; do echo $f; python -c "
import json,sys
try:
    d=json.loads(open('$f').read().strip().splitlines()[-1]); print(' value %.0f ms %.2f wall %.2f e2e %s' % (d['value'], d['ms_per_step'], d['host_wall_ms_per_step'], (d.get('e2e') or {}).get('value'))); print({k: round(v['ms_per_step'],1) for k,v in d['roofline']['kernels'].items()})
except Exception as e: print(' ??', e)
"; done
