#!/bin/bash
# Round 2, GPU call A: full GPU test-suite (BASELINE configs with bounded tolerances), the bench
# line, the other single-GPU configs with per-kernel times, ncu launch list + full capture of the
# real C3 batch, north-star / C5 on one GPU.  Keeps gpurun_out/ small (ncu reports -> csv).
cd "$(dirname "$0")/.."
mkdir -p gpurun_out/parity
export SB_PARITY_DIR=gpurun_out/parity
nvidia-smi --query-gpu=name,clocks.sm,clocks.max.sm,power.draw --format=csv > gpurun_out/a_smi.txt 2>&1
( time timeout 1500 python -m pytest tests -m gpu -q ) > gpurun_out/a_tests.log 2>&1
echo "tests rc=$?" >> gpurun_out/a_tests.log
timeout 300 python scratch/fft_bench.py > gpurun_out/a_fft_bench.json 2> gpurun_out/a_fft_bench.err
timeout 600 python bench.py --steps 3 --warmup 3 > gpurun_out/a_bench_c3.json 2> gpurun_out/a_bench_c3.err
for w in c1 c2 c4; do
  timeout 600 python bench.py --workload $w --steps 5 --warmup 3 --no-cpu-baseline > gpurun_out/a_bench_$w.json 2> gpurun_out/a_bench_$w.err
done
timeout 900 python bench.py --workload ns --steps 1 --warmup 1 --no-cpu-baseline > gpurun_out/a_bench_ns_1gpu.json 2> gpurun_out/a_bench_ns_1gpu.err
timeout 600 python bench.py --workload c5 --ages 1 --steps 1 --warmup 1 --no-cpu-baseline > gpurun_out/a_bench_c5_1age_1gpu.json 2> gpurun_out/a_bench_c5_1age_1gpu.err
# launch list of one bench step (cold-cache, serialised: shares only)
timeout 900 ncu --metrics gpu__time_duration.sum --clock-control none --csv --log-file gpurun_out/a_launches.csv \
  python bench.py --steps 1 --warmup 1 --e2e-steps 1 --no-cpu-baseline --no-dropin > gpurun_out/a_launch_run.log 2>&1
# full capture of the dominant kernels at the real C3 batch (60 templates = 2 angles x 30 ages)
timeout 1200 ncu --set full --clock-control none --import-source on -k regex:'k_conv_cols_p|k_fit_rows_g' -s 20 -c 2 \
  -o /tmp/a_prof -f python bench.py --steps 1 --warmup 1 --e2e-steps 1 --no-cpu-baseline --no-dropin > gpurun_out/a_ncu.log 2>&1
ncu -i /tmp/a_prof.ncu-rep --page raw --csv > gpurun_out/a_prof_raw.csv 2>/dev/null
ncu -i /tmp/a_prof.ncu-rep --page source --csv --print-source sass > gpurun_out/a_prof_source.csv 2>/dev/null
gzip -f gpurun_out/a_prof_source.csv
timeout 600 ncu --set full --clock-control none -k regex:'k_curv_cols|k_tmpl_rows|k_conv_cols_f|k_fit_rows_g' -s 10 -c 5 \
  -o /tmp/a_prof_c1 -f python bench.py --workload c1 --steps 1 --warmup 1 --e2e-steps 1 --no-cpu-baseline --no-dropin > gpurun_out/a_ncu_c1.log 2>&1
ncu -i /tmp/a_prof_c1.ncu-rep --page raw --csv > gpurun_out/a_prof_c1_raw.csv 2>/dev/null
du -sh gpurun_out
tail -15 gpurun_out/a_tests.log
for f in gpurun_out/a_bench_*.json; do echo $f; python -c "
import json,sys
try:
    d=json.loads(open('$f').read().strip().splitlines()[-1]); print(' value %.0f ms %.2f e2e %s' % (d['value'], d['ms_per_step'], (d.get('e2e') or {}).get('value')))
except Exception as e: print(' ??', e)
"; done
cat gpurun_out/a_fft_bench.json
