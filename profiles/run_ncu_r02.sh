#!/bin/bash
# ncu captures of round 2 (run under gpurun from the repo root): full-set capture of each kernel, raw metrics + source
# page exported to CSV (the .ncu-rep files stay on the box except the two headline ones), and the launch list of the bench.
set -u
mkdir -p gpurun_out/ncu
cap() {   # name, kernel regex, target, skip
  ncu --set full --clock-control none --import-source on -k "regex:$2" -s "$4" -c 1 -f -o gpurun_out/ncu/$1 \
      python profiles/prof_targets.py $3 > gpurun_out/ncu/$1.log 2>&1
  ncu -i gpurun_out/ncu/$1.ncu-rep --page raw --csv > gpurun_out/ncu/$1_raw.csv 2>/dev/null
  ncu -i gpurun_out/ncu/$1.ncu-rep --page details --csv > gpurun_out/ncu/$1_details.csv 2>/dev/null
  ncu -i gpurun_out/ncu/$1.ncu-rep --page source --csv > gpurun_out/ncu/$1_source.csv 2>/dev/null
  if [ "${5:-}" != "keep" ]; then rm -f gpurun_out/ncu/$1.ncu-rep; fi
}
cap r02_step_e100k k_group_step_e step_e100k 2
cap r02_step_e500k k_group_step_e step_e500k 2 keep
cap r02_step_e5m   k_group_step_e step_e5m 2
cap r02_eval_d128 k_eval_tiled eval_d128 1 keep
cap r02_rows_update k_rows_update opt 2
cap r02_rows_sqnorm k_rows_sqnorm opt 2
cap r02_step_dense k_group_step_e opt 2
cap r02_transr_project k_transr_project transr_eval 2
cap r02_rec_tile k_rec_tile tup_step 2
cap r02_eval_gumbel "k_eval<" gumbel_eval 1
ncu --metrics gpu__time_duration.sum --clock-control none -c 1500 --csv --log-file gpurun_out/ncu/launches_r02_bench.csv \
    python bench.py --steps 2 --warmup 3 --launches-per-step 4 --no-cpu-baseline > gpurun_out/ncu/bench_under_ncu.log 2>&1
ls -la gpurun_out/ncu | head -60
