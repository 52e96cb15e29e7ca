#!/bin/bash
# The measurements kept under profiles/ for a round: bench lines (engine + reference arm, cfg3 / cfg1 / cfg2), the launch
# list of a short bench run, full ncu captures of the fused pipeline's kernels and of the ifit kernel.
#   tools/final_profiles.sh r02f
tag=${1:-r02f}
mkdir -p gpurun_out
python bench.py --steps 5 --warmup 3 > gpurun_out/${tag}_bench_cfg3.json 2> gpurun_out/${tag}_bench_cfg3.err; echo "bench cfg3 exit $?"
python bench.py --impl reference --steps 5 --warmup 3 > gpurun_out/${tag}_bench_cfg3_reference.json 2> gpurun_out/${tag}_bench_cfg3_reference.err; echo "reference exit $?"
python bench.py --workload cfg1 --steps 5 --warmup 3 > gpurun_out/${tag}_bench_cfg1.json 2> gpurun_out/${tag}_bench_cfg1.err; echo "cfg1 exit $?"
python bench.py --workload cfg2 --steps 5 --warmup 3 > gpurun_out/${tag}_bench_cfg2.json 2> gpurun_out/${tag}_bench_cfg2.err; echo "cfg2 exit $?"
python tools/ifit_phases.py 100000 768 unit > gpurun_out/${tag}_ifit_phases.log 2>&1
python tools/ifit_phases.py 30000 256 whitened >> gpurun_out/${tag}_ifit_phases.log 2>&1
python tools/categorize_time.py >> gpurun_out/${tag}_ifit_phases.log 2>&1
python bench.py --steps 2 --warmup 1 --no-cpu-baseline > gpurun_out/plain.log 2>&1 &&
ncu --metrics gpu__time_duration.sum --clock-control none -c 3000 --csv --log-file gpurun_out/${tag}_launches.csv \
    python bench.py --steps 2 --warmup 1 --no-cpu-baseline > gpurun_out/ncu_launches.log 2>&1
python tools/fused_once.py > gpurun_out/once.log 2>&1 &&
ncu --set full --import-source on --clock-control none -k regex:"h_score_kernel|fn_|hq_build|small_scores|paths_small" -s 12 -c 10 \
    -o gpurun_out/${tag}_fused python tools/fused_once.py > gpurun_out/ncu_full.log 2>&1
tail -2 gpurun_out/ncu_full.log
python tools/ifit_small.py 3000 768 unit > gpurun_out/ifit_small.log 2>&1 &&
ncu --set full --import-source on --clock-control none -k regex:ifit_kernel -c 1 -o gpurun_out/${tag}_ifit python tools/ifit_small.py 3000 768 unit > gpurun_out/ncu_ifit.log 2>&1
tail -2 gpurun_out/ncu_ifit.log
