#!/bin/bash
# Everything profiles/ is built from, in one GPU-box call:   gpurun --timeout 1500 -- 'bash tools/profile_round.sh r02'
# then here:   python tools/summarize_profiles.py r02 4500
#   1. the bench line and the reference arm (never under a profiler)
#   2. ncu launch list of one bench step (per-launch durations -> kernel shares)
#   3. ncu --set full of one launch of each hot kernel on a 4500-pair chunk
#   4. one short bench line per BASELINE config, the head-size sweep
TAG=${1:-r02}
PAIRS=${PAIRS:-4500}
cd "$(dirname "$0")/.."
mkdir -p gpurun_out
python bench.py > gpurun_out/${TAG}_bench.json 2> gpurun_out/${TAG}_bench.err
python bench.py --impl reference > gpurun_out/${TAG}_bench_reference.json 2> gpurun_out/${TAG}_bench_reference.err
ncu --metrics gpu__time_duration.sum --clock-control none --csv --log-file gpurun_out/${TAG}_launches.csv \
    python bench.py --steps 1 --warmup 1 --no-cpu-baseline > gpurun_out/${TAG}_launches.log 2>&1
cap() {  # name kernel-regex skip
  ncu --set full --clock-control none --import-source on -k regex:$2 -s $3 -c 1 -f -o gpurun_out/${TAG}_$1 \
      python bench.py --no-cpu-baseline --steps 1 --warmup 0 --pairs $PAIRS > gpurun_out/${TAG}_$1.log 2>&1
}
cap tc tc_count_kernel 1      # launch 0 is the mid stage, 1 the bulk first pass
cap bound bound_kernel 1   # launch 0 is the mid stage
cap lm lm_warp_kernel 0
cap score_survivors score_kernel 1
cap solve solve2_kernel 0
bash tools/all_configs_bench.sh > gpurun_out/${TAG}_all_configs.txt 2>&1
ls -la gpurun_out | head -40
