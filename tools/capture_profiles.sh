#!/bin/bash
# Round evidence in ONE gpurun call (every profiled command first runs to completion without ncu):
#   tools/capture_profiles.sh r02      -> gpurun_out/prof_<tag>_*.ncu-rep, launches_<tag>_*.csv, bench_<tag>_*.json
tag=${1:-r02}
out=gpurun_out
set -x
python bench.py --steps 20 > $out/bench_${tag}_n1.json 2> $out/bench_${tag}_n1.err || exit 1
python bench.py --impl reference --steps 5 --warmup 1 > $out/bench_${tag}_reference_arm.json 2>/dev/null
python bench.py --steps 3 --warmup 3 --no-extras > /dev/null 2>&1 && \
ncu --metrics gpu__time_duration.sum --clock-control none --nvtx --nvtx-include "timed/" --csv --log-file $out/launches_${tag}_timed_region.csv \
    python bench.py --steps 3 --warmup 3 --no-extras > /dev/null 2>&1
python tools/run_features.py 600 > /dev/null 2>&1 && \
ncu --metrics gpu__time_duration.sum --clock-control none --nvtx --nvtx-include "features/" --csv --log-file $out/launches_${tag}_features_1h.csv \
    python tools/run_features.py 600 > /dev/null 2>&1
ncu --set full --clock-control none --import-source on -k regex:extract_kernel -s 3 -c 1 -o $out/prof_${tag}_800 -f python bench.py --steps 2 --warmup 3 --no-extras > /dev/null 2>&1
ncu --set full --clock-control none --import-source on -k regex:extract_kernel -s 3 -c 1 -o $out/prof_${tag}_1600 -f python bench.py --steps 2 --warmup 3 --no-extras --n-fft 1600 > /dev/null 2>&1
ncu --set full --clock-control none --import-source on -k regex:"extract_kernel|mfcc_dct" -s 2 -c 2 -o $out/prof_${tag}_mfcc -f python tools/time_features.py mfcc > /dev/null 2>&1
ls -la $out/*${tag}*
