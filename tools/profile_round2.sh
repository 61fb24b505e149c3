#!/bin/bash
# Round-2 profile evidence, one gpurun call (B200 x1):  bash tools/profile_round2.sh
# 1. launch list of the bench command (cold-cache, serialised: compare SHARES with bench.py's stage_ms, not absolutes)
# 2. ncu --set full of the sketch+lookup pair on a 4 M-read batch (176 MB of input > the 126 MB L2) WITHOUT ncu's cache
#    flush between replays, so the DRAM traffic is what a real step sees (the resolve kernel finds the queue in L2)
# 3. the same pair on 1 M reads, once without and once with ncu's cache flush (the round-1 way), for comparison
# 4. compute-sanitizer memcheck / racecheck on the test subsets that cover every kernel family
set -x
mkdir -p gpurun_out
ncu --metrics gpu__time_duration.sum --clock-control none --kernel-name-base demangled -k regex:'drprg::' -c 400 --csv --log-file gpurun_out/r2_launches_final.csv \
    python bench.py --steps 2 --warmup 3 --no-extras --no-cpu-baseline > gpurun_out/r2_launches_final.bench 2>&1
DRPRG_SCREEN=1 ncu --set full --import-source on --clock-control none --cache-control none \
    -k regex:'screen_kernel|resolve_kernel' --launch-skip 10 -c 2 -f -o gpurun_out/r2_screen4m \
    python tools/screen_bench.py run 4000000 > gpurun_out/r2_screen4m.log 2>&1
ncu -i gpurun_out/r2_screen4m.ncu-rep --page raw --csv > gpurun_out/r2_screen4m_raw.csv 2>/dev/null
DRPRG_SCREEN=1 ncu --set full --clock-control none --cache-control none \
    -k regex:'screen_kernel|resolve_kernel' --launch-skip 10 -c 2 -f -o gpurun_out/r2_screen1m_nc \
    python tools/screen_bench.py run 1000000 > gpurun_out/r2_screen1m_nc.log 2>&1
ncu -i gpurun_out/r2_screen1m_nc.ncu-rep --page raw --csv > gpurun_out/r2_screen1m_nc_raw.csv 2>/dev/null
DRPRG_SCREEN=1 ncu --set full --clock-control none \
    -k regex:'screen_kernel|resolve_kernel' --launch-skip 10 -c 2 -f -o gpurun_out/r2_screen1m \
    python tools/screen_bench.py run 1000000 > gpurun_out/r2_screen1m.log 2>&1
ncu -i gpurun_out/r2_screen1m.ncu-rep --page raw --csv > gpurun_out/r2_screen1m_raw.csv 2>/dev/null
compute-sanitizer --tool memcheck python -m pytest tests/test_gpu_parity.py -m gpu -x -q \
    -k "toy_config1 or device_fastq_ingest_matches or low_min_cluster or drop_in_call" > gpurun_out/r2_memcheck.log 2>&1
compute-sanitizer --tool racecheck python -m pytest tests/test_gpu_parity.py -m gpu -x -q \
    -k "toy_config1 or low_min_cluster" > gpurun_out/r2_racecheck.log 2>&1
tail -n 4 gpurun_out/r2_memcheck.log; tail -n 4 gpurun_out/r2_racecheck.log
