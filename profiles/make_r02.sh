#!/bin/bash
# Round-2 measurement recipe (run on the B200 box through gpurun from the repo root):
#   the default bench line, the launch list of a short bench command (ncu gpu__time_duration: cold-cache, serialised --
#   compare shares), one full capture of single-step launches (defender + attacker turn), one of a fused launch, the
#   per-type exclusion sweep
mkdir -p gpurun_out
python bench.py > gpurun_out/r02_bench.json 2> gpurun_out/r02_bench.err
python bench.py --steps 24 --warmup 4 --no-cpu-baseline --no-e2e --no-legs > gpurun_out/r02_plain.log 2>&1 && \
ncu --metrics gpu__time_duration.sum --clock-control none -k regex:cyg_ -c 80 --csv --log-file gpurun_out/r02_launches.csv \
    python bench.py --steps 24 --warmup 4 --no-cpu-baseline --no-e2e --no-legs > gpurun_out/r02_ncu_list.log 2>&1
python bench.py --fuse 1 --steps 9 --warmup 3 --no-cpu-baseline --no-e2e --no-legs > gpurun_out/r02_plain2.log 2>&1 && \
ncu --set full --clock-control none --import-source on -k regex:cyg_step_kernel -s 8 -c 2 -o gpurun_out/r02_step_kernel \
    python bench.py --fuse 1 --steps 9 --warmup 3 --no-cpu-baseline --no-e2e --no-legs > gpurun_out/r02_ncu_full.log 2>&1
ncu --set full --clock-control none -k regex:cyg_step_kernel -s 4 -c 2 -o gpurun_out/r02_step_kernel_fused \
    python bench.py --steps 24 --warmup 4 --no-cpu-baseline --no-e2e --no-legs > gpurun_out/r02_ncu_full_fused.log 2>&1
bash profiles/exclude_sweep.sh gpurun_out/r02_exclude_sweep.txt > /dev/null 2>&1
tail -1 gpurun_out/r02_bench.json | cut -c1-300
