#!/bin/bash
# ncu passes of the bench command (B200_PROFILING.md): launch list + full capture of the step kernel, written to $OUT
# (default profile_out/), where scripts/ncu_summarize.py reads them.
export OMP_NUM_THREADS=1 PYTHONUNBUFFERED=1
OUT=${OUT:-profile_out}
mkdir -p "$OUT"
CFG=${CFG:-c3}
timeout 300 ncu --metrics gpu__time_duration.sum --clock-control none -s 30 -c 200 --csv --log-file "$OUT/launches_${CFG}.csv" \
    python bench.py --config $CFG --steps 150 --warmup 8 --no-graph --no-cpu-baseline --no-extras --e2e-steps 10 > "$OUT/ncu_launch_${CFG}.log" 2>&1
timeout 400 ncu --set full --clock-control none --import-source on -k regex:qs_step_kernel -s 20 -c 2 -f -o "$OUT/prof_${CFG}" \
    python bench.py --config $CFG --steps 40 --warmup 8 --no-graph --no-cpu-baseline --no-extras --e2e-steps 10 > "$OUT/ncu_full_${CFG}.log" 2>&1
ls -la "$OUT"
