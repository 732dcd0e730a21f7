#!/bin/bash
# One GPU-box session. Usage (repo root, under gpurun):  bash tools/gpu_round.sh <tag> [steps...]
#   steps: test bench sweep launches ncu configs reference latency   (default: test bench sweep launches ncu)
TAG=${1:-r01}; shift
STEPS=${@:-test bench sweep launches ncu}
OUT=gpurun_out/$TAG
mkdir -p $OUT
nvidia-smi --query-gpu=name,clocks.sm,clocks.max.sm,power.draw --format=csv > $OUT/smi.txt 2>&1
nproc > $OUT/nproc.txt; grep -m1 'model name' /proc/cpuinfo >> $OUT/nproc.txt
for s in $STEPS; do case $s in
test) echo "== pytest gpu"; timeout 900 python -m pytest tests -m gpu -x -q 2>&1 | tail -15 | tee $OUT/pytest_gpu.txt;;
bench) echo "== bench"; timeout 900 python bench.py --steps 10 --warmup 3 > $OUT/bench.json 2> $OUT/bench.err; tail -c 3000 $OUT/bench.json; tail -5 $OUT/bench.err;;
sweep) echo "== sweep"; timeout 600 python tools/sweep.py --frames 1024 --chunks ${SWEEP_CHUNKS:-32,256} --reps 5 2>&1 | tee $OUT/sweep.jsonl;;
launches) echo "== ncu launches"; timeout 600 ncu --metrics gpu__time_duration.sum --clock-control none -c 400 --csv --log-file $OUT/launches.csv \
   python bench.py --steps 2 --warmup 3 --frames 512 --e2e-frames 16 --no-cpu-baseline --no-latency --parity-frames 0 > $OUT/bench_under_ncu.log 2>&1; grep -c k_ $OUT/launches.csv;;
ncu) echo "== ncu full"; timeout 900 ncu --set full --clock-control none --import-source on -k "regex:${NCU_KERNELS:-k_transform_bin|k_label_bev|k_quad_reduce|k_outline}" -s ${NCU_SKIP:-8} -c ${NCU_COUNT:-4} \
   -o $OUT/prof python bench.py --steps 1 --warmup 3 --frames 512 --e2e-frames 16 --no-cpu-baseline --no-latency --parity-frames 0 > $OUT/ncu_full.log 2>&1; tail -3 $OUT/ncu_full.log | cut -c1-300;;
configs) echo "== configs"; for c in 0 1 3 4; do timeout 600 python bench.py --config $c --steps 5 --warmup 3 --no-cpu-baseline > $OUT/bench_config$c.json 2> $OUT/bench_config$c.err; tail -c 300 $OUT/bench_config$c.json; echo; done;;
reference) echo "== reference arm"; timeout 600 python bench.py --impl reference --steps 3 --warmup 1 > $OUT/bench_reference.json 2> $OUT/bench_reference.err; tail -c 400 $OUT/bench_reference.json;;
latency) echo "== latency"; (python tools/latency.py; python tools/latency.py --w 640 --h 480) | tee $OUT/latency.jsonl;;
esac; done
ls -la $OUT
