#!/bin/bash
# round-2 multi-GPU runs on one box of G GPUs: correctness check, then the three BASELINE.json multi-GPU configs.
# usage: bash scripts/gpu_8gpu_r2.sh G [OUT]   (logs and JSON lines go to OUT, default a new temporary directory)
G=${1:-8}
OUT=${2:-$(mktemp -d)}
mkdir -p "$OUT"
echo "output in $OUT"
TR="python -m torch.distributed.run --nnodes=1 --nproc-per-node=$G --master-addr 127.0.0.1"
timeout 240 $TR --master-port 29611 scripts/multi_gpu_check.py > $OUT/r2_multi_check_${G}gpu.log 2>&1
tail -3 $OUT/r2_multi_check_${G}gpu.log
timeout 420 $TR --master-port 29612 bench.py --gpus $G --steps 2 --warmup 2 > $OUT/r2_bench_C_${G}gpu.json 2> $OUT/r2_bench_C_${G}gpu.err
grep "warmup\|Error\|error" $OUT/r2_bench_C_${G}gpu.err | tail -6; head -c 300 $OUT/r2_bench_C_${G}gpu.json; echo
timeout 420 $TR --master-port 29613 bench.py --gpus $G --workload E --steps 1 --warmup 1 --e2e-steps 0 > $OUT/r2_bench_E_${G}gpu.json 2> $OUT/r2_bench_E_${G}gpu.err
grep "warmup\|Error\|error" $OUT/r2_bench_E_${G}gpu.err | tail -4; head -c 300 $OUT/r2_bench_E_${G}gpu.json; echo
timeout 600 $TR --master-port 29614 bench.py --gpus $G --workload D --steps 1 --warmup 1 > $OUT/r2_bench_D_${G}gpu.json 2> $OUT/r2_bench_D_${G}gpu.err
grep "warmup\|counts\|Error\|error" $OUT/r2_bench_D_${G}gpu.err | tail -6; head -c 300 $OUT/r2_bench_D_${G}gpu.json; echo
nvidia-smi --query-gpu=index,memory.used,memory.total --format=csv | head -3
