#!/bin/bash
# SAC-v2: the checkpoint and fp32-graph tests, then the learning comparison in the r02f setting (experiment 6, 8192
# envs, a 33,554,432-slot ring, 2 updates per iteration, 40,000 iterations): v1 and v2 (fp32 learner) for seeds 0-2
# and v2 with the tcgen05 learner; the seven runs share the GPU
OUT="${1:?usage: $0 OUTPUT_DIR}"   # logs, JSON results and experiment trees go here
mkdir -p "$OUT"
timeout 600 python -m pytest tests/test_sac2.py -m gpu -q -s -rA -k "checkpoint or fp32_graph" > $OUT/sac2_gpu_tests_b.log 2>&1
grep -E "worst|passed|failed|Error" $OUT/sac2_gpu_tests_b.log | tail -n 8
run() {  # name, extra flags
  timeout 1500 python examples/train_sac.py --envs 8192 --iters 40000 --warmup-iters 20 --updates-per-iter 2 \
    --experiment 6 --buffer 33554432 --log-every 1000 --experiments-root $OUT/sac2_learning/$1 "${@:2}" \
    > $OUT/sac2_learning_$1.log 2>&1
}
for s in 0 1 2; do
  run v1_s$s --seed $s &
  run v2_s$s --seed $s --algorithm sac2 &
done
run v2tc_s0 --seed 0 --algorithm sac2 --learner-precision tcgen05 &
wait
for f in $OUT/sac2_learning_*.log; do echo "== $f"; tail -n 1 $f | cut -c1-400; done
