#!/bin/bash
# Prioritized against uniform replay: learning runs in the r02f setting of profiles/sac2_learning.md (experiment 6,
# 8192 envs, a 33,554,432-slot ring, 2 updates per iteration, 40,000 iterations, fp32 learner) for one algorithm,
# seeds 0-2, each with and without --prioritized (default priority parameters); the six runs share the GPU.
OUT="${1:?usage: $0 OUTPUT_DIR ALGORITHM}"   # logs, JSON results and experiment trees go here
ALGO="${2:?usage: $0 OUTPUT_DIR ALGORITHM}"  # sac1 or sac2
mkdir -p "$OUT"
run() {  # name, extra flags
  timeout 560 python examples/train_sac.py --envs 8192 --iters 40000 --warmup-iters 20 --updates-per-iter 2 \
    --experiment 6 --buffer 33554432 --log-every 1000 --algorithm "$ALGO" \
    --experiments-root "$OUT/per_learning/$1" "${@:2}" > "$OUT/per_learning_$1.log" 2>&1
}
for s in 0 1 2; do
  run ${ALGO}_uniform_s$s --seed $s &
  run ${ALGO}_per_s$s --seed $s --prioritized &
done
wait
for f in "$OUT"/per_learning_${ALGO}_*.log; do echo "== $f"; tail -n 1 "$f" | cut -c1-600; done
