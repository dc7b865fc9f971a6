#!/bin/bash
# SAC-v2: build + smoke, the new GPU tests, the per-update and population timings, the driver, the benchmark, the
# whole GPU suite
OUT="${1:?usage: $0 OUTPUT_DIR}"   # logs, JSON results and experiment trees go here
mkdir -p "$OUT"
python -c "import __graft_entry__ as g; g.build(); g.smoke()" > $OUT/build_smoke.log 2>&1
tail -n 3 $OUT/build_smoke.log
timeout 1200 python -m pytest tests/test_sac2.py -m gpu -q -s -rA > $OUT/sac2_gpu_tests.log 2>&1
grep -E "worst|passed|failed|Error" $OUT/sac2_gpu_tests.log | tail -n 25
timeout 600 python profiles/sac2_eval.py --out $OUT/sac2_eval.json > $OUT/sac2_eval.log 2>&1
tail -n 14 $OUT/sac2_eval.log
for alg in sac2 sac1; do
  timeout 300 python examples/train_sac.py --envs 8192 --policy-precision tcgen05 --collect-steps 8 --updates-per-iter 8 \
    --learner-precision tcgen05 --algorithm $alg --iters 200 > $OUT/example_$alg.log 2>&1
  tail -n 1 $OUT/example_$alg.log | cut -c1-600
done
timeout 300 python bench.py --gpus 1 --steps 200 --warmup 20 > $OUT/bench.json 2> $OUT/bench.err
tail -c 600 $OUT/bench.json
timeout 2400 python -m pytest tests -m gpu -q --deselect tests/test_sac2.py > $OUT/gpu_suite.log 2>&1
tail -n 15 $OUT/gpu_suite.log
