#!/bin/bash
# imx_step_eval on one B200.  $1: output directory (default results); $2: "eval" (the new tests, the closed-loop bookkeeping
# benchmark, the CUDA-graph RL loop example, bench.py and smoke(); default) or "suite" (the rest of the GPU suite).
# Everything writes straight into files under $1 as it runs.
OUT=${1:-results}
mkdir -p "$OUT"
nvidia-smi --query-gpu=name,power.limit,clocks.max.sm --format=csv,noheader | tee "$OUT/r3_card.txt"
if [ "${2:-eval}" = "suite" ]; then
    timeout 560 python -m pytest tests -m gpu -q -p no:cacheprovider --deselect tests/test_gpu_step_eval.py > "$OUT/r3_tests_gpu.log" 2>&1
    tail -8 "$OUT/r3_tests_gpu.log"
    exit 0
fi
timeout 300 python -m pytest tests/test_gpu_step_eval.py -q -p no:cacheprovider > "$OUT/r3_tests_step_eval.log" 2>&1
tail -6 "$OUT/r3_tests_step_eval.log"
timeout 600 python benchmarks/bench_step_eval.py ${BENCH_ARGS} --out "$OUT/r3_step_eval.jsonl" > "$OUT/r3_step_eval.out" 2>&1
python - "$OUT/r3_step_eval.jsonl" <<'PY'
import json, sys
for l in open(sys.argv[1]):
    d = json.loads(l)
    print(d["workload"], d["io"], d["identical_outputs"], d["kernel_variant"]["b"], d["kernel_variant"]["b_ret"],
          *[round(d[a]["us_per_period"], 2) for a in ("a", "b", "a_ret", "b_ret", "c")], d["b_le_a"], d["b_ret_le_a_ret"],
          round(d["bookkeeping_us_per_period"], 3))
print(d["gpu"], d["power_limit_and_max_sm_clock"])
PY
timeout 300 python examples/rl_loop_cuda_graph.py > "$OUT/r3_rl_loop_example.json" 2>&1; tail -1 "$OUT/r3_rl_loop_example.json"
timeout 600 python bench.py --gpus 1 --steps 30 --warmup 5 > "$OUT/r3_bench_1gpu.json" 2> "$OUT/r3_bench_1gpu.err"
head -c 200 "$OUT/r3_bench_1gpu.json"; echo
timeout 300 python -c "import __graft_entry__ as g; g.smoke()" > "$OUT/r3_smoke.log" 2>&1; tail -1 "$OUT/r3_smoke.log"
