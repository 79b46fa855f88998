#!/bin/bash
# imx_replay_episode at the final state: the whole GPU suite, smoke(), bench.py and the episode benchmark (one job).
# $1: output directory (default results).
OUT=${1:-results}
mkdir -p "$OUT"
timeout 2400 python -m pytest tests -m gpu -q 2>&1 | tail -15 > "$OUT/r3_tests_gpu.log"
tail -4 "$OUT/r3_tests_gpu.log"
timeout 300 python -c "import __graft_entry__ as g; g.smoke()" 2>&1 | tail -2
timeout 900 python bench.py --gpus 1 --steps 30 --warmup 5 > "$OUT/r3_bench_1gpu.json" 2> "$OUT/r3_bench_1gpu.err"
tail -c 600 "$OUT/r3_bench_1gpu.json"; tail -2 "$OUT/r3_bench_1gpu.err"
timeout 900 python benchmarks/bench_replay_episode.py --out "$OUT/r3_replay_episode.jsonl" > "$OUT/r3_replay_episode.out" 2>&1
python - "$OUT/r3_replay_episode.jsonl" <<'PY'
import json, sys
for l in open(sys.argv[1]):
    d = json.loads(l)
    print(d["workload"], d["outputs"], d["identical_outputs"], d["replay_episode_kernel_variant"],
          round(d["composition"]["ms_per_episode"], 4), round(d["replay_episode"]["ms_per_episode"], 4), round(d["speedup"], 3))
print(d["gpu"], d["power_limit_and_max_sm_clock"])
PY
