#!/bin/bash
# imx_replay_episode: the feature's GPU tests and the episode benchmark (one job).  $1: output directory (default results).
OUT=${1:-results}
mkdir -p "$OUT"
timeout 1500 python -m pytest tests/test_gpu_replay_episode.py -x -q 2>&1 | tail -25 > "$OUT/r3_replay_episode_tests.log"
tail -5 "$OUT/r3_replay_episode_tests.log"
timeout 900 python benchmarks/bench_replay_episode.py --out "$OUT/r3_replay_episode.jsonl" > "$OUT/r3_replay_episode.out" 2>&1
python - "$OUT/r3_replay_episode.jsonl" <<'PY'
import json, sys
for l in open(sys.argv[1]):
    d = json.loads(l)
    print(d["workload"], d["outputs"], d["identical_outputs"], d["replay_episode_kernel_variant"],
          round(d["composition"]["ms_per_episode"], 4), round(d["replay_episode"]["ms_per_episode"], 4), round(d["speedup"], 3))
print(d["gpu"], d["power_limit_and_max_sm_clock"])
PY
tail -3 "$OUT/r3_replay_episode.out"
