#!/bin/bash
# Per-period records of imx_replay_episode_records: the records tests, then the benchmark (one job).
# $1: output directory (default results); the benchmark's lines go to $1/r3_replay_records.jsonl (profiles/ keeps a copy).
OUT=${1:-results}
mkdir -p "$OUT"
nvidia-smi --query-gpu=name,power.limit,clocks.max.sm --format=csv,noheader
timeout 1500 python -u -m pytest tests/test_gpu_replay_records.py -m gpu -q > "$OUT/r3_tests_replay_records.log" 2>&1
tail -5 "$OUT/r3_tests_replay_records.log"
timeout 1200 python -u benchmarks/bench_replay_records.py --out "$OUT/r3_replay_records.jsonl" > "$OUT/r3_replay_records.out" 2>&1
tail -3 "$OUT/r3_replay_records.out"
python - "$OUT/r3_replay_records.jsonl" <<'PY'
import json, sys
for l in open(sys.argv[1]):
    d = json.loads(l)
    arms = ("composition", "records", "records_composed", "no_records")
    print(d["workload"], "obs" if d["observations"] else "noobs", d["identical_outputs"], d["kernel_variant"],
          " ".join(f"{a}={d[a]['us_per_episode']:.1f}" for a in arms))
print(d["gpu"], d["power_limit_and_max_sm_clock"], round(d["hbm_copy_peak_GB_per_s"]))
PY
