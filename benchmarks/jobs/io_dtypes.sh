#!/bin/bash
# bfloat16 observations / float32 actions: build, the new GPU tests, smoke(), the I/O dtype benchmark, bench.py and the rest of
# the GPU suite (one job).  $1: output directory (default results).
OUT=${1:-results}
mkdir -p "$OUT"
python -c "import __graft_entry__ as g; g.build()" > "$OUT/r3_build.log" 2>&1 || { tail -20 "$OUT/r3_build.log"; exit 1; }
timeout 1200 python -m pytest tests/test_gpu_io_dtypes.py -m gpu -q -p no:cacheprovider 2>&1 | tail -60 > "$OUT/r3_tests_io_dtypes.log"
tail -25 "$OUT/r3_tests_io_dtypes.log"
timeout 300 python -c "import __graft_entry__ as g; g.smoke()" 2>&1 | tail -2
timeout 1200 python benchmarks/bench_io_dtypes.py --out "$OUT/r3_io_dtypes.jsonl" > "$OUT/r3_io_dtypes.out" 2>&1
tail -3 "$OUT/r3_io_dtypes.out"
python - "$OUT/r3_io_dtypes.jsonl" <<'PY'
import json, sys
for l in open(sys.argv[1]):
    d = json.loads(l)
    t = next(d[k] for k in ("us_per_launch", "us_per_call", "us_per_episode", "us_per_step", "us_per_period") if k in d)
    print(d["measurement"], d["workload"], d.get("obs_dtype", d.get("variant")), d.get("action_dtype", ""), d.get("zero_copy", ""),
          round(t, 2), d.get("identical_outputs", ""), round(d.get("copy_peak_fraction", 0), 3))
print(d["gpu"], d["power_limit_and_max_sm_clock"])
PY
timeout 900 python bench.py --gpus 1 --steps 30 --warmup 5 > "$OUT/r3_bench_1gpu.json" 2> "$OUT/r3_bench_1gpu.err"
tail -c 300 "$OUT/r3_bench_1gpu.json"; tail -2 "$OUT/r3_bench_1gpu.err"
timeout 1500 python -m pytest tests -m gpu -q -p no:cacheprovider --ignore=tests/test_gpu_io_dtypes.py 2>&1 | tail -25 > "$OUT/r3_tests_gpu.log"
tail -8 "$OUT/r3_tests_gpu.log"
# a fault the runtime reports fails the job even where the failing step's exit code was swallowed by a pipe
if grep -l "illegal memory access\|CUDA error" "$OUT"/*; then exit 1; fi
