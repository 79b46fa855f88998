#!/bin/bash
mkdir -p gpurun_out
timeout 900 python -m pytest tests/test_gpu_rollout_et.py tests/test_gpu_rollout.py tests/test_gpu_dfo_div.py tests/test_gpu_full_size.py -x -q 2>&1 | tail -25 > gpurun_out/r2_t5_tests.log
tail -3 gpurun_out/r2_t5_tests.log
for et in 0 1; do
  IMX_ROLLOUT_ET=$et timeout 300 python benchmarks/bench_configs.py --only rollout > gpurun_out/r2_rollouts_et$et.jsonl 2> gpurun_out/r2_rollouts_et$et.err
done
cat gpurun_out/r2_rollouts_et1.jsonl | cut -c1-200
# step kernel policy sweep: pipe on/off at large N, CTA sizes
timeout 600 python benchmarks/pipe_sweep.py --configs serial4 --envs 524288,1048576,4194304 --threads 128,256 --stages 4 --ctas 2,4 --reps 8 > gpurun_out/r2_pipe_sweep_large.jsonl 2> gpurun_out/r2_pipe_sweep_large.err
timeout 600 python benchmarks/pipe_sweep.py --configs serial8,serial2 --envs 65536,262144,1048576 --threads 64,128 --stages 3,4 --ctas 4,6,8 --reps 10 > gpurun_out/r2_pipe_sweep_s8s2.jsonl 2> gpurun_out/r2_pipe_sweep_s8s2.err
