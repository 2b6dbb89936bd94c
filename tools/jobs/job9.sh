#!/bin/bash
# GPU job 9: sticky rollout mode (n <= lanes): tests + ARS fused rollout at 32 768 and 37 888 environments
timeout 600 python -m pytest tests/test_gpu_rollout.py tests/test_gpu_branches.py tests/test_gpu_world_invariance.py -m gpu -q -p no:cacheprovider 2>&1 | tail -4
echo hybrid; timeout 300 python tools/bench_callers.py ars --fused --envs-per-gpu 32768 2>&1 | tail -1 | python -c "import sys,json; d=json.loads(sys.stdin.read()); print(d['env_steps_per_s'], d['ms_per_sweep'], d['ticks_per_env_step'])"
timeout 300 python bench.py --steps 5 --warmup 3 --no-cpu-baseline --no-bullet-order --e2e-steps 2 --envs 131072 > gpurun_out/b9.log 2> gpurun_out/b9.err
python -c "import json;d=json.loads(open('gpurun_out/b9.log').read().strip().splitlines()[-1]);print('bench 131072',round(d['value']),d['config4_ars_sweep'])"
