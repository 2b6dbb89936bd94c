#!/bin/bash
# GPU job 8: fused ARS rollout at 32 768 environments (one GPU's share of config 4 at N=8): default and forced warp counts
echo hybrid; timeout 300 python tools/bench_callers.py ars --fused --envs-per-gpu 32768 2>&1 | tail -1 | cut -c1-500
for w in 7 6 5 4; do SNK_EXACT_WARPS=$w timeout 300 python tools/bench_callers.py ars --fused --envs-per-gpu 32768 > gpurun_out/ars_w$w.log 2>&1; echo warps $w; tail -1 gpurun_out/ars_w$w.log | cut -c1-400; done
timeout 200 python tools/bench_callers.py ars --envs-per-gpu 32768 > gpurun_out/ars_step.log 2>&1; echo stepwise; tail -1 gpurun_out/ars_step.log | cut -c1-400
