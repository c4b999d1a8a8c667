#!/bin/bash
# round-2 GPU session 1: sanity, pipe microbenchmarks, phase timeline, host-path ceiling
cd "${GRAFT_REPO_ROOT:-.}"
O=gpurun_out
timeout 300 python -m pytest tests -m gpu -x -q 2>&1 | tail -3 > $O/r2_pytest1.log
timeout 120 tools/microbench/xu_bench > $O/r2_xu_bench.txt 2>&1
timeout 60 tools/microbench/trace_bench > $O/r2_trace.txt 2>&1
timeout 120 python tools/host_path_ceiling.py > $O/r2_host_ceiling_n1.json 2>&1
timeout 120 python tools/host_path_ceiling.py --bytes-per-sample 2 >> $O/r2_host_ceiling_n1.json 2>&1
timeout 300 python bench.py --steps 20 --warmup 3 > $O/r2_bench1.json 2> $O/r2_bench1.err
echo done
