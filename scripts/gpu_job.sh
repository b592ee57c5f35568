#!/bin/bash
# usage: scripts/gpu_job.sh TAG  -- GPU test suite, bench, optional microbenchmark / ncu captures into gpurun_out/TAG_*
T=$1
mkdir -p gpurun_out
if [ -z "$NO_TESTS" ]; then timeout 1200 python -m pytest tests -m gpu -q ${PYTEST_FLAGS} > gpurun_out/${T}_gputests.log 2>&1; echo "pytest rc=$?" >> gpurun_out/${T}_gputests.log; tail -8 gpurun_out/${T}_gputests.log; fi
if [ -z "$NO_BENCH" ]; then timeout 900 python bench.py ${BENCH_FLAGS:---steps 5 --warmup 3} > gpurun_out/${T}_bench.log 2> gpurun_out/${T}_bench.err; echo "bench rc=$?"; tail -1 gpurun_out/${T}_bench.log | cut -c1-3000; tail -5 gpurun_out/${T}_bench.err; fi
if [ -x scripts/microbench/pipes ] && [ -n "$PIPES" ]; then timeout 60 ./scripts/microbench/pipes > gpurun_out/${T}_pipes.txt 2>&1; fi
if [ -n "$NCU_NTT" ]; then timeout 300 ncu --set full --clock-control none --import-source on -k regex:ntt_tile_kernel -s 3 -c 3 -o gpurun_out/${T}_ntt -f python scripts/prof_kernels.py ntt > gpurun_out/${T}_ncu_ntt.log 2>&1; fi
if [ -n "$NCU_MSM" ]; then timeout 300 ncu --set full --clock-control none --import-source on -k regex:"msm_acc_chunk|msm_wsum_level|msm_acc_levelN|msm_digits" -s 8 -c 8 -o gpurun_out/${T}_msm -f python scripts/prof_kernels.py msm > gpurun_out/${T}_ncu_msm.log 2>&1; fi
if [ -n "$MULTI" ]; then timeout ${MULTI_TIMEOUT:-300} python -m torch.distributed.run --nnodes=1 --nproc-per-node $MULTI --master-addr 127.0.0.1 --master-port 29517 scripts/multi_gpu_check.py ${MULTI_ARGS} > gpurun_out/${T}_multi.log 2>&1; echo "multi rc=$?"; tail -3 gpurun_out/${T}_multi.log | cut -c1-2500; fi
if [ -n "$MULTI_BENCH" ]; then ZKB_TRACE=${ZKB_TRACE} timeout ${MBENCH_TIMEOUT:-600} python -m torch.distributed.run --nnodes=1 --nproc-per-node $MULTI_BENCH --master-addr 127.0.0.1 --master-port 29519 bench.py --gpus $MULTI_BENCH --steps 3 --warmup 3 > gpurun_out/${T}_mbench.log 2> gpurun_out/${T}_mbench.err; echo "mbench rc=$?"; tail -1 gpurun_out/${T}_mbench.log | cut -c1-3000; grep -v "^W0\|^\*\*\*\|^$" gpurun_out/${T}_mbench.err | tail -40; fi
if [ -n "$TRACE_VARIANTS" ]; then
  for v in "default" "ZKB_NTT_MAX_A=8" "ZKB_MSM_SHIFT_GB=0"; do
    echo "== $v" >> gpurun_out/${T}_variants.log
    if [ "$v" = "default" ]; then timeout 300 python scripts/proof_trace.py super 20 128 >> gpurun_out/${T}_variants.log 2>&1; else env $v timeout 300 python scripts/proof_trace.py super 20 128 >> gpurun_out/${T}_variants.log 2>&1; fi
  done
  grep -E "^==|seconds_traced|zkb trace" gpurun_out/${T}_variants.log | cut -c1-400
fi
if [ -n "$LAUNCH_LIST" ]; then timeout 600 ncu --metrics gpu__time_duration.sum --clock-control none --csv --log-file gpurun_out/${T}_launches_bench.csv python bench.py --steps 1 --warmup 3 --no-extras --no-cpu-baseline > gpurun_out/${T}_launches_bench.log 2>&1; wc -l gpurun_out/${T}_launches_bench.csv; fi
if [ -n "$NCU_PROOF" ]; then
  timeout 400 ncu --set full --clock-control none --import-source on -k regex:expr_kernel -s 55 -c 2 -o gpurun_out/${T}_expr -f python scripts/proof_trace.py super 20 128 > gpurun_out/${T}_ncu_expr.log 2>&1
  timeout 400 ncu --set full --clock-control none --import-source on -k regex:msm_acc_chunk -s 2 -c 1 -o gpurun_out/${T}_msmacc -f python scripts/proof_trace.py super 20 128 > gpurun_out/${T}_ncu_msmacc.log 2>&1
fi
if [ -n "$SMOKE" ]; then timeout 300 python -c "import __graft_entry__ as g; g.smoke()" 2>&1 | tail -2; fi
ls -la gpurun_out | tail -12
