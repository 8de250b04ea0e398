#!/bin/bash
# One gpurun call = the whole GPU check list; each stage in its own process (a CUDA trap poisons only its
# own context) under its own timeout; everything lands in gpurun_out/.
# usage: tools/gpu_suite.sh [stages...]   stages: gemm kernels bench ref ncu
set -u
mkdir -p gpurun_out
STAGES="${@:-gemm kernels bench ref}"
export PYTHONUNBUFFERED=1
nvidia-smi --query-gpu=name,clocks.sm,clocks.max.sm,power.draw,memory.used --format=csv > gpurun_out/smi.txt 2>&1
for s in $STAGES; do
  case $s in
    gemm)    timeout 600 python -m pytest tests/test_gpu_gemm.py -m gpu -q -x --timeout 300 > gpurun_out/test_gemm.log 2>&1; echo "gemm rc=$?" ;;
    gemmall) timeout 900 python -m pytest tests/test_gpu_gemm.py -m gpu -q --timeout 300 > gpurun_out/test_gemm.log 2>&1; echo "gemmall rc=$?" ;;
    kernels) timeout 900 python -m pytest tests/test_gpu_kernels.py -m gpu -q --timeout 300 > gpurun_out/test_kernels.log 2>&1; echo "kernels rc=$?" ;;
    attn)    timeout 600 python -m pytest tests/test_gpu_attention.py -m gpu -q --timeout 300 > gpurun_out/test_attn.log 2>&1; echo "attn rc=$?" ;;
    tests)   timeout 1500 python -m pytest tests -m gpu -q --timeout 600 > gpurun_out/test_all.log 2>&1; echo "tests rc=$?" ;;
    smoke)   timeout 300 python -c "import __graft_entry__ as g; g.smoke()" > gpurun_out/smoke.log 2>&1; echo "smoke rc=$?" ;;
    bench)   timeout 900 python bench.py --steps ${BENCH_STEPS:-3} --warmup 3 ${BENCH_ARGS:-} > gpurun_out/bench_ours.json 2> gpurun_out/bench_ours.err; echo "bench rc=$?"; tail -c 1500 gpurun_out/bench_ours.json ;;
    ref)     timeout 1200 python bench.py --impl reference --steps ${BENCH_STEPS:-3} --warmup 3 ${BENCH_ARGS:-} > gpurun_out/bench_ref.json 2> gpurun_out/bench_ref.err; echo "ref rc=$?"; tail -c 1500 gpurun_out/bench_ref.json ;;
    fp8)     timeout 600 python -m pytest tests/test_gpu_fp8.py -m gpu -q --timeout 300 > gpurun_out/test_fp8.log 2>&1; echo "fp8 rc=$?"; tail -15 gpurun_out/test_fp8.log ;;
    gemmbench) timeout 600 python tools/gemm_bench.py ${GEMMBENCH_ARGS:-} > gpurun_out/gemm_bench.json 2> gpurun_out/gemm_bench.err; echo "gemmbench rc=$?"; tail -c 3000 gpurun_out/gemm_bench.json ;;
    launches) timeout 900 ncu --metrics gpu__time_duration.sum --clock-control none -c 3000 --csv --log-file gpurun_out/launches.csv python bench.py --steps 1 --warmup 1 --accum 1 --no-e2e > gpurun_out/launches.log 2>&1; echo "launches rc=$?" ;;
    ncu_gemm) timeout 600 ncu --set full --clock-control none --import-source on -k regex:gemm_pair_kernel -s 12 -c 2 -f -o gpurun_out/prof_gemm python tools/gemm_bench.py --only ${NCU_SHAPE:-ffn1_fwd} > gpurun_out/ncu_gemm.log 2>&1; echo "ncu_gemm rc=$?" ;;
    ncu_elt)  timeout 600 ncu --set full --clock-control none --import-source on -k regex:"ln_fwd2|ln_bwd2|gelu_fwd|dgelu_bwd" -s 20 -c 4 -f -o gpurun_out/prof_elt python tools/elt_bench.py > gpurun_out/ncu_elt.log 2>&1; echo "ncu_elt rc=$?" ;;
    ncu_all)  timeout 900 ncu --set full --profile-from-start off --clock-control none --import-source on -f -o gpurun_out/prof_all python tools/ncu_targets.py > gpurun_out/ncu_all.log 2>&1; echo "ncu_all rc=$?"; tail -3 gpurun_out/ncu_all.log ;;
    sanitize) timeout 420 compute-sanitizer --tool ${SAN_TOOL:-memcheck} --error-exitcode 9 python -m pytest tests/test_gpu_kernels.py tests/test_gpu_gemm.py -q -x --timeout 400 -k "layer_norm_fwd_bwd or gelu_kernels or colsum or embedding_fwd_bwd or mlm_compact or (gemm_nt and 256-256-128)" > gpurun_out/sanitize_${SAN_TOOL:-memcheck}.log 2>&1; echo "sanitize rc=$?"; tail -6 gpurun_out/sanitize_${SAN_TOOL:-memcheck}.log ;;
    eltbench) timeout 300 python tools/elt_bench.py > gpurun_out/elt_bench.json 2> gpurun_out/elt_bench.err; echo "eltbench rc=$?"; cat gpurun_out/elt_bench.json ;;
    ncu_attn) timeout 600 ncu --set full --clock-control none --import-source on -k regex:attn_ -s 6 -c 3 -f -o gpurun_out/prof_attn python tools/attn_bench.py > gpurun_out/ncu_attn.log 2>&1; echo "ncu_attn rc=$?" ;;
    attnbench) timeout 300 python tools/attn_bench.py > gpurun_out/attn_bench.json 2> gpurun_out/attn_bench.err; echo "attnbench rc=$?"; cat gpurun_out/attn_bench.json ;;
    trace)   timeout 600 python tools/trace_step.py > gpurun_out/trace_step.log 2>&1; echo "trace rc=$?"; cat gpurun_out/trace_step.log | tail -30 ;;
    trace2)  PHASE=2 timeout 600 python tools/trace_step.py > gpurun_out/trace_step2.log 2>&1; echo "trace2 rc=$?"; cat gpurun_out/trace_step2.log | tail -30 ;;
    push)    timeout 300 python -m torch.distributed.run --nnodes=1 --nproc-per-node ${NGPU:-2} --master-addr 127.0.0.1 --master-port 29578 tools/push_check.py > gpurun_out/push_check.log 2>&1; echo "push rc=$?"; grep "^{" gpurun_out/push_check.log | tail -1 | cut -c1-3000; tail -5 gpurun_out/push_check.log | cut -c1-500 ;;
    peer)    timeout 600 python -m torch.distributed.run --nnodes=1 --nproc-per-node ${NGPU:-2} --master-addr 127.0.0.1 --master-port 29577 tools/peer_check.py ${PEER_ARGS:-} > gpurun_out/peer_check.log 2>&1; echo "peer rc=$?"; tail -20 gpurun_out/peer_check.log ;;
    experimental)  # opt-in kernels written without GPU access (NOTES.md): correctness under a short timeout, then timing
             B200_LN_FINALIZE_SPLIT=8 timeout 200 python -m pytest tests/test_gpu_kernels.py -m gpu -q -x --timeout 120 -k "layer_norm or pretrainer_matches" > gpurun_out/test_lnsplit.log 2>&1; echo "ln split test rc=$?"; tail -3 gpurun_out/test_lnsplit.log
             B200_LN_ROWS=2 timeout 200 python -m pytest tests/test_gpu_kernels.py tests/test_gpu_fp8.py -m gpu -q -x --timeout 120 -k "layer_norm or pretrainer_matches or producer" > gpurun_out/test_lnrows.log 2>&1; echo "ln rows test rc=$?"; tail -3 gpurun_out/test_lnrows.log
             for r in 1 2; do B200_LN_ROWS=$r timeout 200 python tools/elt_bench.py 2>/dev/null | grep -i "layer_norm_fwd" | sed "s/^/rows=$r /"; done | tee gpurun_out/elt_bench_lnrows.txt
             for z in 1 8; do B200_LN_FINALIZE_SPLIT=$z timeout 200 python tools/elt_bench.py 2>/dev/null | grep -i "ln_bwd\|layer_norm_bwd" | sed "s/^/split=$z /"; done | tee gpurun_out/elt_bench_lnsplit.txt ;;
    *) echo "unknown stage $s" ;;
  esac
done
tail -n 30 gpurun_out/test_*.log 2>/dev/null | tail -n 80
