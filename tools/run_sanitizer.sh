#!/bin/bash
# compute-sanitizer over the kernel numerics tests (SURVEY §5.2: the in-kernel producer / consumer
# flag protocol, the mbarrier pipelines and the DSMEM statistics exchange are the race surface).
#   tools/run_sanitizer.sh [memcheck|racecheck|synccheck|initcheck] [suite]
# suite:  gemm     tcgen05 GEMM incl. the GEMM + LayerNorm cluster kernel
#         rows     LayerNorm fwd/bwd, column sums, softmax-CE, fused optimizers
#         attn     attention fwd/bwd (head size 64 and the other head sizes)
#         layers   embeddings + block + pooler + classifier through the layer classes (embed_fwd /
#                  embed_bwd / small_linear kernels) and the flag handshake (peer_copy_signal,
#                  wait_flags, flag-gated GEMM) on one GPU
#         all      everything above (default)
# Runs on ONE GPU; reports land in gpurun_out/sanitizer_<tool>_<suite>.log.  The sanitizer slows
# kernels 10-100x: the 4 s flag-wait timeouts are only meaningful under memcheck / synccheck.
set -uo pipefail
TOOL=${1:-memcheck}
SUITE=${2:-all}
mkdir -p gpurun_out
run() {  # name, pytest args...
  local name=$1; shift
  compute-sanitizer --tool "$TOOL" --print-limit 50 --error-exitcode 7 \
    --log-file "gpurun_out/sanitizer_${TOOL}_${name}.log" \
    python -m pytest -x -q -p no:cacheprovider "$@" 2>&1 | tail -3
  echo "[sanitizer] tool=$TOOL suite=$name exit=$? $(grep -c 'ERROR SUMMARY: 0 errors' gpurun_out/sanitizer_${TOOL}_${name}.log) clean-summaries"
  tail -n 2 "gpurun_out/sanitizer_${TOOL}_${name}.log"
}
case "$SUITE" in gemm|all)
  run gemm tests/test_kernels_gpu.py -k "(gemm_kk and 1024-1024-1024) or gelu_dual or residual_and_dgelu or dgrad_layout or wgrad_layout or layernorm_epilogue" ;;
esac
case "$SUITE" in rows|all)
  run rows tests/test_kernels_gpu.py tests/test_optim_gpu.py -k "layernorm_fwd_bwd or colsum or softmax_ce or dropout_mask_consistent or fused_optimizer" ;;
esac
case "$SUITE" in attn|all)
  run attn tests/test_kernels_gpu.py tests/test_attention_head_dims_gpu.py -k "attention and not engine and not span and not two_gpu" ;;
esac
case "$SUITE" in layers|all)
  run layers tests/test_layers_gpu.py tests/test_kernels_gpu.py -k "embeddings_pooler_classifier or handshake or signals_panels" ;;
esac
