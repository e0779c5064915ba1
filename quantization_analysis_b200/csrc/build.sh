#!/bin/sh
# Build libqa_b200.so in-tree for sm_100a (cross-compiles without a GPU).
set -e
cd "$(dirname "$0")"
NVCC=${NVCC:-/usr/local/cuda/bin/nvcc}
OUT=../libqa_b200.so
$NVCC -gencode arch=compute_100a,code=sm_100a -O3 -lineinfo -std=c++17 \
      -Xcompiler -fPIC -shared ${QA_NVCC_EXTRA} \
      -o "$OUT" qa_recon.cu qa_stats.cu qa_scores.cu qa_assign.cu qa_greedy_par.cu qa_perm_apply.cu qa_faithful.cu qa_stats_f32.cu qa_transpose.cu
echo "built $OUT"
