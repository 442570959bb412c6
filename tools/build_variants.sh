#!/bin/bash
# builds qgemm_bench variants into tools/variants/ (git-ignored), each with different -D switches
set -e
cd "$(dirname "$0")/.."
mkdir -p tools/variants
SRC="tools/qgemm_bench.cu quantum_systems_b200/csrc/quarter_gemm.cu quantum_systems_b200/csrc/core.cu"
FLAGS="-gencode arch=compute_100a,code=sm_100a -O3 -std=c++17 -lineinfo"
build() { name=$1; shift; nvcc $FLAGS "$@" -o tools/variants/$name $SRC & }
build base
build nostore -DQS_DBG_NOSTORE
build phase -DQS_DBG_PHASE_CLOCKS
build phase_nostore -DQS_DBG_PHASE_CLOCKS -DQS_DBG_NOSTORE
build noload -DQS_DBG_NOLOAD
build noload_nostore -DQS_DBG_NOLOAD -DQS_DBG_NOSTORE
build nolds -DQS_DBG_NOLDS -DQS_DBG_NOSTORE
build nowait -DQS_DBG_NOWAIT -DQS_DBG_NOLOAD -DQS_DBG_NOSTORE
build nolds_nowait -DQS_DBG_NOLDS -DQS_DBG_NOWAIT -DQS_DBG_NOLOAD -DQS_DBG_NOSTORE
wait
ls -la tools/variants
