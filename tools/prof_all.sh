#!/bin/bash
# Per-kernel `ncu --set full` capture of every kernel family of libqsb200.so (one GPU).  Only our kernels are
# profiled (-k regex), the report is converted to CSV on the box and removed (it exceeds the 64 MiB pull limit).
set -e
OUT=${1:-gpurun_out/prof_all}
KERNELS='regex:quarter_gemm|build_.*image_kernel|pad_rows_kernel|add_spin|antisym_kernel|spin2_tb_kernel|fock_kernel|tdho_coulomb_kernel|pair_product_kernel|extract_block_kernel|scale_add_kernel|occupied_traces_kernel'
python tools/prof_all.py > ${OUT}_plain.log 2>&1
ncu --set full --clock-control none -k "$KERNELS" -c 80 -o /tmp/prof_all python tools/prof_all.py > ${OUT}_ncu.log 2>&1
ncu -i /tmp/prof_all.ncu-rep --page raw --csv > ${OUT}_raw.csv
python tools/ncu_summary.py ${OUT}_raw.csv > ${OUT}_summary.csv
gzip -f ${OUT}_raw.csv
ls -la ${OUT}*
