#!/bin/bash
# tools/build_variant.sh NAME "-DMREFSR_T_BATCH=4 ..."  -> mrefsr_b200/lib/variants/NAME.so (tuning builds, git-ignored)
set -e
cd "$(dirname "$0")/.."
mkdir -p mrefsr_b200/lib/variants
/usr/local/cuda/bin/nvcc -gencode arch=compute_100a,code=sm_100a -O3 -std=c++17 -lineinfo -Xcompiler -fPIC -Xcompiler -fvisibility=hidden \
  --expt-relaxed-constexpr -Xptxas -v $2 -shared -cudart static -o mrefsr_b200/lib/variants/$1.so mrefsr_b200/csrc/*.cu 2>&1 | grep -A2 "dcn_tc_split_kernel" | grep -E "registers|spill" || true
