#!/bin/bash
# Build-time variants of the warp QP kernels for A/B runs on the GPU box:  profiles/build_variants.sh name "-DFLAG=.. -DFLAG2"
# -> profiles/_variants/librevs_<name>.so ; select with REVS_LIB=profiles/_variants/librevs_<name>.so
set -e
cd "$(dirname "$0")/.."
mkdir -p profiles/_variants
name=$1; shift
src="contract_f64.cu home_solve.cu dual_update.cu utility_qp.cu utility_qp_warp.cu tree_newton.cu feeder_build.cu network_check.cu repair.cu central.cu certify.cu hosting.cu screen_bf16.cu screen_tc5.cu revs_capi.cu"
nvcc -gencode arch=compute_100a,code=sm_100a -lineinfo -O3 -std=c++17 --threads 0 -shared -Xcompiler -fPIC $@ \
  -o profiles/_variants/librevs_$name.so $(for f in $src; do echo revs-admm_b200/csrc/$f; done)
echo profiles/_variants/librevs_$name.so
