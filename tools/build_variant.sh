#!/bin/bash
# developer build of a library variant: tools/build_variant.sh <out.so> <extra nvcc flags...>
set -e
cd "$(dirname "$0")/.."
out=$1; shift
nvcc -gencode arch=compute_100a,code=sm_100a -O3 -lineinfo -std=c++17 -fmad=false -Xcompiler -fPIC "$@" \
  -shared -o "$out" gladsgp_b200/csrc/ggp_api.cu gladsgp_b200/csrc/ggp_loglik.cu \
  gladsgp_b200/csrc/ggp_mcmc.cu gladsgp_b200/csrc/ggp_predict.cu gladsgp_b200/csrc/ggp_rsvd_tc.cu \
  gladsgp_b200/csrc/ggp_ingest.cu gladsgp_b200/csrc/ggp_sobol.cu -cudart static
