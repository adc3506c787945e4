#!/bin/bash
# developer build of the library with phase timers (not the product build)
set -e
cd "$(dirname "$0")/.."
mkdir -p build_var
nvcc -gencode arch=compute_100a,code=sm_100a -O3 -lineinfo -std=c++17 -fmad=false -Xcompiler -fPIC -DGGP_PHASES \
  -shared -o build_var/libggp_phases.so gladsgp_b200/csrc/ggp_api.cu gladsgp_b200/csrc/ggp_loglik.cu \
  gladsgp_b200/csrc/ggp_mcmc.cu gladsgp_b200/csrc/ggp_predict.cu gladsgp_b200/csrc/ggp_rsvd_tc.cu gladsgp_b200/csrc/ggp_ingest.cu gladsgp_b200/csrc/ggp_sobol.cu -cudart static
