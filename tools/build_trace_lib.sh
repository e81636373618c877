#!/bin/bash
# builds a trace variant of the library (clock64 trace points of the env kernel: -DCM_ENV_TRACE -DCM_TC_TRACE) -> $1
# usage: bash tools/build_trace_lib.sh tests/native/lib_trace.so ; COM_MARL_B200_LIB=tests/native/lib_trace.so python tests/native/trace_env.py c3
set -e
OUT=${1:-tests/native/lib_trace.so}
cd "$(dirname "$0")/.."
SRC="env_kernels.cu policy_forward.cu policy_tc_kernel.cu policy_attn_mma_kernel.cu policy_cent_kernel.cu host_abi.cu ppo_kernels.cu ppo_net_kernels.cu abi.cu"
mkdir -p /tmp/trace_obj
for f in $SRC; do
  nvcc -gencode arch=compute_100a,code=sm_100a -O3 -lineinfo -std=c++17 -Xcompiler -fPIC -DCM_ENV_TRACE -DCM_TC_TRACE -I include -I com_marl_b200/csrc -c com_marl_b200/csrc/$f -o /tmp/trace_obj/${f%.cu}.o &
done
wait
nvcc -gencode arch=compute_100a,code=sm_100a -shared -Xcompiler -fPIC -o $OUT /tmp/trace_obj/*.o
echo built $OUT
