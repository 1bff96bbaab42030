#!/bin/bash
# Developer tool: build a kernel variant next to the product library: tools/build_variant.sh <name> <MINB> [extra nvcc flags]
# -> cpuvox_b200/variants/lib_<name>.so ; select with CPUVOX_B200_LIB=cpuvox_b200/variants/lib_<name>.so
set -e
cd "$(dirname "$0")/../cpuvox_b200/csrc"
name=$1; minb=$2; shift 2
mkdir -p ../variants /tmp/cvxvar_$name
NV="/usr/local/cuda/bin/nvcc $* -DCVXD_MIN_CTAS_PER_SM=$minb -gencode arch=compute_100a,code=sm_100a -lineinfo -O3 -std=c++17 -fmad=false -Xcompiler -fPIC"
$NV -c -o /tmp/cvxvar_$name/k.o raybuffer_kernels.cu
$NV -c -o /tmp/cvxvar_$name/c.o capi.cu
make -s raycast_kernels.o world_builder_gpu.o host_setup.o world_builder.o jpeg_encoder.o
/usr/local/cuda/bin/nvcc -shared -o ../variants/lib_$name.so /tmp/cvxvar_$name/k.o /tmp/cvxvar_$name/c.o raycast_kernels.o world_builder_gpu.o host_setup.o world_builder.o jpeg_encoder.o -Xcompiler -pthread -cudart static -ldl
echo built ../variants/lib_$name.so
