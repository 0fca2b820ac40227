#!/bin/bash
# developer tool: build libbp4 with extra nvcc flags into mf_data_locality_b200/variants/libbp4_NAME.so
# usage: scripts/build_variant.sh NAME [nvcc flags, e.g. -DBP4_PHASE_TIMING]; copy the result over libbp4.so to probe it
set -e
name=$1; shift
root=$(cd "$(dirname "$0")/.." && pwd)
pkg=$root/mf_data_locality_b200
mkdir -p $pkg/variants /tmp/bp4v_$name
nccl=$(python -c "import sys,os
for p in sys.path:
    d=os.path.join(p,'nvidia','nccl')
    if os.path.isdir(os.path.join(d,'lib')): print(d); break")
flags="-gencode arch=compute_100a,code=sm_100a -lineinfo -O3 -std=c++17 -Xcompiler -fPIC -I $nccl/include"
nvcc $flags "$@" -c $pkg/csrc/bp4_kernels.cu -o /tmp/bp4v_$name/k.o &
nvcc $flags "$@" -c $pkg/csrc/bp4_capi.cu -o /tmp/bp4v_$name/c.o &
wait
nvcc -shared -gencode arch=compute_100a,code=sm_100a -o $pkg/variants/libbp4_$name.so /tmp/bp4v_$name/k.o /tmp/bp4v_$name/c.o \
  -L $nccl/lib -l:libnccl.so.2 -Xlinker -rpath -Xlinker $nccl/lib -lcudart
echo built $pkg/variants/libbp4_$name.so
