#!/bin/bash
# Builds a tuning variant of the engine next to the product library:
#   tools/build_variant.sh <name> <nvcc -D flags...>   ->  build/variants/lib_<name>.so  (load with MSBWT_LIBRARY_PATH)
set -e
name=$1; shift
cd "$(dirname "$0")/../rust-msbwt_b200/csrc"
g++ -O3 -std=c++17 -fPIC -Wall -Wextra -pthread -c hostpack.cpp -o /tmp/hostpack_variant.o
g++ -O3 -std=c++17 -fPIC -Wall -Wextra -c codec.cpp -o /tmp/codec_variant.o
mkdir -p ../../build/variants
nvcc -O3 -std=c++17 -gencode arch=compute_100a,code=sm_100a -lineinfo -Xcompiler -fPIC,-O3 -shared "$@" \
  -o ../../build/variants/lib_${name}.so capi.cu hostpath.cu kernels.cu quad_kernels.cu stats_kernels.cu wide_kernels.cu final_kernels.cu ext_kernels.cu loader.cu builder.cu pair_builder.cu quad_builder.cu \
  oct_builder.cu fin_builder.cu bwt_build.cu bwt_merge.cu spectrum.cu unitigs.cu correct.cu /tmp/hostpack_variant.o /tmp/codec_variant.o 2>&1 | grep -E "error|Segmentation" || true
ls -la ../../build/variants/lib_${name}.so
