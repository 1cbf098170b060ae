#!/bin/bash
# Builds a variant of the library with extra nvcc flags: tools/build_variant.sh NAME -DFOO ...  ->
# esp-audio-libs_b200/variants/lib_NAME.so (selected at run time with ESPB_LIBRARY=path)
set -e
name=$1; shift
here=$(cd "$(dirname "$0")/.." && pwd)
src=$here/esp-audio-libs_b200/csrc
out=$here/esp-audio-libs_b200/variants
mkdir -p $out/build_$name
for f in api.cu resample_kernel.cu resample_ni_kernel.cu resample_fs_kernel.cu pcm_kernels.cu biquad_kernel.cu util_kernels.cu q15_kernels.cu groups.cu multi.cu plan.cpp wav.cpp; do
  ( nvcc -O3 -std=c++17 -lineinfo -gencode arch=compute_100a,code=sm_100a -Xcompiler -fPIC,-O2,-ffp-contract=off "$@" -c $src/$f -o $out/build_$name/$f.o ) &
done
wait
nvcc -shared -gencode arch=compute_100a,code=sm_100a -o $out/lib_$name.so $out/build_$name/*.o -ldl
rm -rf $out/build_$name
echo built $out/lib_$name.so
