#!/bin/bash
# developer aid: build minimal-sdr_b200/csrc/variants/libmsdr_<tag>.so with extra -D flags for ONE kernel file; select with MSDR_LIBMSDR
# usage: tools/build_variant.sh <tag> <file.cu> <-Dflags...>
set -e
tag=$1; file=$2; shift 2
cd "$(dirname "$0")/../minimal-sdr_b200/csrc"
mkdir -p variants
NV="/usr/local/cuda/bin/nvcc -gencode arch=compute_100a,code=sm_100a -O3 -std=c++17 -lineinfo -Xcompiler -fPIC --expt-relaxed-constexpr"
$NV "$@" -c -o variants/${file%.cu}_$tag.o $file
objs=""
for f in $(sed -n 's/^SRCS *:= *//p' Makefile); do # the library's sources, as the Makefile lists them
  f=${f%.cu}
  if [ "$f.cu" = "$file" ]; then objs="$objs variants/${f}_$tag.o"; else objs="$objs $f.o"; fi
done
/usr/local/cuda/bin/nvcc -gencode arch=compute_100a,code=sm_100a -shared -o variants/libmsdr_$tag.so $objs
echo variants/libmsdr_$tag.so
