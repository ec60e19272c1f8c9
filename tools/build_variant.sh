#!/bin/bash
# Build an A/B variant of the library with extra -D flags into arap_flow_b200/variants/libarapb200_<name>.so
#   tools/build_variant.sh trial "-DTRIAL_SWITCH=1"
#   SRC_OVERRIDE=<other tree>/arap_flow_b200/csrc tools/build_variant.sh parent ""
# Select it at run time with ARAPB200_LIB=<path> (arap_flow_b200/lib.py).  Measurement aid only.
set -e
name=$1; defs=$2
root=$(cd "$(dirname "$0")/.." && pwd)
src=${SRC_OVERRIDE:-$root/arap_flow_b200/csrc}   # SRC_OVERRIDE: build another revision of the sources (bisecting)
bld=$root/arap_flow_b200/csrc/build_$name
out=$root/arap_flow_b200/variants
mkdir -p "$bld" "$out"
flags="-O3 -std=c++17 -gencode arch=compute_100a,code=sm_100a $defs -lineinfo -fmad=false -prec-div=true -prec-sqrt=true -Xcompiler -fPIC,-fvisibility=hidden"
objs=""
for f in solver_stream solver_resident solver_lm plan pipeline warp composite opt_api arapb200_api; do
  ( /usr/local/cuda/bin/nvcc $flags -c -o "$bld/$f.o" "$src/$f.cu" 2> "$bld/$f.log" || { cat "$bld/$f.log"; exit 1; } ) &
  objs="$objs $bld/$f.o"
done
wait
/usr/local/cuda/bin/nvcc -gencode arch=compute_100a,code=sm_100a -shared -o "$out/libarapb200_$name.so" $objs -Xcompiler -fPIC
echo "built $out/libarapb200_$name.so"
