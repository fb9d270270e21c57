#!/bin/bash
# Builds a variant of libpt_core.so with extra nvcc flags into scratch/variants/<name>/ (A/B
# experiments on the GPU box: PT_CORE_LIB=scratch/variants/<name>/libpt_core.so python bench.py ...).
#   tools/build_variant.sh <name> [-f "file1 file2"] <extra nvcc flags ...>
# -f lists the sources the flags apply to (default: wavefront — the only one the numeric tuning parameters
# such as -DPT_NODE_LOOP_LANES=8 or -DPT_TRACE_MIN_BLOCKS=6 touch); the other objects are taken from the
# in-tree build (run make there first).
set -e
name=$1; shift
files="wavefront"
if [ "$1" = "-f" ]; then files=$2; shift; shift; fi
root=$(cd "$(dirname "$0")/.." && pwd)
out=$root/scratch/variants/$name
mkdir -p "$out"
cd "$root/path-tracing_b200/csrc"
objs=""
for f in pt_core bvh_build textures wavefront postprocess unit_kernels; do
  if [[ " $files " == *" $f "* ]]; then
    nvcc -O3 -std=c++17 -gencode arch=compute_100a,code=sm_100a -lineinfo -fmad=false \
         -Xcompiler -fPIC,-fvisibility=hidden --expt-relaxed-constexpr -Wno-deprecated-gpu-targets -Xptxas -v "$@" \
         -c $f.cu -o "$out/$f.o" 2> "$out/$f.ptxas.log" &
    objs="$objs $out/$f.o"
  else
    objs="$objs $f.o"
  fi
done
wait
nvcc -gencode arch=compute_100a,code=sm_100a -shared -o "$out/libpt_core.so" $objs -cudart static
rm -f "$out"/*.o
echo "$out/libpt_core.so"
