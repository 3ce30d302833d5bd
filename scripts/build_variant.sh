#!/bin/bash
# Build a kernel-variant library for an A/B run on the GPU box without touching the default build:
#
#   scripts/build_variant.sh NAME "merge"        -DTSGU_MERGE_P=4096 ...     # recompile only merge.cu
#   scripts/build_variant.sh NAME "spmm sddmm"   -DTSGU_TILE_ROWS_DEFAULT=256
#
# -> variants_tmp/lib_NAME.so (git-ignored, travels with gpurun).  The other objects are taken from the default
# in-tree build (csrc/_obj), so run `python -m torchsparsegradutils_b200.csrc.build` first.  Select a variant at run
# time with TSGU_B200_LIB=$PWD/variants_tmp/lib_NAME.so; scripts/merge_variant_sweep.sh loops bench configs over all
# of them (LIBS=..., CONFIGS="2 3 5").  Several variants can be built in parallel (one nvcc per source file).
set -e
ROOT=$(cd "$(dirname "$0")/.." && pwd)
cd "$ROOT/torchsparsegradutils_b200/csrc"
NAME=$1; FILES=$2; shift; shift
TMP=${TMPDIR:-/tmp}
mkdir -p "$ROOT/variants_tmp"
OBJS=""
for f in api spmm sddmm index merge window trisolve; do
  if [[ " $FILES " == *" $f "* ]]; then
    nvcc -gencode arch=compute_100a,code=sm_100a -O3 -std=c++17 -lineinfo -Xcompiler -fPIC,-fvisibility=hidden \
      --expt-relaxed-constexpr -Xptxas -v -DTSGU_BUILD "$@" -c $f.cu -o $TMP/${f}_$NAME.o > $TMP/${f}_$NAME.log 2>&1 &
    OBJS="$OBJS $TMP/${f}_$NAME.o"
  else
    OBJS="$OBJS _obj/$f.o"
  fi
done
wait
nvcc -shared -o "$ROOT/variants_tmp/lib_$NAME.so" $OBJS -gencode arch=compute_100a,code=sm_100a
echo "built variants_tmp/lib_$NAME.so ($FILES: $*)"
