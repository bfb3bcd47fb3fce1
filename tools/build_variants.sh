#!/bin/bash
# Builds tuning variants of libpm_b200.so into variants/ (git-ignored; they travel to the GPU box):
#   tools/build_variants.sh NAME "-DFLAG=..." [unit.cu ...]     (default unit: backplane_kernels.cu)
# Only the listed translation units are recompiled with -DPM_TUNING and the flags; the rest of
# the library is linked from the product build's objects.
set -e
ROOT="$(cd "$(dirname "$0")/.." && pwd)"
NAME="$1"; FLAGS="$2"; shift 2 || true
UNITS="${@:-backplane_kernels.cu}"
CSRC="$ROOT/planetmapper_b200/csrc"
OUT="$ROOT/variants"; mkdir -p "$OUT/obj_$NAME"
make -C "$CSRC" -j8 >/dev/null
OBJS=""
for o in backplane_kernels proj_kernels gather_kernels smooth_kernels stage_kernels host_ephem regrid_kernels capi; do
  if echo "$UNITS" | grep -q "$o.cu"; then
    /usr/local/cuda/bin/nvcc -O3 -std=c++17 -lineinfo -gencode arch=compute_100a,code=sm_100a -Xcompiler -fPIC -Xptxas -v \
       $( [ "$o" = backplane_kernels ] && echo -fmad=false ) -DPM_TUNING $FLAGS -c "$CSRC/$o.cu" -o "$OUT/obj_$NAME/$o.o" 2> "$OUT/obj_$NAME/$o.ptxas.log"
    OBJS="$OBJS $OUT/obj_$NAME/$o.o"
  else
    OBJS="$OBJS $CSRC/build/$o.o"
  fi
done
/usr/local/cuda/bin/nvcc -gencode arch=compute_100a,code=sm_100a -shared -o "$OUT/libpm_$NAME.so" $OBJS
echo "built $OUT/libpm_$NAME.so"
