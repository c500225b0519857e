#!/bin/sh
# Builds libpointdae_b200.so (sm_100a only) next to the Python host package.
# usage: sh build.sh [extra nvcc flags]
set -e
HERE="$(cd "$(dirname "$0")" && pwd)"
OUT="$HERE/../lib"
mkdir -p "$OUT" "$HERE/../_obj"
NVCC="${NVCC:-/usr/local/cuda/bin/nvcc}"
FLAGS="-gencode arch=compute_100a,code=sm_100a -O3 -lineinfo -std=c++17 -Xcompiler -fPIC -I$HERE/../../include $*"
for f in api step chamfer chamfer_tc fps patchify knn knn3 knn4 featknn ballquery interp corrupt edgeconv conv_tc exchange pairloss reverse emd pointops; do
  src="$HERE/$f.cu"; obj="$HERE/../_obj/$f.o"
  if [ ! -f "$obj" ] || [ "$src" -nt "$obj" ] || [ "$HERE/common.cuh" -nt "$obj" ] || [ "$HERE/knn_select.cuh" -nt "$obj" ] || [ "$HERE/fps_rank.cuh" -nt "$obj" ] || [ "$HERE/reverse.cuh" -nt "$obj" ] || [ "$HERE/../../include/pointdae_b200.h" -nt "$obj" ]; then
    "$NVCC" $FLAGS -c "$src" -o "$obj" &
  fi
done
wait
"$NVCC" -gencode arch=compute_100a,code=sm_100a -shared -o "$OUT/libpointdae_b200.so" "$HERE"/../_obj/api.o "$HERE"/../_obj/step.o "$HERE"/../_obj/chamfer.o "$HERE"/../_obj/chamfer_tc.o "$HERE"/../_obj/fps.o "$HERE"/../_obj/patchify.o \
  "$HERE"/../_obj/knn.o "$HERE"/../_obj/knn3.o "$HERE"/../_obj/knn4.o "$HERE"/../_obj/featknn.o "$HERE"/../_obj/ballquery.o "$HERE"/../_obj/interp.o "$HERE"/../_obj/corrupt.o "$HERE"/../_obj/edgeconv.o "$HERE"/../_obj/conv_tc.o "$HERE"/../_obj/exchange.o "$HERE"/../_obj/pairloss.o "$HERE"/../_obj/reverse.o "$HERE"/../_obj/emd.o "$HERE"/../_obj/pointops.o -cudart static
echo "built $OUT/libpointdae_b200.so"
