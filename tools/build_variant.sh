#!/bin/bash
# A/B helper: build a variant of libhh_b200.so with extra -D flags on selected sources.
#   tools/build_variant.sh NAME "-DHH_GEMM_TRACE" gemm_tcgen05.cu [more.cu ...]
# -> tools/ab/libhh_b200_NAME.so (git-ignored, travels with gpurun); run with HH_B200_LIB=tools/ab/libhh_b200_NAME.so
set -e
ROOT=$(cd "$(dirname "$0")/.." && pwd)
NAME=$1; FLAGS=$2; shift 2
CSRC=$ROOT/helping_hand_for_egocentric_videos_b200/csrc
make -C $CSRC -j8 >/dev/null
OBJ=$ROOT/build/obj; VOBJ=$ROOT/build/obj_$NAME; mkdir -p $VOBJ $ROOT/tools/ab
OBJS=$(ls $OBJ/*.o)
for f in "$@"; do
  b=${f%.cu}
  /usr/local/cuda/bin/nvcc -gencode arch=compute_100a,code=sm_100a -O3 -std=c++17 -lineinfo -Xcompiler -fPIC \
    --expt-relaxed-constexpr $FLAGS -c $CSRC/$f -o $VOBJ/$b.o
  OBJS=$(echo "$OBJS" | grep -v "/$b.o"); OBJS="$OBJS $VOBJ/$b.o"
done
/usr/local/cuda/bin/nvcc -gencode arch=compute_100a,code=sm_100a -shared -o $ROOT/tools/ab/libhh_b200_$NAME.so $OBJS -cudart static -ldl
echo built tools/ab/libhh_b200_$NAME.so
