#!/bin/sh
# Build libradiofm_b200.so (in-tree) for sm_100a.  -fmad=false: see rfm_math.cuh.
#   sh build.sh                      the product library: reads no environment variable at run time
#   RFM_EXPERIMENTS=1 sh build.sh    libradiofm_b200_exp.so: the same sources with the RFM_DEBUG_* / RFM_LANES_* /
#                                    RFM_RES_* measurement knobs compiled in (select it with RFM_LIB_PATH in Python)
set -e
cd "$(dirname "$0")"
NVCC=${NVCC:-/usr/local/cuda/bin/nvcc}
ARCH="-gencode arch=compute_100a,code=sm_100a"
DEFS=""
OUT=../libradiofm_b200.so
B=build
if [ "${RFM_EXPERIMENTS:-0}" = 1 ]; then
  DEFS="-DRFM_EXPERIMENTS"
  OUT=../libradiofm_b200_exp.so
  B=build_exp
fi
NVFLAGS="$ARCH -O3 -std=c++17 -lineinfo -fmad=false $DEFS -Xcompiler -fPIC,-fvisibility=hidden,-ffp-contract=off"
CXXFLAGS="-O2 -std=c++17 -fPIC -fvisibility=hidden -ffp-contract=off $DEFS"
mkdir -p $B
pids=""
for f in rfm_kernels rfm_api rfm_probe rfm_freqshift rfm_downconvert rfm_primitives rfm_scan rfm_iqcorr; do
  $NVCC $NVFLAGS -c $f.cu -o $B/$f.o &
  pids="$pids $!"
done
for f in rfm_plan rfm_rdssync rfm_rdsgroup rfm_source; do
  g++ $CXXFLAGS -c $f.cpp -o $B/$f.o &
  pids="$pids $!"
done
g++ $CXXFLAGS -I/usr/local/cuda/include -c rfm_demux.cpp -o $B/rfm_demux.o &
pids="$pids $!"
for p in $pids; do
  wait $p
done
$NVCC $ARCH -shared -o $OUT $B/rfm_kernels.o $B/rfm_api.o $B/rfm_probe.o $B/rfm_freqshift.o $B/rfm_downconvert.o $B/rfm_primitives.o $B/rfm_scan.o $B/rfm_iqcorr.o $B/rfm_plan.o $B/rfm_rdssync.o $B/rfm_rdsgroup.o $B/rfm_source.o $B/rfm_demux.o -lcudart_static -lpthread -ldl -lrt
echo "built $(readlink -f $OUT)"
