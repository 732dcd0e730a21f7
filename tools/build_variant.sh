#!/bin/bash
# A/B build of the library with extra nvcc flags:  tools/build_variant.sh <name> [-D...]   ->  build/libssd_<name>.so
# (use on the GPU box with SSD_GPU_LIB=build/libssd_<name>.so)
set -e
cd "$(dirname "$0")/.."
name=$1; shift
mkdir -p build
C=stair_step_detector_b200/csrc
/usr/local/cuda/bin/nvcc -gencode arch=compute_100a,code=sm_100a -lineinfo -O3 -std=c++17 -fmad=false \
  -Xcompiler -fPIC,-ffp-contract=off,-fvisibility=default -Xptxas -v -shared -cudart static "$@" -o build/libssd_$name.so \
  $C/ssd_gpu.cu $C/ssd_host.cpp $C/host/transformation.cpp $C/host/stairs.cpp $C/host/pointcloud.cpp $C/host/segmentation.cpp \
  $C/host/quadrilateralTest.cpp $C/host/defaultContext.cpp $C/host/calibrationTriangle.cpp $C/host/geometricCalibration.cpp > build/ptxas_$name.log 2>&1
echo "build/libssd_$name.so (resource report: build/ptxas_$name.log)"
