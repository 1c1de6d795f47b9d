#!/bin/bash
# build the current tree as a named library, to A/B it against another revision through NEXAR_LIB (tools/ab2.sh):
#   tools/build_variant.sh NAME [nvcc flags ...]   -> vision_collision_detection_b200/exp_NAME.so
cd "$(dirname "$0")/.."
n=$1; shift
nvcc -O3 -std=c++17 -gencode arch=compute_100a,code=sm_100a -lineinfo -shared -Xcompiler -fPIC -diag-suppress 550 -I include "$@" -o vision_collision_detection_b200/exp_$n.so vision_collision_detection_b200/csrc/clip_transform.cu
