#!/bin/bash
# Build a variant of libwildfire_b200.so for an A/B on one GPU box:  tools/build_variant.sh NAME [nvcc flags / -D switches]
#   -> build_ab/libNAME.so   (use it with WILDFIRE_B200_LIB=build_ab/libNAME.so python tools/ab_rollout.py c2)
# WARP_SRC / TILE_SRC / API_SRC may name alternative source files (e.g. an older revision extracted with `git show`).
set -e
cd "$(dirname "$0")/.."
name=$1; shift
src=wildfire_control_python_b200/csrc
out=build_ab/obj_$name
mkdir -p "$out"
FLAGS="-O3 -std=c++17 -gencode arch=compute_100a,code=sm_100a -lineinfo -Xcompiler -fPIC,-O2 -ccbin g++ -I$src -I$src/../../include"
nvcc $FLAGS "$@" -c "${API_SRC:-$src/wf_api.cu}" -o "$out/wf_api.o" &
nvcc $FLAGS "$@" -c "${WARP_SRC:-$src/wf_warp.cu}" -o "$out/wf_warp.o" &
nvcc $FLAGS "$@" -c "${TILE_SRC:-$src/wf_tile.cu}" -o "$out/wf_tile.o" &
nvcc $FLAGS "$@" -c "$src/wf_learn.cu" -o "$out/wf_learn.o" &
nvcc $FLAGS "$@" -c "$src/wf_hostpool.cpp" -o "$out/wf_hostpool.o" &
wait
nvcc --shared -gencode arch=compute_100a,code=sm_100a -ccbin g++ "$out"/*.o -o "build_ab/lib$name.so"
echo "build_ab/lib$name.so"
