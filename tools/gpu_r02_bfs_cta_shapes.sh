#!/bin/bash
# CTA shapes of the fused BFS kernel (profiles/r02_bfs_levels_and_cta_shapes.txt).
# The variants are builds of the same library with other macros, made on the CPU box:
#   NV="nvcc -gencode arch=compute_100a,code=sm_100a -O3 -std=c++17 -w -lineinfo -shared \
#       -Xcompiler -fPIC,-fvisibility=hidden -I include -I graphblast_b200/csrc -I graphblast_b200/csrc/shim"
#   $NV -DGB_BFS_NT=1024 -DGB_BFS_MINB=2 -o build/variants/nt1024x2.so graphblast_b200/csrc/capi.cu
#   $NV -DGB_BFS_NT=768  -DGB_BFS_MINB=2 -o build/variants/nt768x2.so  graphblast_b200/csrc/capi.cu
#   $NV -DGB_BFS_NT=512  -DGB_BFS_MINB=3 -o build/variants/nt512x3.so  graphblast_b200/csrc/capi.cu
#   $NV -DGB_BFS_NT=1024 -DGB_BFS_MINB=1 -o build/variants/nt1024x1.so graphblast_b200/csrc/capi.cu
# and selected at run time through GB200_LIB.  Each variant's stderr goes to $LOG.
LOG=build/cta_shapes
mkdir -p $LOG
run() {  # name lib
  GB200_LIB=$PWD/build/variants/$2 timeout 600 python bench.py --steps 20 --warmup 5 --no-cpu-baseline 2> $LOG/bfsv_$1.err | python -c "
import json,sys
d=json.loads(sys.stdin.read()); print('$1: bfs ms/step %.4f' % d['ms_per_step'])"
  GB200_BFS_TRACE=1 GB200_LIB=$PWD/build/variants/$2 timeout 600 python bench.py --steps 2 --warmup 3 --no-cpu-baseline 2>&1 >/dev/null | grep "bfs trace" | tail -1
}
run nt1024x2 nt1024x2.so
run nt768x2 nt768x2.so
run nt512x3 nt512x3.so
run nt1024x1 nt1024x1.so
