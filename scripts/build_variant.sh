#!/bin/bash
# usage: [EXTRA_FLAGS="..."] build_variant.sh N [sources]  -> erp_match_eightpoint_test_b200/lib/exp_N/liberp_b200.so built
# with -DERP_TC_COUNTERS=N (0: none, 1: clock64 phase timers in knn_tc1.cu, 2: insert-path event counters) and $EXTRA_FLAGS
# on the given sources (default knn_tc1), linked with the objects of the regular build for the others (build.py SOURCES);
# run with ERP_B200_LIB=<that .so> scripts/tc_profile.py ...
set -e
cd "$(dirname "$0")/.."
N=$1; P=erp_match_eightpoint_test_b200; O=$P/lib/exp_$N; mkdir -p $O
FL="-gencode arch=compute_100a,code=sm_100a -O3 -lineinfo -std=c++17 -Xcompiler -fPIC,-fvisibility=hidden -ccbin /usr/bin/g++ --fmad=false -I include -I $P/csrc -DERP_TC_COUNTERS=$N $EXTRA_FLAGS"
for f in ${2:-knn_tc1}; do nvcc $FL -c $P/csrc/$f.cu -o $O/$f.o & done; wait
OBJS=""
for f in $(python3 -c "import sys; sys.path.insert(0, '$P'); from build import SOURCES; print(' '.join(s[:-3] for s in SOURCES))"); do
    if [ -f $O/$f.o ]; then OBJS="$OBJS $O/$f.o"; else OBJS="$OBJS $P/lib/$f.o"; fi
done
nvcc -shared -o $O/liberp_b200.so $OBJS -gencode arch=compute_100a,code=sm_100a -cudart static -ldl -lpthread -ccbin /usr/bin/g++
echo $O/liberp_b200.so
