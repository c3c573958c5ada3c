#!/bin/bash
# usage: build_variant.sh <suffix> <extra nvcc flags...>   -- DEV_SMALL build of libhipgp_b200.so into hipgp_b200/csrc/variants/lib_<suffix>.so
set -e
SUF=$1; shift
cd "$(dirname "$0")/../../hipgp_b200/csrc"
mkdir -p variants build/v_$SUF
FLAGS="-gencode arch=compute_100a,code=sm_100a -lineinfo -O3 -std=c++17 -Xcompiler -fPIC $@"
nvcc $FLAGS -c plan.cu -o build/v_$SUF/plan.o &
for g in 0 1 4 5; do nvcc $FLAGS -DHIPGP_INST_GROUP=$g -c fast_inst.cu -o build/v_$SUF/fi_$g.o & done
nvcc $FLAGS -DHIPGP_INST_GROUP=2 -c fast_inst.cu -o build/v_$SUF/fi_2.o &
nvcc $FLAGS -DHIPGP_INST_GROUP=3 -c fast_inst.cu -o build/v_$SUF/fi_3.o &
nvcc $FLAGS -DHIPGP_INST_GROUP=6 -c fast_inst.cu -o build/v_$SUF/fi_6.o &
nvcc $FLAGS -DHIPGP_INST_GROUP=7 -c fast_inst.cu -o build/v_$SUF/fi_7.o &
nvcc $FLAGS -DHIPGP_INST_GROUP=8 -c fast_inst.cu -o build/v_$SUF/fi_8.o &
nvcc $FLAGS -DHIPGP_INST_GROUP=9 -c fast_inst.cu -o build/v_$SUF/fi_9.o &
wait
for g in 0 1 2 3 4 5 6 7 8 9; do test -f build/v_$SUF/fi_$g.o || { echo "group $g failed"; exit 1; }; done
test -f build/v_$SUF/plan.o || { echo plan failed; exit 1; }
nvcc -gencode arch=compute_100a,code=sm_100a -shared -o variants/lib_$SUF.so build/v_$SUF/*.o
echo built variants/lib_$SUF.so
