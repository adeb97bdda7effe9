#!/bin/bash
# Build an instrumented libfea_b200.so: k_pcg_cluster.cu / k_pcg.cu with extra nvcc flags, the other
# objects from the regular build.  The flags are FEA_CLUSTER_PROFILE / ACCOUNT / TRACE / DEBUG, which
# only observe the solver (cycle counts, per-system timeline, printf); see tools/cluster_timeline.py.
#   tools/build_variant.sh <name> [-DFLAG ...]   ->  build/variants/lib_<name>.so
set -e
cd "$(dirname "$0")/.."
name=$1; shift
mkdir -p build/variants
F="-O3 -std=c++17 -gencode arch=compute_100a,code=sm_100a -lineinfo -Xcompiler -fPIC -Xptxas -v -I include -I fea_diffusion_b200/csrc"
nvcc $F "$@" -c fea_diffusion_b200/csrc/k_pcg_cluster.cu -o build/variants/k_pcg_cluster_$name.o 2> build/variants/$name.ptxas.log &
nvcc $F "$@" -c fea_diffusion_b200/csrc/k_pcg.cu -o build/variants/k_pcg_$name.o 2>> build/variants/$name.k_pcg.log &
wait
objs=$(ls build/*.o | grep -v "k_pcg_cluster.o\|k_pcg.o")
nvcc -shared -gencode arch=compute_100a,code=sm_100a -o build/variants/lib_$name.so $objs build/variants/k_pcg_cluster_$name.o build/variants/k_pcg_$name.o
grep -E "spill" build/variants/$name.ptxas.log | sort | uniq -c
echo built build/variants/lib_$name.so
