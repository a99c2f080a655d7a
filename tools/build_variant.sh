#!/bin/bash
# Diagnostic / tuning builds of the product library: tools/build_variant.sh <name> [-D... flags]
# -> build/libttmpc_<name>.so (select with TTMPC_LIB=build/libttmpc_<name>.so)
set -e
cd "$(dirname "$0")/.."
name=$1; shift
mkdir -p build/var_$name
NVF="-gencode arch=compute_100a,code=sm_100a -lineinfo -O3 -std=c++17 -fmad=false -Xcompiler -fPIC -Xcompiler -O2 -Iinclude"
C=${TT_SRC:-trajtrack_mpcndqn_rlboost_b200/csrc}
for f in ttmpc_solve ttmpc_api ttmpc_fleet ttdqn; do
  nvcc $NVF "$@" -c $C/$f.cu -o build/var_$name/$f.o &
done
wait
nvcc -shared -gencode arch=compute_100a,code=sm_100a -o build/libttmpc_$name.so build/var_$name/*.o -lcudart
echo build/libttmpc_$name.so
