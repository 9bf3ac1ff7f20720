#!/bin/bash
# A/B builds of ONE kernel file with other -D knobs, linked against the other (current) objects:
#   benchmarks/build_variants.sh sim_umma_ts poly1 "-DCOR_SIM_TS_POLY_OF4=1"   ->  cor_b200/build/ab/libcor_b200_poly1.so
# Select one at run time with COR_B200_LIB=<path>.  cor_b200/build/ is git-ignored but travels to the GPU box.
set -e
ROOT=$(cd "$(dirname "$0")/.." && pwd)
FILE=$1; TAG=$2; DEFS=$3
python -m cor_b200.build > /dev/null
mkdir -p "$ROOT/cor_b200/build/ab"
obj="$ROOT/cor_b200/build/ab/${FILE}_${TAG}.o"
nvcc -gencode arch=compute_100a,code=sm_100a -O3 -std=c++17 -lineinfo -Xcompiler -fPIC,-O3 --expt-relaxed-constexpr \
     -I "$ROOT/include" $DEFS -c "$ROOT/cor_b200/csrc/${FILE}.cu" -o "$obj"
others=$(ls "$ROOT"/cor_b200/build/*.o | grep -v "/${FILE}.o")
nvcc -shared -gencode arch=compute_100a,code=sm_100a -cudart static -o "$ROOT/cor_b200/build/ab/libcor_b200_${TAG}.so" $obj $others
echo "built cor_b200/build/ab/libcor_b200_${TAG}.so"
