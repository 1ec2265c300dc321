#!/bin/bash
# A/B variant of the CUDA library that differs only in one translation unit:
#   tools/ab_build.sh NAME "-DAG_LUT_BLOCKS_PER_SM=3 ..." [TU=ag_rollout_lut]
# compiles csrc/$TU.cu with the extra flags and links it with the in-tree objects of the other units
# (abstract_gym_b200/build/*.o from `python -m abstract_gym_b200.build`) into build_ab/NAME.so.
# A flag that more than one unit reads needs a full build instead: -DAG_CMAP_B1/B2 changes the map's layout, which
# ag_cmap.cu (the producer) and ag_rollout_lut.cu, ag_motion.cu, ag_cspace.cu (the readers) must agree on:
#   AG_NVCC_EXTRA="-DAG_CMAP_B1=11" python -m abstract_gym_b200.build --out build_ab/NAME.so
set -e
name=$1; flags=$2; tu=${3:-ag_rollout_lut}
here=$(cd "$(dirname "$0")/.." && pwd)
mkdir -p $here/build_ab
nvcc -gencode arch=compute_100a,code=sm_100a -lineinfo -O3 -std=c++17 -Xcompiler -fPIC,-ffp-contract=off,-fvisibility=hidden \
     -Xptxas -v $flags -I $here/include -c -o $here/build_ab/$name.o $here/abstract_gym_b200/csrc/$tu.cu > $here/build_ab/$name.log 2>&1
others=$(ls $here/abstract_gym_b200/build/*.o | grep -v "/$tu.o")
nvcc --shared -gencode arch=compute_100a,code=sm_100a -o $here/build_ab/$name.so $here/build_ab/$name.o $others
echo build_ab/$name.so
