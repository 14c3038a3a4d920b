#!/bin/bash
# Build kernel-experiment variants of libfxb200.so (never committed; lib/exp/ is git-ignored with every other .so):
#   tools/exp_build.sh name '<extra nvcc flags, e.g. -Xptxas -v>' ['sed-script for csrc/fx_analyse.cu'] ['sed-script for fx_fft.cuh']
# -> feature-extractor_b200/lib/exp/libfxb200_<name>.so ; select it with FXB200_LIB=<path>
set -e
ROOT=$(cd "$(dirname "$0")/.." && pwd)
name=$1; W=/tmp/fxexp_$name
rm -rf $W; mkdir -p $W/feature-extractor_b200 $W/include
cp -r $ROOT/feature-extractor_b200/csrc $W/feature-extractor_b200/
cp $ROOT/include/fx_engine.h $W/include/
[ -n "$3" ] && sed -i -E "$3" $W/feature-extractor_b200/csrc/fx_analyse.cu
[ -n "$4" ] && sed -i -E "$4" $W/feature-extractor_b200/csrc/fx_fft.cuh
mkdir -p $ROOT/feature-extractor_b200/lib/exp
cd $W/feature-extractor_b200
/usr/local/cuda/bin/nvcc -O3 -std=c++17 -gencode arch=compute_100a,code=sm_100a -lineinfo -Xcompiler -fPIC -shared $2 \
  -o $ROOT/feature-extractor_b200/lib/exp/libfxb200_$name.so csrc/fx_analyse.cu csrc/fx_post.cu csrc/fx_pcm.cu csrc/fx_tables.cu csrc/fx_legacy.cu csrc/fx_engine.cu -lcudart -lpthread
echo built $name
