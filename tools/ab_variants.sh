#!/bin/bash
# builds variants of one CUDA source (-D flags; AB_UNIT = gkm_index (default) | gkm_launch | gkm_svm) into
# build/variants/<name>/gkmkern_pylib.so for A/B runs on the GPU:
#   tools/ab_variants.sh name1:"-DFLAG1 -DFLAG2" name2:"" ...    then   GKM_PYLIB=build/variants/name1/gkmkern_pylib.so python tools/probe_r2.py variants
set -e
cd "$(dirname "$0")/.."
make -C gkmqc_b200/csrc -j 16 > /dev/null
for spec in "$@"; do
  name="${spec%%:*}"; flags="${spec#*:}"
  d=build/variants/$name; mkdir -p $d
  unit=${AB_UNIT:-gkm_index}
  src=gkmqc_b200/csrc/$unit.cu
  if [ -n "$AB_SRC" ] && [ "$name" = "head" ]; then src=$AB_SRC; fi
  nvcc -std=c++17 -O3 -lineinfo -gencode arch=compute_100a,code=sm_100a -Xcompiler -fPIC -Xcompiler -fvisibility=default $flags -Igkmqc_b200/csrc -c $src -o $d/$unit.o &
done
wait
for spec in "$@"; do
  name="${spec%%:*}"; d=build/variants/$name
  unit=${AB_UNIT:-gkm_index}
  objs=$(ls build/csrc/*.o | grep -v /$unit.o)
  nvcc -shared -gencode arch=compute_100a,code=sm_100a -cudart static -o $d/gkmkern_pylib.so $objs $d/$unit.o -lpthread -lm
  echo built $d/gkmkern_pylib.so
done
