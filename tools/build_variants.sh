#!/bin/bash
# Kernel-tuning helper: builds libgvpm_b200 variants with different -D settings of gather_bre.cu into build/variants/
# (git-ignored; they travel to the GPU box).  Usage: tools/build_variants.sh name1 "-DA=1 -DB=2" name2 "..." ...
# The other objects are the library's own sources, as __graft_entry__.CU_SOURCES lists them.
set -e
cd "$(dirname "$0")/.."
CS=gvpm_b200/csrc
FL="-gencode arch=compute_100a,code=sm_100a -lineinfo -O3 -std=c++17 -Xcompiler -fPIC"
OTHERS=$(python3 -c "import __graft_entry__ as g; print(' '.join(s[:-3] for s in g.CU_SOURCES if s != 'gather_bre.cu'))")
mkdir -p build/variants/obj
for f in $OTHERS; do
  if [ ! -f build/variants/obj/$f.o ] || [ $CS/$f.cu -nt build/variants/obj/$f.o ]; then nvcc $FL -c $CS/$f.cu -o build/variants/obj/$f.o & fi
done
wait
OBJS=$(for f in $OTHERS; do printf 'build/variants/obj/%s.o ' $f; done)
while [ $# -ge 2 ]; do
  name=$1; defs=$2; shift 2
  ( nvcc $FL $defs -c $CS/gather_bre.cu -o build/variants/obj/gather_bre_$name.o && \
    nvcc -shared -o build/variants/lib_$name.so $OBJS build/variants/obj/gather_bre_$name.o && echo "built $name ($defs)" ) &
done
wait
