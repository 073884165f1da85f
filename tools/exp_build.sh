#!/bin/bash
# Builds an experimental variant of the library next to the shipped one:
#   tools/exp_build.sh NAME "-DLCB_EXP_FOO -DLCB_EXP_BAR=3"  ->  lattice_cryptography_b200/liblcb200_exp_NAME.so
# Select it at run time with LCB200_LIB=<path> (lattice_cryptography_b200/_ffi.py).  The variants are git-ignored (*.so)
# but travel to the GPU box with the rest of the working tree.  The sources are the Makefile's SRCS, so a variant carries
# every entry point of the shipped library.
set -e
NAME=$1; FLAGS=$2
cd "$(dirname "$0")/../lattice_cryptography_b200/csrc"
SRCS=$(make -s --no-print-directory -f Makefile -f - print-srcs <<< 'print-srcs: ; @echo $(SRCS)')
mkdir -p exp_$NAME
rm -f exp_$NAME/*.o
for f in $SRCS; do
  nvcc -gencode arch=compute_100a,code=sm_100a -O3 -std=c++17 -lineinfo -Xcompiler -fPIC $FLAGS -c $f -o exp_$NAME/${f%.cu}.o &
done
wait
nvcc -gencode arch=compute_100a,code=sm_100a -shared -o ../liblcb200_exp_$NAME.so exp_$NAME/*.o
echo built ../liblcb200_exp_$NAME.so
