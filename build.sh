#!/usr/bin/env bash
# Builds libvp8r.so (host parser + runtime + sm_100a kernels) in-tree, the synthetic-stream
# tool, and the test-only oracle.  nvcc cross-compiles without a GPU.
set -euo pipefail
cd "$(dirname "$0")"
OUT=vp8_b200/_lib
mkdir -p "$OUT" vp8_b200/_build
NVCC=${NVCC:-/usr/local/cuda/bin/nvcc}
ARCH="-gencode arch=compute_100a,code=sm_100a"
CXXFLAGS="-O3 -std=c++17 -Iinclude -Ivp8_b200/csrc ${VP8R_EXTRA_FLAGS:-}"
$NVCC $ARCH -lineinfo $CXXFLAGS -Xcompiler -fPIC,-fvisibility=hidden -c vp8_b200/csrc/cuda/recon_kernels.cu -o vp8_b200/_build/recon_kernels.o
$NVCC $ARCH -lineinfo $CXXFLAGS -Xcompiler -fPIC,-fvisibility=hidden -c vp8_b200/csrc/cuda/filter_swar.cu -o vp8_b200/_build/filter_swar.o
$NVCC $ARCH -lineinfo $CXXFLAGS -Xcompiler -fPIC,-fvisibility=hidden -c vp8_b200/csrc/cuda/enc_kernels.cu -o vp8_b200/_build/enc_kernels.o
$NVCC $ARCH -lineinfo $CXXFLAGS -Xcompiler -fPIC,-fvisibility=hidden -c vp8_b200/csrc/cuda/token_kernel.cu -o vp8_b200/_build/token_kernel.o
$NVCC $ARCH -lineinfo $CXXFLAGS -Xcompiler -fPIC,-fvisibility=hidden -c vp8_b200/csrc/rt/engine.cu -o vp8_b200/_build/engine.o
g++ -O3 -funroll-loops -std=c++17 -Iinclude -Ivp8_b200/csrc -march=x86-64-v3 -fPIC -fvisibility=hidden -Wall -Wextra -c vp8_b200/csrc/host/frame_parser.cc -o vp8_b200/_build/frame_parser.o
g++ -O2 -std=c++17 -Iinclude -Ivp8_b200/csrc -Ivp8_b200/csrc/host -fPIC -fvisibility=hidden -Wall -Wextra -c vp8_b200/csrc/host/frame_writer.cc -o vp8_b200/_build/frame_writer.o
g++ $CXXFLAGS -fPIC -fvisibility=hidden -Wall -Wextra -c vp8_b200/csrc/capi.cc -o vp8_b200/_build/capi.o
$NVCC $ARCH -shared -o "$OUT/libvp8r.so" vp8_b200/_build/recon_kernels.o vp8_b200/_build/filter_swar.o vp8_b200/_build/enc_kernels.o vp8_b200/_build/token_kernel.o vp8_b200/_build/engine.o \
    vp8_b200/_build/frame_parser.o vp8_b200/_build/frame_writer.o vp8_b200/_build/capi.o -lpthread
g++ -O2 -std=c++17 -Wall -Wextra tools/vp8synth.cc -o "$OUT/vp8synth"
g++ -O2 -std=c++17 -Wall -Wextra -Iinclude tools/vp8dec.cc -o "$OUT/vp8dec" -L"$OUT" -lvp8r -Wl,-rpath,'$ORIGIN'
make -s -C oracle oracle
mkdir -p oracle_inter/_build
gcc -std=c11 -O2 -fPIC -shared -Wall -Wextra -Iinclude -Ioracle -o oracle_inter/_build/liboracle_inter.so oracle_inter/enc_inter_oracle.c
if [ "${SKIP_REF:-0}" != "1" ]; then make -s -C oracle ref; fi
echo "built $OUT/libvp8r.so"
