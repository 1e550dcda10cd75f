#!/bin/sh
# Build libnavtex_b200.so (sm_100a) in-tree.  nvcc cross-compiles without a GPU.
set -e
cd "$(dirname "$0")/csrc"
NVCC=${NVCC:-/usr/local/cuda/bin/nvcc}
FLAGS="-gencode arch=compute_100a,code=sm_100a -O3 -lineinfo -std=c++17 -Xcompiler -fPIC -Xptxas -v"
mkdir -p ../build
for f in fir_cascade fir_long fir_long_tc demod engine synth; do
  $NVCC $FLAGS -c $f.cu -o ../build/$f.o 2> ../build/$f.ptxas.log || { cat ../build/$f.ptxas.log; exit 1; }
done
$NVCC $FLAGS -c message_assembler.cpp -o ../build/message_assembler.o
$NVCC $FLAGS -c capture_frontend.cpp -o ../build/capture_frontend.o
$NVCC -shared -o ../libnavtex_b200.so ../build/fir_cascade.o ../build/fir_long.o ../build/fir_long_tc.o ../build/demod.o ../build/engine.o ../build/synth.o \
      ../build/message_assembler.o ../build/capture_frontend.o -arch=sm_100a -lcudart_static -lpthread -ldl -lrt
g++ -O2 -std=c++17 -fPIC -shared -o ../libnavtex_compat.so navtex_compat.cpp -L.. -lnavtex_b200 -Wl,-rpath,'$ORIGIN'
# SASS evidence (UTCHMMA / LDTM / STTM / UTMALDG / FFMA2 ... per kernel), regenerated with every build next to the objects;
# profiles/sass_r2.txt is a committed copy and the build leaves it alone
sh ../../tools/sass_counts.sh ../libnavtex_b200.so > ../build/sass_counts.txt 2>/dev/null || true
grep -h "registers\|spill" ../build/*.ptxas.log | sort | uniq -c
ls -la ../libnavtex_b200.so ../libnavtex_compat.so
