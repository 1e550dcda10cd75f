#!/bin/sh
# tools/build_variant.sh NAME "-DNVX_...=.. ..."  -> navtex_b200/variants/libnavtex_b200_NAME.so (tuning aid)
set -e
cd "$(dirname "$0")/../navtex_b200/csrc"
mkdir -p ../variants ../build/v_$1
FLAGS="-gencode arch=compute_100a,code=sm_100a -O3 -lineinfo -std=c++17 -Xcompiler -fPIC $2"
for f in fir_cascade fir_long demod engine; do nvcc $FLAGS -c $f.cu -o ../build/v_$1/$f.o; done
nvcc -shared -arch=sm_100a -o ../variants/libnavtex_b200_$1.so ../build/v_$1/fir_cascade.o ../build/v_$1/engine.o ../build/v_$1/demod.o ../build/v_$1/fir_long.o ../build/fir_long_tc.o ../build/resample.o ../build/synth.o \
     ../build/message_assembler.o ../build/capture_frontend.o -lcudart_static -lpthread -ldl -lrt
