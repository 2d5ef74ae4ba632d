#!/bin/bash
# Development: build libraylib_b200.so with extra nvcc flags into software-raytracing_b200/build/variants/<name>.so
#   tools/build_variant.sh <name> "<extra nvcc flags>"
# Links the host objects and the other device objects (rt_denoise.o) of the last `make`.
# On the GPU box: cp software-raytracing_b200/build/variants/<name>.so software-raytracing_b200/lib/libraylib_b200.so
set -e
ROOT="$(cd "$(dirname "$0")/.." && pwd)"
PKG="$ROOT/software-raytracing_b200"
NAME="$1"; shift
mkdir -p "$PKG/build/variants"
nvcc -std=c++17 -O3 -gencode arch=compute_100a,code=sm_100a --fmad=false -lineinfo -Xcompiler -fPIC -Xcompiler -fvisibility=hidden \
     -I"$ROOT/include" -I"$PKG/csrc/host" -I"$PKG/csrc/device" $@ -c "$PKG/csrc/device/rt_device.cu" -o "$PKG/build/variants/$NAME.o"
nvcc -gencode arch=compute_100a,code=sm_100a -shared -o "$PKG/build/variants/$NAME.so" "$PKG"/build/host_*.o "$PKG/build/rt_denoise.o" "$PKG/build/variants/$NAME.o" \
     -Xlinker --no-undefined -lpthread -lz
rm -f "$PKG/build/variants/$NAME.o"
echo "built $PKG/build/variants/$NAME.so"
