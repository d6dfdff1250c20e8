#!/usr/bin/env bash
# Build the host tools into build/ (git-ignored, travels to the GPU box):
#   build/nam_b200_bench        our own C++ tool over the C ABI
#   build/nam_b200_multi_test   a C++ host driving several GPUs through the C ABI (nam_b200_multi_*)
#   build/microbench            design-constant micro-benchmarks (tools/microbench.cu)
# (The reference's own tools, compiled unchanged against include/NAM/*.h, are built by `make -C oracle ref_tools`.)
set -euo pipefail
ROOT="$(cd "$(dirname "$0")/.." && pwd)"
LIBDIR="$ROOT/neuralampmodelercore_b200/lib"
mkdir -p "$ROOT/build"
CXX=${CXX:-g++}
"$CXX" -std=c++17 -O2 -I"$ROOT/include" -o "$ROOT/build/nam_b200_bench" "$ROOT/tools/nam_b200_bench.cpp" \
  -L"$LIBDIR" -lnam_b200 -Wl,-rpath,'$ORIGIN/../neuralampmodelercore_b200/lib'
"$CXX" -std=c++17 -O2 -I"$ROOT/include" -o "$ROOT/build/nam_b200_multi_test" "$ROOT/tools/nam_b200_multi_test.cpp" \
  -L"$LIBDIR" -lnam_b200 -Wl,-rpath,'$ORIGIN/../neuralampmodelercore_b200/lib'
if command -v nvcc >/dev/null 2>&1; then
  nvcc -gencode arch=compute_100a,code=sm_100a -O3 -lineinfo -o "$ROOT/build/microbench" "$ROOT/tools/microbench.cu"
fi
