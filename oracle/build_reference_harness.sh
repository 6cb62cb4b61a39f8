#!/bin/bash
# Compile the nvCOMP project's own benchmarks/examples UNCHANGED (their sources stay in the nvCOMP tree given as
# $1 or $NVCOMP_REFERENCE_DIR, nothing is copied) against this library's headers and libnvcomp.so -> oracle/_ref/.
# Acceptance harness for the drop-in boundary (SURVEY.md 2a: "must compile & link unchanged").  The binaries find
# libnvcomp.so relative to themselves, so the tree can be moved after the build.  No-op without the nvCOMP tree.
set -u
R=${1:-${NVCOMP_REFERENCE_DIR:-}}
ROOT="$(cd "$(dirname "$0")/.." && pwd)"
[ -n "$R" ] && [ -d "$R/benchmarks" ] || { echo "nvCOMP tree not given or not found: skipping"; exit 0; }
mkdir -p "$ROOT/oracle/_ref"
cd "$ROOT/oracle/_ref"
NV="nvcc -gencode arch=compute_100a,code=sm_100a -std=c++17 -O2 -w -DTHRUST_CUB_WRAPPED_NAMESPACE=nvcomp \
  -I$ROOT/include -I$R/benchmarks -L$ROOT/nvcomp_b200/lib -lnvcomp -Xlinker -rpath=\$ORIGIN/../../nvcomp_b200/lib"
fail=0
build() { # name source [extra]
  if [ ! -x "$1" ] || [ "$2" -nt "$1" ] || [ "$ROOT/nvcomp_b200/lib/libnvcomp.so" -nt "$1" ]; then
    $NV -x cu "$2" -o "$1" > "$1.log" 2>&1 || { echo "FAILED: $1 (see oracle/_ref/$1.log)"; return 1; }
  fi
}
for f in lz4 snappy cascaded bitcomp ans gdeflate deflate zstd; do build benchmark_${f}_chunked $R/benchmarks/benchmark_${f}_chunked.cu & done
for f in benchmark_snappy_synth benchmark_lz4_synth benchmark_hlif; do build $f $R/benchmarks/$f.cpp & done
for f in low_level_quickstart_example high_level_quickstart_example; do build $f $R/examples/$f.cpp & done
# the LZ4 CPU-interop examples (known-answer tests of the wire format): liblz4.so.1 is on the image, its header is
# not -> prototype-only shim in tests/shim/
NV_SAVE="$NV"; NV="$NV -I$ROOT/tests/shim -I$R/examples -l:liblz4.so.1"
for f in lz4_cpu_compression lz4_cpu_decompression; do build $f $R/examples/$f.cu & done
wait
NV="$NV_SAVE"
wait
ls -1 | grep -v '\.log$' | wc -l
