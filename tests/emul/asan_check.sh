#!/bin/bash
# TEST INFRASTRUCTURE ONLY: memory and alignment check of the kernel logic without a GPU.  Builds the emulator library
# with -fsanitize=address and -fsanitize=alignment into a scratch directory, points the loader at it and runs a driver:
# the script given as the first argument (tests/emul/asan_driver.py by default), with the remaining arguments.
# (compute-sanitizer is not available on the GPU pool; this catches the same class of indexing bugs on the host, and a
# vector load from an address its type does not allow, which is a misaligned-address fault on the device.  cuda_emul.h
# gives float2 / float4 / double2 their CUDA alignments, so the check sees what the device would.)
set -e
here="$(cd "$(dirname "$0")" && pwd)"
src="$here/../../quantum_inferno_b200/csrc"
out="${TMPDIR:-/tmp}/qi_emul_asan"
driver="${1:-$here/asan_driver.py}"
[ $# -gt 0 ] && shift
san="-fsanitize=address -fsanitize=alignment -fno-sanitize-recover=alignment"
mkdir -p "$out"
# an object is rebuilt when it is missing or older than its source or any header (a second run in the same scratch
# directory, e.g. after a sanitizer abort, only relinks)
stale() {
  [ ! -f "$2" ] || [ "$1" -nt "$2" ] || \
    [ -n "$(find "$src" "$here" -maxdepth 1 \( -name '*.cuh' -o -name '*.h' \) -newer "$2")" ]
}
pids=""
for f in "$src"/*.cu; do
  o="$out/$(basename "$f" .cu).o"
  if stale "$f" "$o"; then
    g++ -std=c++17 -O1 -g -fPIC $san -fno-omit-frame-pointer -DQI_EMUL -I"$here" -I"$src" -x c++ -c "$f" -o "$o" &
    pids="$pids $!"
  fi
done
if stale "$here/cuda_emul.cpp" "$out/cuda_emul.o"; then
  g++ -std=c++17 -O1 -g -fPIC $san -fno-omit-frame-pointer -DQI_EMUL -I"$here" -c "$here/cuda_emul.cpp" -o "$out/cuda_emul.o" &
  pids="$pids $!"
fi
for p in $pids; do wait "$p"; done
g++ -shared $san -o "$out/libqi_emul.so" "$out"/*.o -lpthread
QI_EMUL_LIB="$out/libqi_emul.so" ASAN_OPTIONS=detect_leaks=0:detect_stack_use_after_return=0:halt_on_error=1 \
  UBSAN_OPTIONS=print_stacktrace=1 LD_PRELOAD="$(gcc -print-file-name=libasan.so)" python "$driver" "$@"
