#!/bin/bash
# Builds libdelly_b200.so (sm_100a only) in-tree. Used by __graft_entry__.build().
# Each .cu is compiled to an object in parallel (build/ is git-ignored), then linked.
set -e
cd "$(dirname "$0")"
NVCC=${NVCC:-/usr/local/cuda/bin/nvcc}
mkdir -p build
pids=()
objs=()
for src in delly_b200/csrc/*.cu; do
  obj=build/$(basename "${src%.cu}").o
  objs+=("$obj")
  # rebuild when the source or any shared header is newer than the object
  if [ ! -f "$obj" ] || [ "$src" -nt "$obj" ] || [ -n "$(find delly_b200/csrc include -name '*.cuh' -newer "$obj" -o -name '*.h' -newer "$obj")" ] || [ -n "${DGPU_EXTRA_FLAGS}" ]; then
    $NVCC -std=c++17 -O3 -lineinfo -gencode arch=compute_100a,code=sm_100a \
      -Xcompiler -fPIC -Xcompiler -Wall ${DGPU_EXTRA_FLAGS} -c -o "$obj" "$src" &
    pids+=($!)
  fi
done
for p in "${pids[@]}"; do wait "$p"; done
$NVCC -gencode arch=compute_100a,code=sm_100a -shared -o delly_b200/libdelly_b200.so "${objs[@]}" -lcudart
echo "built delly_b200/libdelly_b200.so"
# C++ host mirror of the reference interface (+ flat test hooks), linked against the CUDA library
g++ -std=c++17 -O2 -fPIC -shared -Wall -Wno-sign-compare -o delly_b200/libdelly_b200_host.so delly_b200/host/capi.cpp \
  -Ldelly_b200 -l:libdelly_b200.so -Wl,-rpath,'$ORIGIN'
echo "built delly_b200/libdelly_b200_host.so"
# the drop-in binding `delly_b200 sr|lr` (bindings/): htslib IO around the batched host mirrors. htslib = the reference's vendored submodule,
# compiled with its public headers into oracle/_ref/hts by tools/build_htslib.sh where the reference tree exists; elsewhere the archive and
# headers already under oracle/_ref/hts (built with the checkers) are used, as are the MEI templates extracted next to them.
bash tools/build_htslib.sh
python tools/extract_mei.py > /dev/null
HTS=oracle/_ref/hts
if [ -f $HTS/include/htslib/sam.h ] && [ -f $HTS/libhts.a ]; then
  mkdir -p delly_b200/bin
  g++ -std=c++17 -O2 -Wall -Wno-sign-compare -o delly_b200/bin/delly_b200 bindings/delly_b200_main.cpp -I$HTS/include \
    -Ldelly_b200 -l:libdelly_b200.so -Wl,-rpath,'$ORIGIN/..' $HTS/libhts.a -lz -lm -lpthread
  echo "built delly_b200/bin/delly_b200"
  # synthetic-sample generator for the pipeline benchmarks / whole-file parity tests (tools/simbam.cpp)
  g++ -std=c++17 -O2 -Wall -o delly_b200/bin/simbam tools/simbam.cpp -I$HTS/include $HTS/libhts.a -lz -lm -lpthread
  echo "built delly_b200/bin/simbam"
else
  echo "htslib (oracle/_ref/hts) not present; delly_b200/bin/delly_b200 not built" >&2
fi
