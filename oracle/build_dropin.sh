#!/bin/bash
# build_dropin.sh -- link the reference's UNMODIFIED host program against the B200 engine (oracle/Makefile, target `ref`).
#   oracle/_ref/kangaroo_b200     = reference main.cpp Kangaroo.cpp Check.cpp Thread.cpp Backup.cpp Network.cpp Merge.cpp
#                             PartMerge.cpp HashTable.cpp Timer.cpp SECPK1/*.cpp   (compiled where they lie, -DWITHGPU)
#                           + kangaroo_b200/csrc/GPUEngine_b200.cpp (replaces GPU/GPUEngine.cu) + libkgx.so
#   oracle/_ref/kangaroo_b200_sym = the same with -DUSE_SYMMETRY on every translation unit (the reference's compile-time
#                             switch, Constants.h:25): symmetric jump table / herd / CheckKey on the host, symmetric
#                             engine mode behind the shim (SURVEY 8f/f4)
#   oracle/_ref/kangaroo_b200_stats, oracle/_ref/kangaroo_b200_sym_stats = both again with the reference's -DSTATS
#   oracle/_ref/kgx_shim_bench    = shim_bench.cpp: end-to-end timing through `class GPUEngine` (bench.py's e2e leg)
# Needs the reference sources at $REF; nothing is copied into the repo.
set -e
REF=${REF:?set REF to the reference source tree}
ROOT=$(cd "$(dirname "$0")/.." && pwd)
HERE=$ROOT/kangaroo_b200/csrc
OUT=$ROOT/oracle/_ref
mkdir -p "$OUT"
[ -f "$HERE/libkgx.so" ] || { echo "build libkgx.so first (__graft_entry__.build())"; exit 1; }
BASEFLAGS="-O2 -m64 -mssse3 -Wno-unused-result -Wno-write-strings -include cstdint -DWITHGPU -I$REF"
SRC="main.cpp Kangaroo.cpp Check.cpp Thread.cpp Backup.cpp Network.cpp Merge.cpp PartMerge.cpp HashTable.cpp Timer.cpp \
     SECPK1/Int.cpp SECPK1/IntMod.cpp SECPK1/IntGroup.cpp SECPK1/Point.cpp SECPK1/SECP256K1.cpp SECPK1/Random.cpp"
LINK="-L$HERE -lkgx -lpthread -Wl,-rpath,\$ORIGIN/../../kangaroo_b200/csrc"

build_variant() {   # $1 = object tag, $2 = extra flags, $3 = output binary
  local tag=$1 flags="$BASEFLAGS $2" bin=$3 objs=""
  for f in $SRC; do
    o="$OUT/obj${tag}_$(echo $f | tr '/' '_' | sed 's/\.cpp$/.o/')"
    g++ $flags -c "$REF/$f" -o "$o" &
    objs="$objs $o"
  done
  g++ $flags -c "$HERE/GPUEngine_b200.cpp" -o "$OUT/obj${tag}_GPUEngine_b200.o" &
  wait
  g++ -o "$bin" $objs "$OUT/obj${tag}_GPUEngine_b200.o" $LINK
}

build_variant "" "" "$OUT/kangaroo_b200"
# end-to-end timing harness through the same class GPUEngine: shim + reference SECPK1 only
SECP_OBJS=$(for f in Int IntMod IntGroup Point SECP256K1 Random; do echo "$OUT/obj_SECPK1_$f.o"; done)
g++ $BASEFLAGS -o "$OUT/kgx_shim_bench" "$HERE/shim_bench.cpp" "$OUT/obj_GPUEngine_b200.o" $SECP_OBJS "$OUT/obj_Timer.o" $LINK
build_variant "S" "-DUSE_SYMMETRY" "$OUT/kangaroo_b200_sym"
# the reference's own statistics switch (Kangaroo.cpp:1010, 1058-1075: exact operation count per solved key, running average in
# units of sqrt(N)) -- used to measure the symmetry gain (tests/test_gpu_symmetry.py)
build_variant "T" "-DSTATS" "$OUT/kangaroo_b200_stats"
build_variant "U" "-DSTATS -DUSE_SYMMETRY" "$OUT/kangaroo_b200_sym_stats"
rm -f $OUT/obj*_*.o
echo "built $OUT/kangaroo_b200 $OUT/kangaroo_b200_sym $OUT/kgx_shim_bench"
