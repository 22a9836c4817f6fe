#!/bin/bash
# Experiment builds of one kernel file (default: the forward, csrc/attn_fwd_tc.cu; VARIANT_SRC=attn_bwd_tc for another): compiles
# it with extra -D flags and links it with the other objects of the current library into lib_variants/<name>/libMFAFFI.so
# (select with MFA_LIBRARY=...).
#   VARIANT_SRC=attn_bwd_tc scripts/build_variant.sh bwd_ra2_rb2 -DMFA_BWD_RA=2 -DMFA_BWD_RB=2
set -e
NAME=$1; shift
HERE=$(cd "$(dirname "$0")/.." && pwd)
PKG="$HERE/universal-metal-flash-attention_b200"
OUT="$HERE/lib_variants/$NAME"; mkdir -p "$OUT"
FLAGS="-gencode arch=compute_100a,code=sm_100a -O3 -std=c++17 -lineinfo --cudart static -Xcompiler -fPIC,-O3 --expt-relaxed-constexpr -ccbin /usr/bin/g++"
grep -q MFA_MBAR_WATCHDOG "$PKG/lib/build_flags.txt" 2>/dev/null && FLAGS="$FLAGS -DMFA_MBAR_WATCHDOG"
SRC=${VARIANT_SRC:-attn_fwd_tc}
nvcc $FLAGS "$@" -c "$PKG/csrc/$SRC.cu" -o "$OUT/$SRC.o" 2>&1 | grep -v deprecated || true
OBJS=$(ls "$PKG"/lib/*.o | grep -v "/$SRC.o")
nvcc -shared --cudart static -ccbin /usr/bin/g++ -o "$OUT/libMFAFFI.so" "$OUT/$SRC.o" $OBJS -ldl -lpthread -lrt -Xlinker --version-script="$PKG/csrc/exports.map" 2>&1 | grep -v deprecated || true
rm -f "$OUT/$SRC.o"
ls -la "$OUT/libMFAFFI.so"
