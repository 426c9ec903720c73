#!/usr/bin/env bash
# TEST INFRASTRUCTURE — builds oracle/_ref/libfsr1_ref.so from the reference's own sources where
# FSR1_REFERENCE_DIR names a checkout of GPUOpen-Effects/FidelityFX-FSR (SURVEY.md §8(c), Appendix A).
# Nothing from the reference is copied into the repo: the rewritten headers live in a mktemp directory
# that is deleted, and the only output is the shared library under oracle/_ref/ (git-ignored).
#
# The rewrite is purely mechanical (HLSL parameter qualifiers -> C++):
#   inout AXn name -> AXn& name ; out AXn name -> AXn& name ; in AXn name -> AXn name
#   and the three AZolZeroPassF{2,3,4} helpers (vector ?: — inexpressible in C++, unused by FSR1) removed.
set -euo pipefail
HERE="$(cd "$(dirname "${BASH_SOURCE[0]}")" && pwd)"
REF="${FSR1_REFERENCE_DIR:-}/ffx-fsr"
OUT="$HERE/_ref"
if [ -z "${FSR1_REFERENCE_DIR:-}" ] || [ ! -f "$REF/ffx_fsr1.h" ]; then
  echo "build_ref: FSR1_REFERENCE_DIR does not name a reference checkout — keeping $OUT as it is (without it the tests compare with the stored digests only)" >&2
  exit 0
fi
mkdir -p "$OUT"
TMP="$(mktemp -d)"
trap 'rm -rf "$TMP"' EXIT
for f in ffx_a.h ffx_fsr1.h; do
  sed -E -e 's/\binout +(A[A-Z]+[0-9])\b/\1\&/g' \
         -e 's/\bout +(A[A-Z]+[0-9])\b/\1\&/g' \
         -e 's/\bin +(A[A-Z]+[0-9])\b/\1/g' \
         -e '/AZolZeroPass[FH][234]\(/d' "$REF/$f" > "$TMP/$f"
done
CXXFLAGS="-std=c++17 -O2 -fPIC -w -fopenmp -ffp-contract=off -I$HERE/shim -I$TMP"
# A_CPU constants from the UNMODIFIED headers.
gcc -std=c11 -O2 -fPIC -w -ffp-contract=off -I"$REF" -c "$HERE/ref_cpu.c" -o "$TMP/ref_cpu.o"
if g++ $CXXFLAGS -DFSR1_REF_HALF -fexcess-precision=16 -c "$HERE/ref_driver.cpp" -o "$TMP/ref_driver.o" 2>"$TMP/half.err"; then
  echo "build_ref: fp32 + packed-half reference paths compiled"
else
  echo "build_ref: packed-half path did not compile (see below); building fp32 only" >&2
  head -30 "$TMP/half.err" >&2
  g++ $CXXFLAGS -c "$HERE/ref_driver.cpp" -o "$TMP/ref_driver.o"
fi
# the reference's compile-time RCAS options (ffx_fsr1.h:647-651), each as its own namespaced variant
VARIANTS=""
HALFFLAGS=""
if [ ! -s "$TMP/half.err" ]; then HALFFLAGS="-DFSR1_REF_HALF -fexcess-precision=16"; fi
for v in "dn:-DFSR_RCAS_DENOISE=1" "pa:-DFSR_RCAS_PASSTHROUGH_ALPHA=1" "dnpa:-DFSR_RCAS_DENOISE=1 -DFSR_RCAS_PASSTHROUGH_ALPHA=1"; do
  tag="${v%%:*}"; defs="${v#*:}"
  g++ $CXXFLAGS $HALFFLAGS $defs -DREFNS=fsr1ref_$tag -DREFSUF=_$tag -c "$HERE/ref_driver.cpp" -o "$TMP/ref_driver_$tag.o"
  VARIANTS="$VARIANTS $TMP/ref_driver_$tag.o"
done
g++ -shared -fopenmp -o "$OUT/libfsr1_ref.so" "$TMP/ref_driver.o" $VARIANTS "$TMP/ref_cpu.o" -lm
echo "build_ref: wrote $OUT/libfsr1_ref.so"
