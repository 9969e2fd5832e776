#!/bin/bash
# Builds variant libraries next to the default one, for A/B measurements on the GPU box (select with PTAP_LIB=<path>):
#   pathtracerap_b200/variants/libptap_ctas7.so    PTAP_TRACE_MIN_CTAS=7: k_trace_bvh compiled for 7 resident CTAs per SM instead of 8
# usage: tools/build_variants.sh [name=flags ...]      e.g.  tools/build_variants.sh ctas7=-DPTAP_TRACE_MIN_CTAS=7
set -euo pipefail
ROOT="$(cd "$(dirname "$0")/.." && pwd)"
[ $# -gt 0 ] || set -- "ctas7=-DPTAP_TRACE_MIN_CTAS=7"
mkdir -p "$ROOT/pathtracerap_b200/variants"
for spec in "$@"; do
  name="${spec%%=*}"; flags="${spec#*=}"
  TMP=$(mktemp -d /tmp/ptap_variant.XXXXXX)
  mkdir -p "$TMP/pathtracerap_b200" "$TMP/include"
  cp -r "$ROOT/pathtracerap_b200/csrc" "$TMP/pathtracerap_b200/csrc"; cp "$ROOT/include/ptap.h" "$TMP/include/"
  rm -f "$TMP"/pathtracerap_b200/csrc/*.o
  # both compilers must see the flag: the host builder and the kernels share device_types.h
  make -s -C "$TMP/pathtracerap_b200/csrc" EXTRA="$flags" CXXFLAGS="-O2 -std=c++17 -fPIC -ffp-contract=off -Wall -I/usr/local/cuda/include $flags" OUT="$ROOT/pathtracerap_b200/variants/libptap_$name.so"
  rm -rf "$TMP"
  echo "built pathtracerap_b200/variants/libptap_$name.so ($flags)"
done
