#!/bin/sh
# CTA shape sweep of the 8-bit fused kernel (DESIGN.md 3.1): warps per CTA x ring stages of the reference-class, two-channel
# variant, each as its own library (tools/build_variant.sh), timed by tools/bench_u8.py --kernel-only beside the int16 and float
# variants of the same library.
#   tools/run_u8_sweep.sh OUT_DIR     (one JSON line per shape in OUT_DIR, a summary line per shape on stdout)
set -e
OUT=${1:?usage: tools/run_u8_sweep.sh OUT_DIR}
mkdir -p "$OUT"
OUT=$(cd "$OUT" && pwd)
cd "$(dirname "$0")/.."
for v in "w12s2 12 2" "w8s3 8 3" "w16s1 16 1" "w12s3 12 3" "w4s6 4 6"; do
  set -- $v
  lib=navtex_b200/variants/libnavtex_b200_u8_$1.so
  [ -f "$lib" ] || sh tools/build_variant.sh "u8_$1" "-DNVX_U8_WARPS_PER_CTA=$2 -DNVX_U8_STAGES=$3" > /dev/null
  NVX_LIB=$lib python tools/bench_u8.py --kernel-only --rounds 3 --steps 3 --out "$OUT/$1.json" > /dev/null
  python3 -c "import json,sys; r=json.load(open(sys.argv[1])); print(sys.argv[2], {f: round(r['kernel_ms'][f]['median'], 3) for f in r['kernel_ms']}, r['check'])" "$OUT/$1.json" "$1"
done
