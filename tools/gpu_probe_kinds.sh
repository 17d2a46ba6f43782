#!/bin/bash
# Exactness of the tcgen05 search in every configuration the library runs: the probe dumps every accumulator and
# compares it with CPU integers and the winners with the direct search (B = 4, 8, 16; kind::i8 and kind::f16 where
# they exist; CTA pairs off and on where they exist; patterns 1 = structured, 3 = binary 0/255 noise, 4 = binary
# 0/255 cells), then the GPU test suite.  Run from the repository root after a build with the probe
# (python fractal-image-compression_b200/build.py --probe).  Exit code 0 only if everything passed.
# Usage: tools/gpu_probe_kinds.sh [log directory]   (default: a new temporary directory)
OUT=${1:-$(mktemp -d)}
mkdir -p "$OUT"
echo "logs in $OUT"
P=fractal-image-compression_b200/lib/umma_probe
fail=0
# "B W kind pair": kind 1 = kind::i8, 2 = kind::f16; pair 0 = auto (kernels without a pair form), 1 = off, 2 = on
for cfg in "4 256 1 0" "4 256 2 1" "4 256 2 2" "8 256 1 0" "8 256 2 1" "8 256 2 2" "16 512 1 1" "16 512 1 2"; do
  set -- $cfg
  for pattern in 1 3 4; do
    log=$OUT/probe_B$1_k$3_p$4_pat$pattern.log
    timeout 300 $P check $1 $2 $pattern $3 $4 > "$log" 2>&1
    rc=$?
    echo "== check B=$1 W=$2 pattern=$pattern kind=$3 pair=$4: rc=$rc"
    grep -E "pairs=|accumulator check|winner check|PROBE|rror" "$log" | head -5
    [ $rc -eq 0 ] || fail=1
  done
done
echo "== pytest -m gpu =="
timeout 1500 python -m pytest tests -m gpu -q > "$OUT/pytest_gpu.log" 2>&1
rc=$?
echo "rc=$rc"; tail -5 "$OUT/pytest_gpu.log"
[ $rc -eq 0 ] || fail=1
exit $fail
