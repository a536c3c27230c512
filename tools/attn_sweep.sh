#!/bin/bash
# usage: tools/attn_sweep.sh [LOG]  (default build/attn_sweep.log) ; each attention shape in its own process + timeout, then
# the per-row kernel tests against the fp64 reference (slow paths included); prints every line that is not an OK
cd "$(dirname "$0")/.."
L=${1:-build/attn_sweep.log}
mkdir -p "$(dirname "$L")"
: > $L
for shp in "2 17 2" "3 128 4" "2 160 3" "4 197 12" "2 256 3" "3 288 5" "2 300 3" "3 320 12" "32 320 12 time" "32 320 16 time"; do
  echo "=== $shp" >> $L
  timeout 90 python tools/attn_bwd_check.py $shp >> $L 2>&1
  echo "rc=$?" >> $L
done
echo "=== tests/test_attention_kernels_gpu.py" >> $L
timeout 600 python -m pytest -q -m gpu tests/test_attention_kernels_gpu.py >> $L 2>&1
echo "rc=$?" >> $L
grep -v " OK$" $L
