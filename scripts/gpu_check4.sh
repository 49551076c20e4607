#!/bin/bash
set -x
OUT=${OUT:-out}  # output directory (git-ignored)
mkdir -p "$OUT"
TAG=${1:-r2d}
timeout 900 python -m pytest tests -m gpu -q -x -rs 2>&1 | tail -8 > $OUT/${TAG}_pytest_gpu.txt
cat $OUT/${TAG}_pytest_gpu.txt
VRG_VERBOSE=1 timeout 300 python scripts/sweep_time.py 82x880x880 640x880x880 > $OUT/${TAG}_sweep_time.jsonl 2> $OUT/${TAG}_sweep_time.err
cat $OUT/${TAG}_sweep_time.jsonl; tail -n 5 $OUT/${TAG}_sweep_time.err
