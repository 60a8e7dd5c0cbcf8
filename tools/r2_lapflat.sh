#!/bin/bash
# thread-per-level laplacians: parity, then the pipeline-shape variants and the grid size in waves
set -u
OUT=gpurun_out
timeout 900 python -m pytest tests/test_parity_gpu.py -q -m gpu -k "weak_form or biharmonic or linear" > $OUT/lf_pytest.log 2>&1; echo "pytest rc=$?" >> $OUT/lf_pytest.log
: > $OUT/lf_bench.jsonl
run() { echo "# $*" >> $OUT/lf_bench.jsonl; timeout 300 "$@" >> $OUT/lf_bench.jsonl 2>> $OUT/lf_bench.err; }
for L in 72 128 30; do
  run python tools/levelop_bench.py --ops lap,lapt --modes fast --nlev $L
done
for W in 2 4; do
  CAAR_LEVELOP_WAVES=$W run python tools/levelop_bench.py --ops lap,lapt --modes fast --nlev 72
  echo "# ^ waves=$W" >> $OUT/lf_bench.jsonl
done
for v in a b c d; do
  for L in 72 128; do
    run python tools/levelop_bench.py --ops lap,lapt --modes fast --nlev $L --lib tools/_variants/libcaar_b200_lf_$v.so
  done
done
CAAR_LEVELOP_WAVES=2 run python tools/levelop_bench.py --ops lap,lapt --modes fast --nlev 72 --lib tools/_variants/libcaar_b200_lf_c.so
echo "# ^ c waves=2" >> $OUT/lf_bench.jsonl
