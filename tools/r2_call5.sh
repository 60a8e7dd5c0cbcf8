#!/bin/bash
set -u
OUT=gpurun_out
mkdir -p $OUT
timeout 900 python -m pytest tests/test_parity_gpu.py -m gpu -x -q -k "euler_step or weak_form or biharmonic" > $OUT/r2e_pytest.log 2>&1
echo "pytest rc=$?" >> $OUT/r2e_pytest.log
{
for q in 1 4 8; do timeout 300 python tools/levelop_bench.py --nelem 21600 --nlev 72 --qsize $q --ops euler --modes fast; done
timeout 300 python tools/levelop_bench.py --nelem 2700 --nlev 72 --qsize 35 --ops euler --modes fast
timeout 300 python tools/levelop_bench.py --nelem 10800 --nlev 128 --qsize 8 --ops euler --modes fast
timeout 300 python tools/levelop_bench.py --nelem 43200 --nlev 72 --qsize 1 --ops divwk,lap,lapt
timeout 300 python tools/levelop_bench.py --nelem 43200 --nlev 30 --qsize 1 --ops lap --modes fast
CAAR_LEVELOP_WAVES=1 timeout 300 python tools/levelop_bench.py --nelem 21600 --nlev 72 --qsize 4 --ops euler,lap --modes fast
CAAR_LEVELOP_WAVES=4 timeout 300 python tools/levelop_bench.py --nelem 21600 --nlev 72 --qsize 4 --ops euler,lap --modes fast
} > $OUT/r2e_levelops.log 2>&1
