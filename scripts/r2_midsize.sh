#!/bin/bash
# mid-size batches (128 / 256 images per GPU: steps of 6-12 k rows, not power capped): CTA-pair dataflow (default) vs the
# single-CTA dataflow form with 128 x 96 tiles (twice the tiles per worker) vs per-layer launches
mkdir -p gpurun_out
L=gpurun_out/r2_midsize.log
: > $L
run() {
  echo "== $1 images=$2" >> $L
  env $3 timeout 600 python bench.py --images $2 --steps 3 --warmup 3 --no-e2e --no-cpu-baseline --no-reference-container 2>> $L | python -c "
import json,sys
d=json.loads(sys.stdin.read()); print('value %.1f enc %.1f dec %.1f sm_mhz %s' % (d['value'], d['encode_mpix_s'], d['decode_mpix_s'], d['clocks']['sm_mhz']))" >> $L
}
for n in 128 256 512; do
  run "pair dataflow (default)" $n "LBIC_DUMMY=0"
  run "single-CTA dataflow below 16384 rows" $n "LBIC_FLOW_MIN_ROWS=1 LBIC_FLOW_PAIR_MIN_ROWS=16384"
  run "per-layer launches" $n "LBIC_FLOW=0"
done
cat $L
