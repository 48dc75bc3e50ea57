#!/bin/bash
# BASELINE config 2 (B4_highrate, KS3311, 24 images of 768x512: steps of at most 2304 rows): per-layer launches (default) vs
# the CTA-pair dataflow form for all steps (KS3311 has no single-CTA dataflow form)
mkdir -p gpurun_out
L=gpurun_out/r2_c2.log
: > $L
run() {
  echo "== $1" >> $L
  env $2 timeout 600 python bench.py --config B4_highrate --images 24 --steps 2 --warmup 2 --no-e2e --no-cpu-baseline --no-reference-container 2>> $L | python -c "
import json,sys
d=json.loads(sys.stdin.read()); print('value %.1f enc %.1f dec %.1f launches %d identical %s' % (d['value'], d['encode_mpix_s'], d['decode_mpix_s'], d['gpu_launches'], d['enc_dec_identical']))" >> $L
}
run "default" "LBIC_DUMMY=0"
run "CTA-pair dataflow for every step" "LBIC_FLOW=2"
run "no PDL" "LBIC_PDL=0"
cat $L
