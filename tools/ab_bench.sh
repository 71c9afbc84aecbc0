#!/bin/bash
# A/B timing of library variants on the same GPU box: [CONFIG=c3] tools/ab_bench.sh ab/libA.so ab/libB.so ...
# (each variant is selected through DVBT2LL_LIB and bench.py is run; variants are alternated twice)
for round in 1 2; do
  for v in "$@"; do
    DVBT2LL_LIB=$PWD/$v python bench.py --config ${CONFIG:-c3} --channels ${CHANNELS:-64} --steps 30 --warmup 5 --no-cpu-baseline --no-extras --no-parity --e2e-steps 1 2>&1 | tail -1 | python -c "
import json,sys
try:
    d=json.loads(sys.stdin.read()); s=d['roofline']['stage_ms']
    print('$v', round(d['ms_per_step'],4), {k:round(x,4) for k,x in s.items()})
except Exception as e:
    print('$v', 'FAILED', e)"
  done
done
