#!/bin/bash
# e2e legs of every config (short device legs) + the request-level shapes of scratch/dense_ab.py
for c in ${CONFIGS:-cfg4 cfg2 cfg1 cfg3 cfg5}; do
  python bench.py --config $c --steps 3 --e2e-steps 8 --no-cpu --extras none 2>/dev/null | python -c "
import json,sys
d=json.loads(sys.stdin.readline()); e=d['e2e']; print('$c e2e %.0f best %.0f worst %.0f launches %d' % (e['value'], e['best'], e['worst'], e['kernel_launches_per_step']))"
done
python scratch/dense_ab.py 2>&1 | tail -4
