#!/bin/bash
# quick GPU iteration: parity subset, then kernel timing (bench --short prints value only)
timeout 900 python -m pytest tests -m gpu -q -x -k "${1:-pg_kernel or one_sweep or multi_sweep or ragged or graph or variants or pg_moments or counters}" 2>&1 | tail -15
timeout 300 python bench.py --short --steps 50 --warmup 5 2>&1 | python -c "
import sys, json
for l in sys.stdin:
    l=l.strip()
    if l.startswith('{'):
        d=json.loads(l); print('value', round(d['value'],1), 'sweeps/s  ms/step', round(d['ms_per_step'],4), d['clocks'], (d.get('roofline') or {}).get('pg_deferred_frac'))
    elif l: print(l[:300])
"
