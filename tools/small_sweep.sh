#!/bin/bash
# lanes per env at the small / medium batch sizes: config 2 (4096 envs), config 3 (65536 envs, 42 rooms), the 8-GPU shard (131072)
for l in $1; do
  for spec in "c2 0" "c3 0" "c4 131072" "c4 262144"; do set -- $spec
    python bench.py --workload $1 --envs $2 --lanes $l --steps 1500 --warmup 100 --no-extras --e2e-steps 3 2>/dev/null | python -c "
import json,sys; d=json.loads(sys.stdin.read()); print('lanes $l', '$1', d['config']['envs_total'], '%.2f us/step' % (d['ms_per_step']*1e3), '%.3g steps/s' % d['value'], 'frac %.3f' % d['roofline']['frac'])"
  done
done
