#!/bin/bash
# e2e leg of the headline workload: synchronous whole-batch calls against async sub-batches (B2_E2E_PARTS),
# (A, B) written straight into the mapped host buffers or staged in HBM and copied (B2_HOST_STAGED=1)
err=$(mktemp)  # bench.py's stderr of the last run
for cfg in "1 0" "2 0" "2 1" "3 1" "4 1"; do
  set -- $cfg
  for round in 1 2; do
  echo -n "parts=$1 staged=$2 r$round: "
  B2_E2E_PARTS=$1 B2_HOST_STAGED=$2 python bench.py --no-secondary --no-cpu-baseline --steps 50 2> "$err" | python -c "
import json,sys
d=json.loads(sys.stdin.read().strip().splitlines()[-1]); e=d['e2e']
print('e2e %.4g  ms %.4f  d2h GB/s %.1f  sync %s' % (e['value'], e['ms_per_step'], e['pcie_gbs_per_gpu']['d2h'], ('%.4g' % e['synchronous']['value']) if 'synchronous' in e else '-'))"
  done
done
tail -3 "$err"
rm -f "$err"
