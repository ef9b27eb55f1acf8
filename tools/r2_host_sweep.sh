#!/bin/bash
# host-pointer path: e2e for section / group schedules (K=10 and K=2)
mkdir -p gpurun_out
run() {
  for k in $KS; do
  env $1 python bench.py --no-cpu-baseline --no-extra --steps 20 --warmup 5 --e2e-steps 60 --classes $k 2>/dev/null | python -c "
import json,sys; d=json.loads(sys.stdin.read()); e=d['e2e']; print('$1 K=$k', 'e2e', round(e['value']), 'ms', round(e['ms_per_step'],3), 'link', round(e['link_bound_ms'],3), 'frac', round(e['frac_of_link'],3))"
  done
}
KS="10"
for s0 in 2 4; do for grow in 1 2 3; do for groups in 8 16; do
  run "TCAMCRF_HOST_SECTION0=$s0 TCAMCRF_HOST_GROW=$grow TCAMCRF_HOST_GROUPS=$groups"
done; done; done
run "TCAMCRF_HOST_SECTION0=8 TCAMCRF_HOST_GROW=1 TCAMCRF_HOST_GROUPS=8"
run "TCAMCRF_HOST_SECTION0=8 TCAMCRF_HOST_GROW=1 TCAMCRF_HOST_GROUPS=16"
run "TCAMCRF_HOST_SECTION0=1 TCAMCRF_HOST_GROW=2 TCAMCRF_HOST_GROUPS=16"
KS="2"
for s0 in 4 8 16; do for grow in 1 2; do for groups in 2 4 8; do
  run "TCAMCRF_HOST_SECTION0=$s0 TCAMCRF_HOST_GROW=$grow TCAMCRF_HOST_GROUPS=$groups"
done; done; done
