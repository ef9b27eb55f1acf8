#!/bin/bash
# host-pointer path: tests, traces, e2e numbers for the default schedule and two first-section sizes
mkdir -p gpurun_out
O=gpurun_out
timeout 900 python -m pytest tests -m gpu -x -q > $O/h_pytest_gpu.log 2>&1
echo "pytest rc=$?" >> $O/h_pytest_gpu.log
tail -4 $O/h_pytest_gpu.log
python tools/host_trace.py 10 2>&1 | tail -45
for knobs in "" "TCAMCRF_HOST_SECTION0=2" "TCAMCRF_HOST_SECTION0=8"; do
  for k in 10 2; do
  env $knobs python bench.py --no-cpu-baseline --no-extra --steps 20 --warmup 5 --e2e-steps 50 --classes $k 2>/dev/null | python -c "
import json,sys; d=json.loads(sys.stdin.read()); e=d['e2e']; print('${knobs:-default} K=$k', 'e2e', round(e['value']), 'ms', round(e['ms_per_step'],3), 'link', round(e['link_bound_ms'],3), 'frac', round(e['frac_of_link'],3), 'trainer_u8', round(d['e2e_trainer']['value']))"
  done
done
