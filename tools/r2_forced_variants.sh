#!/bin/bash
# The whole GPU suite with each kernel variant FORCED for every call (the density hint normally picks): a stand-in for
# the sanitizer runs this pool refuses -- every parity test then exercises the forced kernel on every input.
mkdir -p gpurun_out
O=gpurun_out
: > $O/forced_variants.log
for knobs in "TCAMCRF_BUILD_DEDUP=1" "TCAMCRF_BUILD_DEDUP=0" "TCAMCRF_DENSE=1" "TCAMCRF_DENSE=0" "TCAMCRF_BUILD_DEDUP=1 TCAMCRF_DENSE=1" "TCAMCRF_BUILD_DEDUP=0 TCAMCRF_DENSE=0"; do
  echo "== $knobs" >> $O/forced_variants.log
  env $knobs timeout 900 python -m pytest tests -m gpu -q -p no:cacheprovider 2>&1 | tail -4 >> $O/forced_variants.log
done
cat $O/forced_variants.log
