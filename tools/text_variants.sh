#!/bin/bash
# A/B of text-kernel build variants on the k = 2 edit workload (each variant is compiled on the box: the fingerprint includes the flags)
for v in "" "-DFMB_TEXT_MINB=3" "-DFMB_TEXT_MINB=5" "-DFMB_TEXT_MINB=2"; do
  echo "== variant [$v]"
  FMB_NVCC_EXTRA="$v" python tools/scheme_trace.py 3e9 1e7 2 1 2>&1 | grep "^k="
  FMB_NVCC_EXTRA="$v" python tools/scheme_trace.py 3e9 1e7 1 1 2>&1 | grep "^k="
done
