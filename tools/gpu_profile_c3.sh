#!/bin/bash
# ncu --set full of the head-of-pass launch of C3's two largest kernels (generic photon gather, pair connections).
tag=${1:-r1b}
mkdir -p gpurun_out
for k in k_camera_merge_closure k_camera_connect; do
  timeout 400 ncu --set full --clock-control none --import-source on -k regex:$k -s 2 -c 1 -f -o /tmp/p3_$k python tools/profile_run.py C3 1 > gpurun_out/${tag}_ncu_full_c3_$k.log 2>&1
  if [ -f /tmp/p3_$k.ncu-rep ]; then
    ncu -i /tmp/p3_$k.ncu-rep --page raw --csv > gpurun_out/${tag}_c3_$k.raw.csv 2>/dev/null
  fi
done
ls -la gpurun_out | grep c3_k
exit 0
