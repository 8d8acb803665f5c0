#!/bin/bash
CMD="python tools/bench_configs.py"
$CMD > gpurun_out/plain_panel.log 2>&1 && \
ncu --set full --clock-control none --import-source on -k regex:"trsm_tile_kernel|potrf_tile_pw_kernel" -s 20 -c 4 \
    -o gpurun_out/prof_panel -f $CMD > gpurun_out/ncu_panel.log 2>&1
tail -3 gpurun_out/ncu_panel.log
