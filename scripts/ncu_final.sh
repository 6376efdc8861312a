#!/bin/bash
# ncu --set full of every hot kernel at the bench workloads (C2 mesh, C5 mesh, C3 points) + launch lists; summaries are written
# under profiles/ by scripts/ncu_summary.py on the CPU box.
TAG=${1:-r3z}; OUT=gpurun_out; mkdir -p $OUT
ncu --set full --import-source on --clock-control none -k regex:"mesh_scatter_kernel|mesh_shade_kernel|mesh_backward_kernel|mesh_project_kernel" -s 4 -c 4 -f -o $OUT/${TAG}_mesh_c2 python scripts/one_step.py c2 2 > $OUT/${TAG}_ncu_c2.log 2>&1; tail -1 $OUT/${TAG}_ncu_c2.log
ncu --set full --import-source on --clock-control none -k regex:"mesh_scatter_kernel|mesh_shade_kernel|mesh_backward_kernel" -s 3 -c 3 -f -o $OUT/${TAG}_mesh_c5 python scripts/one_step.py c5 2 > $OUT/${TAG}_ncu_c5.log 2>&1; tail -1 $OUT/${TAG}_ncu_c5.log
ncu --metrics gpu__time_duration.sum --clock-control none -c 400 --csv --log-file $OUT/${TAG}_launches.csv python bench.py --steps 2 --warmup 1 --no-cpu-baseline --extras none > $OUT/${TAG}_b.log 2>&1; tail -1 $OUT/${TAG}_b.log | cut -c1-100
