#!/bin/bash
# A/B of two builds of the library for the config-2 step, in one call on one box (r3_ab_grid2_column_map.txt,
# r3_ab_grid2_pack.txt):
#   bash profiles/tools/ab_grid2_column_map.sh OUT_DIR
# expects generative-physics-informed-pde_b200/build/libPARENT.so (reference build) and build/libNEW.so (variant).
# Card and power limit, alternating bench.py runs (config 2 with its sub-records, then config 1), the step's outputs of
# both builds, and the profiler times of the packing and residual kernels.
OUT=${1:?usage: ab_grid2_column_map.sh OUT_DIR}
mkdir -p $OUT
PKG=generative-physics-informed-pde_b200
nvidia-smi --query-gpu=name,power.limit,clocks.max.sm --format=csv > $OUT/gpu.txt
use() { cp $PKG/build/lib$1.so $PKG/libgpde_b200.so; }
for i in 1 2 3 4 5; do
  for v in PARENT NEW; do
    use $v; timeout 600 python bench.py --gpus 1 --no-cpu-baseline --no-e2e 2>$OUT/bench_err_$v.txt | tail -1 | sed "s/^/$v /" >> $OUT/bench_cfg2.txt
  done
done
for i in 1 2 3; do
  for v in PARENT NEW; do
    use $v; timeout 300 python bench.py --gpus 1 --workload cfg1 --no-sub --no-cpu-baseline --no-e2e 2>>$OUT/bench_err_$v.txt | tail -1 | sed "s/^/$v /" >> $OUT/bench_cfg1.txt
  done
done
for v in PARENT NEW; do
  use $v; timeout 600 python bench.py --gpus 1 --no-sub --no-cpu-baseline --no-e2e --dump-outputs $OUT/dump_$v > /dev/null 2>>$OUT/bench_err_$v.txt
  timeout 300 python profiles/tools/time_grid2_column_map.py --iters 200 2>&1 | tail -1 | sed "s/^/$v /" >> $OUT/kernel_times.txt
done
use NEW
