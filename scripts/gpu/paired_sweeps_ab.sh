#!/bin/bash
# Paired sweeps against single sweeps (the STST_SINGLE_SWEEPS build of the workloads library) on one GPU.
#   ab       card and clocks, smoke(), Jacobi5 16384^2 alternating the two libraries, the dumped outputs
#            of both compared byte for byte
#   default  the default bench invocation once per library, the plan sweep of both libraries
# usage: paired_sweeps_ab.sh [ab|default|all] [output directory, default paired_sweeps_out]
# (no stage: both stages, one after the other)
stage=${1:-all}
out=${2:-paired_sweeps_out}; mkdir -p $out
single=libstst_workloads_single.so
[ -f stencilstream_b200/$single ] ||
  python -c "from stencilstream_b200 import _build; _build.build_variant('single', ['-DSTST_SINGLE_SWEEPS'])" > $out/build_variant.log 2>&1
lib_of() { [ $1 = single ] && echo $single; }

if [ $stage = ab ] || [ $stage = all ]; then
  nvidia-smi --query-gpu=name,power.limit,clocks.sm,clocks.max.sm --format=csv > $out/card.csv
  python -c "import __graft_entry__ as g; g.smoke()" > $out/smoke.log 2>&1; echo "smoke rc=$?" >> $out/smoke.log
  for rep in 1 2 3 4; do
    for arm in paired single; do
      STST_WORKLOADS_LIB=$(lib_of $arm) timeout 200 python bench.py --workload jacobi5 --steps 20 --warmup 3 \
        --no-cpu-baseline > $out/ab_jacobi5_${arm}_$rep.json 2> $out/ab_jacobi5_${arm}_$rep.err
    done
  done
  for arm in paired single; do
    STST_WORKLOADS_LIB=$(lib_of $arm) timeout 200 python bench.py --workload jacobi5 --steps 2 --warmup 1 \
      --no-cpu-baseline --dump-outputs $out/dump_$arm > /dev/null 2> $out/dump_$arm.err
  done
  (cd $out/dump_paired && ls && for f in *; do cmp "$f" ../dump_single/"$f" && echo "identical $f"; done) > $out/dump_compare.txt 2>&1
  rm -rf $out/dump_paired $out/dump_single
  cat $out/card.csv $out/smoke.log $out/dump_compare.txt
fi

if [ $stage = default ] || [ $stage = all ]; then
  for arm in paired single; do
    STST_WORKLOADS_LIB=$(lib_of $arm) timeout 400 python bench.py --steps 10 \
      > $out/bench_default_$arm.json 2> $out/bench_default_$arm.err
  done
  for arm in paired single; do
    STST_WORKLOADS_LIB=$(lib_of $arm) timeout 200 python scripts/sweep_plans.py --workload jacobi5 \
      --fuse 4,5,6,7,8,10 --ctas 1,2 --tile_rows 0,16,32 > $out/sweep_plans_$arm.log 2>&1
  done
  tail -c 300 $out/bench_default_paired.json
fi
