#!/bin/bash
# One B200 job for a frame-kernel change:  bash tools/gpu_job_mirror_ab.sh OUT_DIR
# Builds to compare go in as tools/ab/liblightpath_<name>.so (git-ignored); one of them is named "parent".
# Each is copied over _C/liblightpath.so in turn: the GPU suite and smoke run on every build but the parent,
# then the benchmark and the frame-kernel timings alternate all builds twice.  The card's name and power
# limit are recorded first; the dumped bench frames of every build must be byte-identical to the parent's.
OUT=${1:?output directory}
mkdir -p $OUT
LIB=light_path_tracer_b200/_C/liblightpath.so
DUMPS=$(mktemp -d)                  # (the dumped frames stay out of OUT_DIR: they are large)
trap 'rm -rf "$DUMPS"' EXIT
VARIANTS=$(ls tools/ab/liblightpath_*.so | sed 's#.*/liblightpath_##; s#\.so$##')
nvidia-smi --query-gpu=name,power.limit,clocks.max.sm --format=csv > $OUT/card.txt 2>&1; cat $OUT/card.txt
cp $LIB /tmp/lib_orig.so
for v in $VARIANTS; do
  [ "$v" = parent ] && continue
  cp tools/ab/liblightpath_$v.so $LIB
  timeout 900 python -m pytest tests -q -m gpu > $OUT/pytest_gpu_$v.log 2>&1; echo "pytest gpu $v rc=$?"; tail -2 $OUT/pytest_gpu_$v.log
  timeout 300 python -c "import __graft_entry__ as g; g.smoke()" > $OUT/smoke_$v.log 2>&1; echo "smoke $v rc=$?"; tail -1 $OUT/smoke_$v.log
done
for rep in 1 2; do for v in $VARIANTS; do
  cp tools/ab/liblightpath_$v.so $LIB
  timeout 600 python bench.py --gpus 1 --steps 50 --warmup 5 --no-cpu --dump-outputs $DUMPS/dump_${v}_$rep \
      > $OUT/bench_${v}_$rep.json 2> $OUT/bench_${v}_$rep.err
  echo "bench $v $rep rc=$?: $(python -c "import json,sys; d=json.loads(open(sys.argv[1]).read().strip().splitlines()[-1]); print(d['ms_per_step'], d['ms_per_step_median'])" $OUT/bench_${v}_$rep.json 2>&1)"
done; done
for rep in 1 2; do for v in $VARIANTS; do
  cp tools/ab/liblightpath_$v.so $LIB
  echo "$v: $(timeout 600 python tools/render_knob_perf.py LP_NONE default 2>&1 | tail -1)"
done; done > $OUT/render_perf.log 2>&1
cat $OUT/render_perf.log
cp /tmp/lib_orig.so $LIB
for rep in 1 2; do for v in $VARIANTS; do
  diff -r $DUMPS/dump_parent_$rep $DUMPS/dump_${v}_$rep > /dev/null && echo "dumps $v $rep identical to the parent's" || echo "dumps $v $rep DIFFER"
done; done
