#!/bin/bash
# One GPU: the spec engine's resampling event.  tests/test_gpu_spec_resample.py; bench.py cfg2 with a parent build
# of the library (build/ab/lib_parent.so, copied there by hand) and this build alternated, their dumped outputs
# compared; time_resample.py on cfg2 and cfg4 with both builds (lines in $OUT/r09_resample.jsonl); then the whole
# GPU suite and smoke().  Outputs go to the directory OUT names.
: "${OUT:?set OUT to the output directory}"
mkdir -p "$OUT"
nvidia-smi --query-gpu=name,power.limit,clocks.max.sm --format=csv | tee $OUT/gpu.txt
python -c "import __graft_entry__ as g; g.build()" > $OUT/build.log 2>&1 || { tail -20 $OUT/build.log; exit 1; }
timeout 600 python -m pytest tests/test_gpu_spec_resample.py -q -rA -p no:cacheprovider > $OUT/resample_tests.log 2>&1
echo "resample tests rc=$?"; grep -E "passed|failed|PASSED|FAILED|Error" $OUT/resample_tests.log | tail -12
lib=particlemdi.jl_b200/libpmdi_cuda.so
cp $lib /tmp/lib_branch.so
for v in parent branch parent branch; do
  if [ $v = parent ]; then cp build/ab/lib_parent.so $lib; else cp /tmp/lib_branch.so $lib; fi
  rm -rf $OUT/dump_$v
  timeout 400 python bench.py --gpus 1 --steps 10 --warmup 3 --no-cpu --no-cfg4 --no-pmdi --no-parity \
    --dump-outputs $OUT/dump_$v >> $OUT/bench_$v.json 2> $OUT/bench_$v.err
  echo "bench $v rc=$? ms_per_step=$(python -c "import json;print(json.loads(open('$OUT/bench_$v.json').read().strip().split(chr(10))[-1])['ms_per_step'])")"
done
OUT=$OUT python - <<'PY'
import os
a, b = os.environ["OUT"] + "/dump_parent", os.environ["OUT"] + "/dump_branch"
fa = sorted(os.listdir(a)) if os.path.isdir(a) else []
same = all(open(os.path.join(a, f), "rb").read() == open(os.path.join(b, f), "rb").read() for f in fa)
print("dumped outputs", len(fa), "files, parent == branch:", same)
PY
for cfg in "cfg2_multiomics 40" "cfg4_singlecell 14"; do
  for v in parent branch; do
    if [ $v = parent ]; then cp build/ab/lib_parent.so $lib; else cp /tmp/lib_branch.so $lib; fi
    echo "{\"build\": \"$v\"}" >> $OUT/r09_resample.jsonl
    timeout 600 python scripts/time_resample.py $cfg $OUT/r09_resample.jsonl > $OUT/tr_${v}_${cfg%% *}.log 2>&1
    echo "time_resample $v $cfg rc=$?"; tail -1 $OUT/tr_${v}_${cfg%% *}.log
  done
done
# parent builds with other sub-phases in the timer slots (build/ab/lib_parent_t*.so: scripts/ab/resample_breakdown.py), if present
for f in build/ab/lib_parent_t*.so; do
  [ -e "$f" ] || continue
  v=$(basename $f .so); cp $f $lib
  echo "{\"build\": \"$v\"}" >> $OUT/r09_breakdown.jsonl
  timeout 300 python scripts/time_resample.py cfg2_multiomics 30 $OUT/r09_breakdown.jsonl > $OUT/tr_$v.log 2>&1
  echo "time_resample $v rc=$?"; tail -1 $OUT/tr_$v.log
done
cp /tmp/lib_branch.so $lib
timeout 1500 python -m pytest tests/ -q -m gpu -p no:cacheprovider > $OUT/gpu_suite.log 2>&1
echo "gpu suite rc=$?"; tail -3 $OUT/gpu_suite.log
timeout 120 python -c "import __graft_entry__ as g; g.smoke()" 2>&1 | tail -2
