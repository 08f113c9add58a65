#!/bin/bash
# One GPU: the wide-context tests, the whole GPU suite, smoke(), bench.py cfg2 against a parent build of the library
# (build/ab/lib_parent.so with its capi.py, build/ab/capi_parent.py) alternated in this call, and
# scripts/time_wide.py.  WIDE_ONLY=1: the wide tests and time_wide.py; AB_ONLY=1: the bench A/B alone.  Outputs go to the
# directory OUT names (OUT=some/dir bash scripts/gpu_wide.sh).
: "${OUT:?set OUT to the output directory}"
mkdir -p "$OUT"
nvidia-smi --query-gpu=name,power.limit,clocks.max.sm --format=csv | tee $OUT/gpu.txt
python -c "import __graft_entry__ as g; g.build()" > $OUT/build.log 2>&1 || { tail -20 $OUT/build.log; exit 1; }
if [ -z "$AB_ONLY" ]; then
  timeout 900 python -m pytest tests/test_gpu_wide.py -q -rA -p no:cacheprovider > $OUT/wide_tests.log 2>&1
  echo "wide tests rc=$?"; grep -E "passed|failed|PASSED|FAILED|Error" $OUT/wide_tests.log | tail -25
fi
if [ -z "$WIDE_ONLY" ] && [ -z "$AB_ONLY" ]; then
  timeout 1200 python -m pytest tests/ -q -m gpu -p no:cacheprovider > $OUT/gpu_suite.log 2>&1
  echo "gpu suite rc=$?"; tail -3 $OUT/gpu_suite.log
  timeout 120 python -c "import __graft_entry__ as g; g.smoke()" 2>&1 | tail -2
fi
if [ -z "$WIDE_ONLY" ]; then
  lib=particlemdi.jl_b200/libpmdi_cuda.so capi=particlemdi.jl_b200/capi.py
  cp $lib /tmp/lib_branch.so; cp $capi /tmp/capi_branch.py
  for v in parent branch parent branch; do
    if [ $v = parent ]; then cp build/ab/lib_parent.so $lib; cp build/ab/capi_parent.py $capi
    else cp /tmp/lib_branch.so $lib; cp /tmp/capi_branch.py $capi; fi
    rm -rf $OUT/dump_$v
    timeout 400 python bench.py --gpus 1 --steps 10 --warmup 3 --no-cpu --no-cfg4 --no-pmdi --no-parity \
      --dump-outputs $OUT/dump_$v > $OUT/bench_$v.json 2> $OUT/bench_$v.err
    echo "bench $v rc=$? ms_per_step=$(python -c "import json;print(json.loads(open('$OUT/bench_$v.json').read().strip().split(chr(10))[-1])['ms_per_step'])")"
  done
  cp /tmp/lib_branch.so $lib; cp /tmp/capi_branch.py $capi
  python - <<'PY'
import os, numpy as np
a, b = "$OUT/dump_parent", "$OUT/dump_branch"
fa = sorted(os.listdir(a)) if os.path.isdir(a) else []
same = all(open(os.path.join(a, f), "rb").read() == open(os.path.join(b, f), "rb").read() for f in fa)
print("dumped outputs", len(fa), "files, parent == branch:", same)
PY
fi
[ -n "$AB_ONLY" ] && exit 0
timeout 1500 python scripts/time_wide.py $OUT/r08_wide.jsonl > $OUT/time_wide.log 2>&1; echo "time_wide rc=$?"
tail -4 $OUT/time_wide.log
