#!/bin/bash
# One GPU session: parity tests (default "all" GPU tests), then stage timings for each given morphology band split.
#   tools/gpu_session.sh <tag> <tests|all|none> [bands ...]     (bands = "b55,b29" as LT_MORPH_BANDS, "-" = the launcher's own)
mkdir -p gpurun_out
tag=${1:-s}; tests=${2:-all}; shift; shift
if [ "$tests" = "all" ]; then
  timeout 1500 python -m pytest tests -m gpu -q -x > gpurun_out/${tag}_pytest.log 2>&1
  echo "pytest rc=$?" >> gpurun_out/${tag}_pytest.log
elif [ "$tests" != "none" ]; then
  timeout 1500 python -m pytest $tests -q -x > gpurun_out/${tag}_pytest.log 2>&1
  echo "pytest rc=$?" >> gpurun_out/${tag}_pytest.log
fi
tail -15 gpurun_out/${tag}_pytest.log
: > gpurun_out/${tag}_tool.log
for v in "$@"; do
  if [ "$v" = "-" ]; then unset LT_MORPH_BANDS; else export LT_MORPH_BANDS=$v; fi
  LT_BENCH_SYNTH=1 timeout 300 python tools/morph_bench.py --one >> gpurun_out/${tag}_tool.log 2>&1
done
cat gpurun_out/${tag}_tool.log
