#!/usr/bin/env bash
# One GPU-box visit (round 2).  usage: bash tools/visit.sh <tag> [tests] [issue] [bench] [bench_tf32] [launches_tf32] [launches_fp32] [cfg3] [cfg4]
set -u
OUT=gpurun_out; mkdir -p $OUT; TAG=${1:-r02}; shift || true
for w in "$@"; do
  case $w in
    tests)
      timeout -k 5 1500 python -m pytest tests -m gpu -q -s > $OUT/pytest_$TAG.log 2>&1; echo "pytest exit $?"; grep -E " passed| failed| error" $OUT/pytest_$TAG.log | tail -3
      grep -E "^FAILED|^E  +Assertion" $OUT/pytest_$TAG.log | cut -c1-260 | head -30;;
    issue)
      rm -f $OUT/issue_$TAG.log
      for shape in "1 3 tf32" "48 3 tf32" "16 7 tf32" "1 3 fp32" "48 3 fp32"; do timeout -k 5 300 python tools/issue_time.py $shape >> $OUT/issue_$TAG.log 2>&1; done; grep -E "False both|GRAPH replay both" $OUT/issue_$TAG.log;;
    bench)
      timeout -k 5 900 python bench.py > $OUT/bench_$TAG.json 2> $OUT/bench_$TAG.err; echo "bench exit $?"; cut -c1-330 $OUT/bench_$TAG.json; tail -3 $OUT/bench_$TAG.err;;
    bench_tf32)
      timeout -k 5 900 python bench.py --precision tf32 --no-cpu-baseline --no-gpu-baseline > $OUT/bench_tf32_$TAG.json 2> $OUT/bench_tf32_$TAG.err; echo "bench tf32 exit $?"; cut -c1-330 $OUT/bench_tf32_$TAG.json;;
    cfg3)
      timeout -k 5 900 python bench.py --config 3 --no-cpu-baseline > $OUT/bench_cfg3_$TAG.json 2> $OUT/bench_cfg3_$TAG.err; echo "bench cfg3 exit $?"; cut -c1-330 $OUT/bench_cfg3_$TAG.json;;
    cfg4)
      timeout -k 5 900 python bench.py --config 4 --no-cpu-baseline --no-gpu-baseline > $OUT/bench_cfg4_$TAG.json 2> $OUT/bench_cfg4_$TAG.err; echo "bench cfg4 exit $?"; cut -c1-330 $OUT/bench_cfg4_$TAG.json; tail -3 $OUT/bench_cfg4_$TAG.err;;
    launches_tf32) bash tools/visit_l.sh $TAG tf32 | tail -24;;
    launches_fp32) bash tools/visit_l.sh $TAG fp32 | tail -24;;
    smoke)
      timeout 600 python -c 'import __graft_entry__ as g; g.smoke()' > $OUT/smoke_$TAG.log 2>&1; echo "smoke exit $?"; tail -3 $OUT/smoke_$TAG.log;;
  esac
done
