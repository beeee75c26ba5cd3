#!/bin/bash
# round 3, call a: CRL_STEP_ZONE_OBS_DELTA.  New tests, smoke, rows written per env-step, then the timing of the
# parent build against this tree, alternating, three runs each, with output dumps of both builds; last, the whole GPU
# suite.  The parent build is a copy of the parent commit, built the same way before the call:
#   git archive 4a9232b --prefix=parent/ | tar -x -C build/ && (cd build/parent && python -c "import __graft_entry__ as g; g.build()")
set -u
O=${1:?usage: $0 OUTPUT_DIR}
mkdir -p $O
nvidia-smi --query-gpu=name,power.limit,clocks.max.sm,driver_version --format=csv > $O/r03a_gpu.csv; cat $O/r03a_gpu.csv
t0=$(date +%s)
timeout 900 python -m pytest -q -x -p no:cacheprovider tests/test_gpu_zone_obs_delta.py tests/test_zone_obs_delta_flags.py > $O/r03a_new_tests.log 2>&1; echo "new tests rc=$? $(( $(date +%s) - t0 )) s"; tail -n 3 $O/r03a_new_tests.log
timeout 300 python -c "import __graft_entry__ as g; g.smoke()" > $O/r03a_smoke.log 2>&1; echo "smoke rc=$?"; tail -n 2 $O/r03a_smoke.log
timeout 300 python tools/r03/count_rows.py PointTSP-v0:65536:6000 ColourMatch-v0:262144:3000 PointTTSP-v0:262144:500 > $O/r03_rows.jsonl 2> $O/r03_rows.err; echo "rows rc=$?"; cat $O/r03_rows.jsonl
declare -A ARGS=([head]="--no-cpu-baseline" [r19]="--no-cpu-baseline --no-extra --min-replicas 19" [cm7]="--no-cpu-baseline --no-extra --env ColourMatch-v0 --envs 262144 --min-replicas 7")
for rep in 1 2 3; do
  for arm in parent pr; do
    dir=.; [ $arm = parent ] && dir=build/parent
    for c in head r19 cm7; do
      dump=""; [ $rep = 1 ] && dump="--dump-outputs $O/r03_dump_${arm}_${c}"
      t1=$(date +%s)
      timeout 400 python $dir/bench.py --gpus 1 ${ARGS[$c]} $dump > $O/r03_bench_${arm}_${c}_${rep}.json 2> $O/r03_bench_${arm}_${c}_${rep}.err
      rc=$?
      python - "$O/r03_bench_${arm}_${c}_${rep}.json" "$arm $c $rep rc=$rc $(( $(date +%s) - t1 )) s" <<'PY'
import json, sys
try:
    d = json.loads(open(sys.argv[1]).read().strip().splitlines()[-1])
    x = ' '.join('%s %.5f' % (k, v['ms_per_step']) for k, v in d.get('configs', {}).items())
    print(sys.argv[2], 'ms_per_step %.6f' % d['ms_per_step'], 'R', d['config']['ring_replicas'], x)
except Exception as ex:
    print(sys.argv[2], 'no result', repr(ex))
PY
    done
  done
done
python - "$O" <<'PY'
import glob, os, sys
import numpy as np
for c in ('head', 'r19', 'cm7'):
    a, b = os.path.join(sys.argv[1], 'r03_dump_parent_' + c), os.path.join(sys.argv[1], 'r03_dump_pr_' + c)
    names = sorted(os.listdir(a)) if os.path.isdir(a) else []
    ok = bool(names) and names == sorted(os.listdir(b)) and all(np.array_equal(np.load(os.path.join(a, n)), np.load(os.path.join(b, n))) for n in names)
    print('dump', c, 'arrays', len(names), 'all np.array_equal' if ok else 'MISMATCH')
PY
t2=$(date +%s)
timeout 1800 python -m pytest -q -p no:cacheprovider -m gpu --ignore=tests/test_gpu_zone_obs_delta.py tests > $O/r03a_gpu_suite.log 2>&1; echo "gpu suite rc=$? $(( $(date +%s) - t2 )) s"; tail -n 5 $O/r03a_gpu_suite.log
