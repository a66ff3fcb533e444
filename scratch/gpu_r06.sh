#!/bin/bash
# Round 6 on one B200 (drift without feature tracking): smoke, tests/test_coarse_tracking.py, the whole GPU suite,
# scratch/time_coarse.py, and bench.py parent (scratch/ab/libsid_old.so and scratch/ab/parent/, git-ignored) vs new with
# --dump-outputs, tables compared byte for byte.
set -u
O=${1:?usage: $0 OUTDIR}
mkdir -p $O
OLD=scratch/ab/libsid_old.so
nvidia-smi --query-gpu=name,power.limit,clocks.max.sm --format=csv > $O/gpu_info.txt 2>&1
cat $O/gpu_info.txt
python -c "import __graft_entry__ as g; g.build(); g.smoke()" > $O/smoke.txt 2>&1 || { echo SMOKE FAILED; tail -40 $O/smoke.txt; exit 1; }
tail -n 1 $O/smoke.txt
python -m pytest tests/test_coarse_tracking.py -m gpu -q -p no:cacheprovider -rf > $O/pytest_coarse.txt 2>&1
tail -n 25 $O/pytest_coarse.txt
{ cat $O/gpu_info.txt; python scratch/time_coarse.py; } > $O/r06_coarse.txt 2>&1
cat $O/r06_coarse.txt
# the ordering test on a copy of the tree without the stream synchronise in coarse_tracking (scratch/ab/mutant)
(cd scratch/ab/mutant && SID_LIBRARY=$OLDPWD/sea_ice_drift_b200/libsid_b200.so python -m pytest tests/test_coarse_tracking.py -m gpu -q -p no:cacheprovider -k ordered > $OLDPWD/$O/mutant_no_sync.txt 2>&1)
echo "without the synchronise: $(tail -n 1 $O/mutant_no_sync.txt)"
python -m pytest -m gpu -q -p no:cacheprovider -rf > $O/pytest_gpu.txt 2>&1
tail -n 8 $O/pytest_gpu.txt
# the parent's tree (scratch/ab/parent: git ls-files of the parent commit) runs the parent's bench.py and Python package
for w in old new old new; do
    dir=.; lib=""; [ $w = old ] && { dir=scratch/ab/parent; lib=$PWD/$OLD; }
    (cd $dir && SID_LIBRARY=$lib python bench.py --gpus 1 --steps 30 --warmup 5 --no-cpu-baseline --no-configs --dump-outputs $OLDPWD/$O/bench_$w > $OLDPWD/$O/bench_$w.json 2> $OLDPWD/$O/bench_$w.err)
    python -c "
import json; d = json.loads(open('$O/bench_$w.json').read().strip().splitlines()[-1]); print('bench $w value %.0f ms_per_step %.4f' % (d['value'], d['ms_per_step']))"
done
python - <<PY
import numpy as np, os
for f in sorted(os.listdir('$O/bench_old')):
    a, b = open('$O/bench_old/' + f, 'rb').read(), open('$O/bench_new/' + f, 'rb').read()
    print('bench dump', f, 'identical', a == b)
PY
