#!/bin/bash
# Round 9 on one B200 (per-vector uncertainty): smoke, tests/test_uncertainty.py, bench.py parent (scratch/ab/libsid_old.so
# and scratch/ab/parent/, git-ignored) vs new with --dump-outputs, tables compared byte for byte, the whole GPU suite and
# scratch/time_uncert.py.
set -u
O=${1:?usage: $0 OUTDIR}
mkdir -p $O
OLD=scratch/ab/libsid_old.so
nvidia-smi --query-gpu=name,power.limit,clocks.max.sm --format=csv > $O/gpu_info.txt 2>&1
cat $O/gpu_info.txt
python -c "import __graft_entry__ as g; g.build(); g.smoke()" > $O/smoke.txt 2>&1 || { echo SMOKE FAILED; tail -40 $O/smoke.txt; exit 1; }
tail -n 1 $O/smoke.txt
python -m pytest tests/test_uncertainty.py -m gpu -q -p no:cacheprovider -rf > $O/pytest_uncert.txt 2>&1
tail -n 40 $O/pytest_uncert.txt
for w in old new old new; do
    dir=.; lib=""; [ $w = old ] && { dir=scratch/ab/parent; lib=$PWD/$OLD; }
    (cd $dir && SID_LIBRARY=$lib python bench.py --gpus 1 --steps 30 --warmup 5 --no-cpu-baseline --no-configs --dump-outputs $OLDPWD/$O/bench_$w > $OLDPWD/$O/bench_$w.json 2> $OLDPWD/$O/bench_$w.err)
    python -c "
import json; d = json.loads(open('$O/bench_$w.json').read().strip().splitlines()[-1]); print('bench $w value %.0f ms_per_step %.4f' % (d['value'], d['ms_per_step']))"
done
python - <<PY
import os
for f in sorted(os.listdir('$O/bench_old')):
    a, b = open('$O/bench_old/' + f, 'rb').read(), open('$O/bench_new/' + f, 'rb').read()
    print('bench dump', f, 'identical', a == b)
PY
{ cat $O/gpu_info.txt; python scratch/time_uncert.py scratch/ab/parent; } > $O/r09_uncert.txt 2>&1
cat $O/r09_uncert.txt
python -m pytest -m gpu -q -p no:cacheprovider -rf --deselect tests/test_uncertainty.py > $O/pytest_gpu.txt 2>&1
tail -n 15 $O/pytest_gpu.txt
