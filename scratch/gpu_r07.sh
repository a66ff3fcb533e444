#!/bin/bash
# Round 7 on one B200 (masked correlation): smoke, tests/test_masked_matching.py, bench.py parent (scratch/ab/libsid_old.so
# and scratch/ab/parent/, git-ignored) vs new with --dump-outputs, tables compared byte for byte, the whole GPU suite and
# scratch/time_masked.py.
set -u
O=${1:?usage: $0 OUTDIR}
mkdir -p $O
OLD=scratch/ab/libsid_old.so
nvidia-smi --query-gpu=name,power.limit,clocks.max.sm --format=csv > $O/gpu_info.txt 2>&1
cat $O/gpu_info.txt
python -c "import __graft_entry__ as g; g.build(); g.smoke()" > $O/smoke.txt 2>&1 || { echo SMOKE FAILED; tail -40 $O/smoke.txt; exit 1; }
tail -n 1 $O/smoke.txt
python -m pytest tests/test_masked_matching.py -m gpu -q -p no:cacheprovider -rf -x > $O/pytest_masked.txt 2>&1
tail -n 30 $O/pytest_masked.txt
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
python -m pytest -m gpu -q -p no:cacheprovider -rf > $O/pytest_gpu.txt 2>&1
tail -n 12 $O/pytest_gpu.txt
{ cat $O/gpu_info.txt; python scratch/time_masked.py $OLD; } > $O/r07_masked.txt 2>&1
cat $O/r07_masked.txt
