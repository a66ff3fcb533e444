#!/bin/bash
# Round 4 on one B200: smoke, tests/test_gpu_maps.py on the new library and on three mutants of it (built beforehand into
# scratch/ab/, git-ignored: the map stored after the smoothing, the template of angle 0, offsets one row early), bench.py
# old (parent commit, scratch/ab/libsid_old.so) vs new alternating on cfg2 and cfg1 with --dump-outputs, the cost of
# run_maps (scratch/time_maps.py) and the whole GPU suite.
set -u
O=${1:?usage: $0 OUTDIR}
mkdir -p $O
OLD=scratch/ab/libsid_old.so
nvidia-smi --query-gpu=name,power.limit,clocks.max.sm --format=csv > $O/gpu_info.txt 2>&1
cat $O/gpu_info.txt
python -c "import __graft_entry__ as g; g.build(); g.smoke()" > $O/smoke.txt 2>&1 || { echo SMOKE FAILED; tail -40 $O/smoke.txt; exit 1; }
tail -n 1 $O/smoke.txt
python -m pytest tests/test_gpu_maps.py -m gpu -q -p no:cacheprovider > $O/pytest_maps.txt 2>&1
tail -n 15 $O/pytest_maps.txt
for m in 1 2 3; do
    SID_LIBRARY=scratch/ab/libsid_m$m.so python -m pytest tests/test_gpu_maps.py -m gpu -q -p no:cacheprovider > $O/mutant_m$m.txt 2>&1
    echo "mutant m$m: $(tail -n 1 $O/mutant_m$m.txt)"
done
for r in 1 2 3 4 5; do
    for w in old new; do
        lib=""; [ $w = old ] && lib=$OLD
        SID_LIBRARY=$lib python bench.py --steps 100 --no-cpu-baseline --no-configs --dump-outputs $O/bench_${w}_cfg2 > $O/cfg2_${w}_$r.json 2> $O/cfg2_${w}_$r.err
        SID_LIBRARY=$lib python bench.py --workload cfg1 --steps 400 --no-cpu-baseline --no-configs --dump-outputs $O/bench_${w}_cfg1 > $O/cfg1_${w}_$r.json 2> $O/cfg1_${w}_$r.err
    done
    python -c "
import json
for c in ('cfg2', 'cfg1'):
    for w in ('old', 'new'):
        d = json.loads(open('$O/%s_%s_$r.json' % (c, w)).read().strip().splitlines()[-1])
        print('$r', c, w, 'value %.0f ms_per_step %.4f' % (d['value'], d['ms_per_step']))
"
done
python - <<PY
import numpy as np
for c in ('cfg2', 'cfg1'):
    for f in ('table', 'status'):
        a, b = np.load('$O/bench_old_%s/%s.npy' % (c, f)), np.load('$O/bench_new_%s/%s.npy' % (c, f))
        print('bench dump', c, f, a.shape, 'identical', np.array_equal(a.view(np.uint64), b.view(np.uint64)))
PY
python scratch/time_maps.py > $O/r04_maps.txt 2>&1
cat $O/r04_maps.txt
python -m pytest -m gpu -q -p no:cacheprovider > $O/pytest_gpu.txt 2>&1
tail -n 5 $O/pytest_gpu.txt
