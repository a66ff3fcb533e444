#!/bin/bash
# Round 5 on one B200 (sub-pixel refinement): smoke, tests/test_subpixel.py, the whole GPU suite, scratch/time_subpixel.py
# (parent library scratch/ab/libsid_old.so vs this one, flag off / on), bench.py parent vs new on cfg2 with --dump-outputs,
# and tests/test_subpixel.py against five mutants of the device function (built beforehand into scratch/ab/, git-ignored:
# m1 sign of p - q flipped, m2 neighbours swapped, m3 edge rule dropped (clamped index), m4 c2fg + (dc + dx),
# m5 offsets from the hes_smth map).
set -u
O=${1:?usage: $0 OUTDIR}
mkdir -p $O
OLD=scratch/ab/libsid_old.so
nvidia-smi --query-gpu=name,power.limit,clocks.max.sm --format=csv > $O/gpu_info.txt 2>&1
cat $O/gpu_info.txt
python -c "import __graft_entry__ as g; g.build(); g.smoke()" > $O/smoke.txt 2>&1 || { echo SMOKE FAILED; tail -40 $O/smoke.txt; exit 1; }
tail -n 1 $O/smoke.txt
python -m pytest tests/test_subpixel.py -m gpu -q -p no:cacheprovider > $O/pytest_subpixel.txt 2>&1
tail -n 25 $O/pytest_subpixel.txt
python -m pytest -m gpu -q -p no:cacheprovider > $O/pytest_gpu.txt 2>&1
tail -n 8 $O/pytest_gpu.txt
{ cat $O/gpu_info.txt; python scratch/time_subpixel.py $OLD; } > $O/r05_subpixel.txt 2>&1
cat $O/r05_subpixel.txt
for w in old new old new; do
    lib=""; [ $w = old ] && lib=$OLD
    SID_LIBRARY=$lib python bench.py --gpus 1 --steps 50 --warmup 5 --no-cpu-baseline --no-configs --dump-outputs $O/bench_$w > $O/bench_$w.json 2> $O/bench_$w.err
    python -c "
import json; d = json.loads(open('$O/bench_$w.json').read().strip().splitlines()[-1]); print('bench $w value %.0f ms_per_step %.4f' % (d['value'], d['ms_per_step']))"
done
python - <<PY
import numpy as np
for f in ('table', 'status'):
    a, b = np.load('$O/bench_old/%s.npy' % f), np.load('$O/bench_new/%s.npy' % f)
    print('bench dump', f, a.shape, 'identical', a.tobytes() == b.tobytes())
PY
for m in 1 2 3 4 5; do
    SID_LIBRARY=scratch/ab/libsid_m$m.so python -m pytest tests/test_subpixel.py -m gpu -q -p no:cacheprovider -rf > $O/mutant_m$m.txt 2>&1
    echo "mutant m$m: $(tail -n 1 $O/mutant_m$m.txt)"
    grep "^FAILED" $O/mutant_m$m.txt | sed 's/ - .*//' | sort | uniq | head -60
done
