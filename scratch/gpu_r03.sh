#!/bin/bash
# Round 3 on one B200: smoke, old-vs-new outputs on cfg1 / cfg2 (1, 3, 5 angles) / cfg3 / mixed-border EW, per-kernel times,
# alternating bench A/B (5 rounds each), role profiles (-DSID_WS_PROF builds), GPU suite.
# The parent commit's library is built beforehand into scratch/ab/ (git-ignored).
set -u
O=${1:?usage: $0 OUTDIR}
mkdir -p $O
OLD=scratch/ab/libsid_old.so
nvidia-smi --query-gpu=name,power.limit,clocks.max.sm --format=csv > $O/gpu_info.txt 2>&1
cat $O/gpu_info.txt
python -c "import __graft_entry__ as g; g.build(); g.smoke()" > $O/smoke.txt 2>&1 || { echo SMOKE FAILED; tail -40 $O/smoke.txt; exit 1; }
tail -n 1 $O/smoke.txt
SID_LIBRARY=$OLD python scratch/r03_dump.py $O/dump_old > $O/dump_old.txt 2>&1
python scratch/r03_dump.py $O/dump_new > $O/dump_new.txt 2>&1 || { echo DUMP NEW FAILED; tail -40 $O/dump_new.txt; }
python scratch/r03_dump.py --compare $O/dump_old $O/dump_new | tee $O/compare.txt
grep '{' $O/dump_old.txt $O/dump_new.txt
for r in 1 2 3 4 5; do
    extra="--no-configs"
    [ $r = 1 ] && extra=""
    SID_LIBRARY=$OLD python bench.py --steps 100 --no-cpu-baseline $extra --dump-outputs $O/bench_old > $O/bench_old_$r.json 2> $O/bench_old_$r.err
    python bench.py --steps 100 --no-cpu-baseline $extra --dump-outputs $O/bench_new > $O/bench_new_$r.json 2> $O/bench_new_$r.err
    python -c "
import json
for w in ('old', 'new'):
    d = json.loads(open('$O/bench_%s_$r.json' % w).read().strip().splitlines()[-1])
    print('$r', w, 'value %.0f ms_per_step %.4f' % (d['value'], d['ms_per_step']), 'parity', d.get('parity', {}).get('position_angle_equal'), d.get('parity', {}).get('r_bit_equal'), d.get('parity', {}).get('compared'))
"
done
python - <<EOF
import numpy as np
for f in ('table', 'status'):
    a, b = np.load('$O/bench_old/%s.npy' % f), np.load('$O/bench_new/%s.npy' % f)
    print('bench dump', f, 'identical', np.array_equal(a.view(np.uint64), b.view(np.uint64)))
EOF
SID_LIBRARY=scratch/ab/libsid_old_prof.so python scratch/ws_prof.py > $O/prof_old.txt 2>&1
SID_LIBRARY=scratch/ab/libsid_new_prof.so python scratch/ws_prof.py > $O/prof_new.txt 2>&1
tail -n 8 $O/prof_old.txt $O/prof_new.txt
python -m pytest -m gpu -q -p no:cacheprovider > $O/pytest_gpu.txt 2>&1
tail -5 $O/pytest_gpu.txt
