#!/bin/bash
# cfg1 (2000^2, borders 20..41, two border classes) old vs new library, 5 alternating rounds.
set -u
O=${1:?usage: $0 OUTDIR}
mkdir -p $O
OLD=scratch/ab/libsid_old.so
python -c "import __graft_entry__ as g; g.build()" > $O/build.txt 2>&1
for r in 1 2 3 4 5; do
    SID_LIBRARY=$OLD python bench.py --workload cfg1 --steps 400 --no-cpu-baseline --no-configs > $O/cfg1_old_$r.json 2> $O/cfg1_old_$r.err
    python bench.py --workload cfg1 --steps 400 --no-cpu-baseline --no-configs > $O/cfg1_new_$r.json 2> $O/cfg1_new_$r.err
    python -c "
import json
for w in ('old', 'new'):
    d = json.loads(open('$O/cfg1_%s_$r.json' % w).read().strip().splitlines()[-1])
    print('$r', w, 'value %.0f ms_per_step %.4f' % (d['value'], d['ms_per_step']))
"
done
