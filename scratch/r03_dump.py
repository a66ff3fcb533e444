"""Outputs of the MCC step on several workloads, saved for an old-vs-new library comparison (SID_LIBRARY selects the
library), plus per-kernel device times of the cfg2 step from torch.profiler.
usage: python scratch/r03_dump.py OUTDIR            then   python scratch/r03_dump.py --compare DIR_A DIR_B"""
import json
import os
import sys

import numpy as np

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))


def workloads():
    from sea_ice_drift_b200 import synthetic as syn
    for name in ("cfg1", "cfg2", "cfg3"):
        img1, img2, c1, r1, c2, r2, b, cfg = syn.make_config(name, seed=0)
        yield name, img1, img2, [c1, r1, c2, r2, b], cfg["img_size"], cfg["angles"]
        if name == "cfg2":
            pts = [c1, r1, c2, r2, b]
            yield "cfg2_one_angle", img1, img2, pts, 35, [0]
            yield "cfg2_five_angles", img1, img2, pts, 35, [-6, -3, 0, 3, 6]
            # mixed borders at EW size (prepare_first_guess's distribution: 47 % at 20, the rest up to 50): two border classes
            rng = np.random.default_rng(7)
            side, nk = img1.shape[0], 50000
            m = syn.rotation_matrix(img1.shape, 2.0)
            kx, ky = rng.uniform(40, side - 40, nk), rng.uniform(40, side - 40, nk)
            k2x, k2y = syn.apply_affine(m, kx, ky)
            k2x, k2y = k2x + rng.normal(0, 0.8, nk), k2y + rng.normal(0, 0.8, nk)
            mixed = list(syn.orb_first_guess_inputs(img1, img2, 200, 35, inset=150, matches=(kx, ky, k2x, k2y)))
            yield "ew_mixed_borders", img1, img2, mixed, 35, [-3, 0, 3]


def dump(outdir):
    from sea_ice_drift_b200 import _lib
    os.makedirs(outdir, exist_ok=True)
    ctx = _lib.Context(0)
    for name, img1, img2, pts, s, angles in workloads():
        ctx.set_pair(img1, img2)
        out, st = ctx.run(*pts, s, angles, 0.0, want_status=True)
        np.save(os.path.join(outdir, name + "_table.npy"), out)
        np.save(os.path.join(outdir, name + "_status.npy"), st)
        print(name, len(pts[0]), "valid", int((st == 1).sum()), ctx.last_kernel_name, flush=True)
        if name == "cfg2":
            kernel_times(ctx, pts, s, angles, outdir)
    ctx.close()


def kernel_times(ctx, pts, s, angles, outdir, steps=20):
    import torch
    from torch.profiler import profile, ProfilerActivity
    for _ in range(3):
        ctx.run(*pts, s, angles, 0.0)
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        for _ in range(steps):
            ctx.run(*pts, s, angles, 0.0)
        torch.cuda.synchronize()
    per = {}
    for ev in prof.key_averages():
        if "pm_" in ev.key:
            per[ev.key] = {"count": ev.count, "ms_mean": ev.device_time_total / max(ev.count, 1) / 1e3}
    print(json.dumps(per), flush=True)
    with open(os.path.join(outdir, "kernel_times.json"), "w") as f:
        json.dump(per, f, indent=1)


def compare(da, db):
    ok = True
    names = sorted(f[:-len("_table.npy")] for f in os.listdir(da) if f.endswith("_table.npy"))
    for n in names:
        ta, tb = np.load(os.path.join(da, n + "_table.npy")), np.load(os.path.join(db, n + "_table.npy"))
        sa, sb = np.load(os.path.join(da, n + "_status.npy")), np.load(os.path.join(db, n + "_status.npy"))
        same = np.array_equal(ta.view(np.uint64), tb.view(np.uint64)) and np.array_equal(sa, sb)
        nbad = int((ta.view(np.uint64) != tb.view(np.uint64)).any(axis=1).sum())
        print("%-20s rows %6d  bit-identical %s  (%d rows differ)" % (n, len(ta), same, nbad))
        ok &= same
    print("ALL IDENTICAL" if ok else "DIFFERENCES FOUND")
    return ok


if __name__ == "__main__":
    if sys.argv[1] == "--compare":
        sys.exit(0 if compare(sys.argv[2], sys.argv[3]) else 1)
    dump(sys.argv[1])
