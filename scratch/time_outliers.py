"""Cost and effect of SID_PEAKS / outliers=True on one GPU.

    python scratch/time_outliers.py PARENT_TREE

PARENT_TREE: a checkout of the parent commit with its library built (its Python binds the parent's exports).

1. cfg2 resident step (39 425 points, 3 angles, s 35, b 20): the parent, this library without SID_PEAKS and with it, each
   in its own process, alternating, 4 rounds of 40 timed calls (host clock around Context.run, which ends in the
   table's read-back); the three tables compared byte for byte.
2. torch.profiler, mean device time per launch of every kernel of a cfg2 resident call, with and without SID_PEAKS.
3. bench.py's drop_in_ew call (cfg2's pair, 50 000 matches, 200 x 200 grid): pattern_matching with and without
   outliers=True, alternating, 6 rounds; rows changed, flags, error against the known drift.
4. The coast scene of DESIGN 4.1e (scratch/time_masked.py) with masked=True: what outliers=True does to the recovered
   vectors more than 2 px off, and pm_masked_kernel's device time per launch with and without SID_PEAKS."""
import contextlib
import hashlib
import io
import json
import os
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _root():
    root = sys.argv[sys.argv.index("--root") + 1] if "--root" in sys.argv else ROOT
    sys.path.insert(0, root)
    return root


def child_step(flag, n_calls=40):
    from sea_ice_drift_b200 import _lib, synthetic as syn
    img1, img2, c1, r1, c2, r2, b, cfg = syn.make_config("cfg2", seed=0)
    ctx = _lib.Context(0)
    ctx.set_pair(img1, img2)
    flags = _lib.SID_HES_NORM | (32 if flag else 0)
    for _ in range(5):
        out = ctx.run(c1, r1, c2, r2, b, 35, cfg["angles"], 0.0, flags=flags)
    ts = []
    for _ in range(n_calls):
        t0 = time.perf_counter()
        out = ctx.run(c1, r1, c2, r2, b, 35, cfg["angles"], 0.0, flags=flags)
        ts.append(time.perf_counter() - t0)
    print(json.dumps({"ms": [t * 1e3 for t in ts], "sha": hashlib.sha256(out.tobytes()).hexdigest(),
                      "kernel": ctx.last_kernel_name}))


def kernel_times(prof):
    tot = {}
    for ev in prof.events():
        if ev.device_type.name == "CUDA" and "memcpy" not in ev.name.lower() and "memset" not in ev.name.lower():
            tot.setdefault(ev.name, []).append(ev.device_time if hasattr(ev, "device_time") else ev.cuda_time)
    return {k[:60]: {"launches": len(v), "mean_us": float(np.mean(v))} for k, v in tot.items()}


def child_profile_step():
    from torch.profiler import profile, ProfilerActivity
    from sea_ice_drift_b200 import _lib, synthetic as syn
    img1, img2, c1, r1, c2, r2, b, cfg = syn.make_config("cfg2", seed=0)
    ctx = _lib.Context(0)
    ctx.set_pair(img1, img2)
    res = {}
    for flag in (0, 32):
        flags = _lib.SID_HES_NORM | flag
        ctx.run(c1, r1, c2, r2, b, 35, cfg["angles"], 0.0, flags=flags)
        with profile(activities=[ProfilerActivity.CUDA]) as prof:
            for _ in range(5):
                ctx.run(c1, r1, c2, r2, b, 35, cfg["angles"], 0.0, flags=flags)
        res["peaks_%s" % ("on" if flag else "off")] = kernel_times(prof)
    print(json.dumps(res))


def ew_scene():
    from sea_ice_drift_b200 import synthetic as syn
    img1, img2, *_ = syn.make_config("cfg2", seed=0)
    rng = np.random.default_rng(7)
    side, n_keypoints, grid = img1.shape[0], 50000, 200
    m = syn.rotation_matrix(img1.shape, syn.CONFIGS["cfg2"]["warp"][1])
    kx, ky = rng.uniform(40, side - 40, n_keypoints), rng.uniform(40, side - 40, n_keypoints)
    k2x, k2y = syn.apply_affine(m, kx, ky)
    k2x, k2y = k2x + rng.normal(0, 0.8, n_keypoints), k2y + rng.normal(0, 0.8, n_keypoints)
    n1, n2 = syn.ArrayDomain(img1), syn.ArrayDomain(img2)
    gx, gy = np.meshgrid(np.linspace(150, side - 150, grid), np.linspace(150, side - 150, grid))
    lon, lat = n2.transform_points(gx, gy)
    return n1, n2, kx, ky, k2x, k2y, lon, lat, m


def errors(res, n1, n2, lon, lat, m, sel):
    from sea_ice_drift_b200 import synthetic as syn
    c2, r2 = n2.transform_points(res[5][sel], res[6][sel], 1)
    c1g, r1g = n1.transform_points(lon[sel], lat[sel], 1)
    tx, ty = syn.apply_affine(m, c1g, r1g)
    return np.hypot(c2 - (tx - 1), r2 - (ty - 1))


def changed(a, b):
    return ~((a == b) | (np.isnan(a) & np.isnan(b)))


def child_drop_in_ew():
    from sea_ice_drift_b200 import pmlib
    n1, n2, kx, ky, k2x, k2y, lon, lat, m = ew_scene()
    ts = {False: [], True: []}
    res = {}
    for rnd in range(6):
        for outliers in (False, True):
            t0 = time.perf_counter()
            with contextlib.redirect_stdout(io.StringIO()):
                res[outliers] = pmlib.pattern_matching(lon, lat, n1, kx, ky, n2, k2x, k2y, angles=[-3, 0, 3], img_size=35,
                                                       outliers=outliers)
            if rnd:
                ts[outliers].append(time.perf_counter() - t0)
    off, on = res[False], res[True]
    ch = changed(off[0], on[0]) | changed(off[1], on[1])
    rejected = np.isfinite(off[0]) & np.isnan(on[0])
    e_off = errors(off, n1, n2, lon, lat, m, np.isfinite(off[0]))
    e_on = errors(on, n1, n2, lon, lat, m, np.isfinite(on[0]))
    print(json.dumps({"grid_points": int(lon.size), "valid_off": int(np.isfinite(off[0]).sum()),
                      "ms_median_off": 1e3 * float(np.median(ts[False])), "ms_median_on": 1e3 * float(np.median(ts[True])),
                      "ms_all_off": [1e3 * t for t in ts[False]], "ms_all_on": [1e3 * t for t in ts[True]],
                      "rows_changed": int(ch.sum()), "rows_rejected": int(rejected.sum()),
                      "rows_replaced": int((ch & ~rejected).sum()),
                      "error_off_px": {"median": float(np.median(e_off)), "over_2px": int((e_off > 2).sum())},
                      "error_on_px": {"median": float(np.median(e_on)), "over_2px": int((e_on > 2).sum())}}))


def child_coast():
    from torch.profiler import profile, ProfilerActivity
    from sea_ice_drift_b200.seaicedrift import SeaIceDrift
    sys.path.insert(0, os.path.join(ROOT, "scratch"))
    from time_masked import coast_scene
    n1, n2, kx, ky, k2x, k2y, lon, lat, m = coast_scene()
    sid = SeaIceDrift(n1, n2)
    ll = (*n1.transform_points(kx, ky), *n2.transform_points(k2x, k2y))
    kw = dict(angles=[-3, 0, 3], img_size=35)
    with contextlib.redirect_stdout(io.StringIO()):
        plain = sid.get_drift_PM(lon, lat, *ll, **kw)
        masked = sid.get_drift_PM(lon, lat, *ll, masked=True, **kw)
        fixed = sid.get_drift_PM(lon, lat, *ll, masked=True, outliers=True, **kw)
    recovered = np.isfinite(masked[0]) & ~np.isfinite(plain[0])
    e_rec = errors(masked, n1, n2, lon, lat, m, recovered)
    bad = np.flatnonzero(recovered)[e_rec > 2]
    good = np.flatnonzero(recovered)[e_rec <= 2]
    rej_bad = np.isnan(fixed[0].ravel()[bad])
    ch_bad = changed(masked[0].ravel()[bad], fixed[0].ravel()[bad]) & ~rej_bad
    fixed_sub = tuple(g.ravel()[bad][ch_bad] for g in fixed)
    e_fixed_bad = errors(fixed_sub, n1, n2, lon.ravel()[bad][ch_bad], lat.ravel()[bad][ch_bad], m,
                         np.ones(int(ch_bad.sum()), bool)) if ch_bad.any() else np.zeros(0)
    rej_good = np.isnan(fixed[0].ravel()[good])
    ch_all = changed(masked[0], fixed[0]) | changed(masked[1], fixed[1])
    prof_res = {}
    for outliers in (False, True):
        with contextlib.redirect_stdout(io.StringIO()):
            with profile(activities=[ProfilerActivity.CUDA]) as prof:
                for _ in range(3):
                    sid.get_drift_PM(lon, lat, *ll, masked=True, outliers=outliers, **kw)
        prof_res["outliers_%s" % ("on" if outliers else "off")] = {k: v for k, v in kernel_times(prof).items()
                                                                    if "masked" in k or "tail" in k or "outlier" in k}
    print(json.dumps({"recovered": int(recovered.sum()), "recovered_over_2px": int(bad.size),
                      "of_those_rejected": int(rej_bad.sum()), "of_those_replaced": int(ch_bad.sum()),
                      "replaced_error_px": [float(e) for e in e_fixed_bad],
                      "recovered_within_2px_rejected": int(rej_good.sum()), "recovered_within_2px": int(good.size),
                      "rows_changed_whole_grid": int(ch_all.sum()), "valid_masked": int(np.isfinite(masked[0]).sum()),
                      "profile": prof_res}))


def run_child(args, root=ROOT):
    env = dict(os.environ)
    env.pop("SID_LIBRARY", None)
    r = subprocess.run([sys.executable, os.path.abspath(__file__)] + args + ["--root", root], env=env, cwd=root,
                       capture_output=True, text=True)
    if r.returncode:
        raise RuntimeError(r.stderr[-3000:])
    return json.loads(r.stdout.strip().splitlines()[-1])


def main():
    parent = os.path.abspath(sys.argv[1])
    arms = [("parent", ["--step", "0"], parent), ("new_off", ["--step", "0"], ROOT), ("new_on", ["--step", "1"], ROOT)]
    times = {a: [] for a, _, _ in arms}
    sha = {}
    print("1. cfg2 resident step, host clock around Context.run (40 calls per process, 4 rounds, arms alternating)")
    for rnd in range(4):
        for name, args, root in arms:
            d = run_child(args, root)
            times[name] += d["ms"]
            sha[name] = d["sha"]
            print("  round %d %-8s median %.3f ms  min %.3f ms  (%s)" % (rnd, name, np.median(d["ms"]), min(d["ms"]), d["kernel"]),
                  flush=True)
    for name in times:
        t = np.array(times[name])
        print("  %-8s median %.3f ms  p10 %.3f  p90 %.3f  (%d calls)" % (name, np.median(t), np.percentile(t, 10),
                                                                      np.percentile(t, 90), t.size))
    print("  tables parent == new without flag == new with flag (bytes): %s" % (sha["parent"] == sha["new_off"] == sha["new_on"]))
    print("2. torch.profiler, cfg2 resident call, mean device time per launch (5 calls each)", flush=True)
    for arm, ks in run_child(["--profile-step"]).items():
        for k, v in sorted(ks.items()):
            print("  %-10s %-60s %3d launches  %9.1f us" % (arm, k, v["launches"], v["mean_us"]))
    print("3. drop_in_ew: pattern_matching with and without outliers=True", flush=True)
    print(json.dumps(run_child(["--drop-in-ew"]), indent=1), flush=True)
    print("4. coast scene of DESIGN 4.1e, get_drift_PM(masked=True) with and without outliers=True", flush=True)
    print(json.dumps(run_child(["--coast"]), indent=1), flush=True)


if __name__ == "__main__":
    if "--step" in sys.argv:
        _root()
        child_step(int(sys.argv[sys.argv.index("--step") + 1]))
    elif "--profile-step" in sys.argv:
        _root()
        child_profile_step()
    elif "--drop-in-ew" in sys.argv:
        _root()
        child_drop_in_ew()
    elif "--coast" in sys.argv:
        _root()
        child_coast()
    else:
        main()
