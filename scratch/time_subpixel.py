"""Cost and accuracy of SID_SUBPIXEL (subpixel=True) on one GPU.

    python scratch/time_subpixel.py PARENT_LIB.so [OUTDIR]

1. cfg2 resident step (39 425 points, 3 angles, s 35, b 20): the parent library, this library without the flag and this
   library with the flag, each in its own process, alternating, 6 rounds of 40 timed calls (host clock around
   Context.run, which ends in the table's read-back); tables of parent and flag-off compared byte for byte.
2. Per-kernel device times of the same step, flag off / on, from torch.profiler in a separate process.
3. cfg1 with the ORB first guess (2 500 points, 1 angle, borders 20 ... 41): flag off / on alternating in one process.
4. bench.py's drop_in_ew call (pattern_matching on the EW-sized pair, 50 000 matches, 200 x 200 grid): call time and
   median error against the known drift, with and without subpixel=True."""
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
sys.path.insert(0, ROOT)


def child_step(flag, n_calls=40):
    from sea_ice_drift_b200 import _lib, synthetic as syn
    img1, img2, c1, r1, c2, r2, b, cfg = syn.make_config("cfg2", seed=0)
    ctx = _lib.Context(0)
    ctx.set_pair(img1, img2)
    flags = _lib.SID_HES_NORM | (_lib.SID_SUBPIXEL if flag else 0)
    for _ in range(5):
        out = ctx.run(c1, r1, c2, r2, b, 35, cfg["angles"], 0.0, flags=flags)
    ts = []
    for _ in range(n_calls):
        t0 = time.perf_counter()
        out = ctx.run(c1, r1, c2, r2, b, 35, cfg["angles"], 0.0, flags=flags)
        ts.append(time.perf_counter() - t0)
    print(json.dumps({"ms": [t * 1e3 for t in ts], "sha": hashlib.sha256(out.tobytes()).hexdigest(),
                      "kernel": ctx.last_kernel_name}))


def child_profile():
    import torch
    from torch.profiler import profile, ProfilerActivity
    from sea_ice_drift_b200 import _lib, synthetic as syn
    img1, img2, c1, r1, c2, r2, b, cfg = syn.make_config("cfg2", seed=0)
    ctx = _lib.Context(0)
    ctx.set_pair(img1, img2)
    res = {}
    for flag in (0, 1):
        flags = _lib.SID_HES_NORM | (_lib.SID_SUBPIXEL if flag else 0)
        for _ in range(3):
            ctx.run(c1, r1, c2, r2, b, 35, cfg["angles"], 0.0, flags=flags)
        with profile(activities=[ProfilerActivity.CUDA]) as prof:
            for _ in range(10):
                ctx.run(c1, r1, c2, r2, b, 35, cfg["angles"], 0.0, flags=flags)
        tot = {}
        for ev in prof.events():
            if ev.device_type.name == "CUDA" and "kernel" in ev.name:
                tot.setdefault(ev.name, []).append(ev.device_time if hasattr(ev, "device_time") else ev.cuda_time)
        res["flag_%s" % ("on" if flag else "off")] = {k: {"calls": len(v), "mean_us": float(np.mean(v))} for k, v in tot.items()}
    print(json.dumps(res))


def cfg1_and_drop_in():
    from sea_ice_drift_b200 import _lib, pmlib, synthetic as syn
    out = {}
    # cfg1: ORB first guess, resident pair
    img1, img2, _, _, _, _, _, cfg = syn.make_config("cfg1", seed=0)
    c1, r1, c2, r2, b = syn.orb_first_guess_inputs(img1, img2, cfg["grid"], cfg["img_size"])
    ctx = _lib.default_context()
    ctx.set_pair(img1, img2)
    ts = {0: [], 1: []}
    tabs = {}
    for rnd in range(8):
        for flag in (0, 1):
            flags = _lib.SID_HES_NORM | (_lib.SID_SUBPIXEL if flag else 0)
            for k in range(60):
                t0 = time.perf_counter()
                tabs[flag] = ctx.run(c1, r1, c2, r2, b, 35, cfg["angles"], 0.0, flags=flags)
                if rnd or k >= 10:
                    ts[flag].append(time.perf_counter() - t0)
    tx, ty = syn.apply_affine(cfg["matrix"], c1, r1)
    err = {f: float(np.nanmedian(np.hypot(tabs[f][:, 0] - (tx - 1), tabs[f][:, 1] - (ty - 1)))) for f in (0, 1)}
    out["cfg1_orb"] = {"points": int(c1.size), "borders": [float(b.min()), float(b.max())], "kernel": ctx.last_kernel_name,
                       "ms_median_off": 1e3 * float(np.median(ts[0])), "ms_median_on": 1e3 * float(np.median(ts[1])),
                       "ms_p10_off": 1e3 * float(np.percentile(ts[0], 10)), "ms_p10_on": 1e3 * float(np.percentile(ts[1], 10)),
                       "median_error_px_off": err[0], "median_error_px_on": err[1]}
    # drop_in_ew: bench.py's scene
    img1, img2, *_ = syn.make_config("cfg2", seed=0)
    rng = np.random.default_rng(7)
    side, nk, grid = img1.shape[0], 50000, 200
    m = syn.rotation_matrix(img1.shape, syn.CONFIGS["cfg2"]["warp"][1])
    kx, ky = rng.uniform(40, side - 40, nk), rng.uniform(40, side - 40, nk)
    k2x, k2y = syn.apply_affine(m, kx, ky)
    k2x, k2y = k2x + rng.normal(0, 0.8, nk), k2y + rng.normal(0, 0.8, nk)
    n1, n2 = syn.ArrayDomain(img1), syn.ArrayDomain(img2)
    gx, gy = np.meshgrid(np.linspace(150, side - 150, grid), np.linspace(150, side - 150, grid))
    lon, lat = n2.transform_points(gx, gy)
    ts = {False: [], True: []}
    res = {}
    for rnd in range(6):
        for sub in (False, True):
            t0 = time.perf_counter()
            with contextlib.redirect_stdout(io.StringIO()):
                res[sub] = pmlib.pattern_matching(lon, lat, n1, kx, ky, n2, k2x, k2y, angles=[-3, 0, 3], img_size=35,
                                                  subpixel=sub)
            if rnd:
                ts[sub].append(time.perf_counter() - t0)
    errs = {}
    for sub in (False, True):
        ok = np.isfinite(res[sub][0])
        c2, r2 = n2.transform_points(res[sub][5][ok], res[sub][6][ok], 1)
        c1g, r1g = n1.transform_points(lon[ok], lat[ok], 1)
        tx, ty = syn.apply_affine(m, c1g, r1g)
        e = np.hypot(c2 - (tx - 1), r2 - (ty - 1))
        errs[sub] = (float(np.median(e)), float(np.percentile(e, 90)), int(ok.sum()))
    out["drop_in_ew"] = {"ms_median_off": 1e3 * float(np.median(ts[False])), "ms_median_on": 1e3 * float(np.median(ts[True])),
                         "median_error_px_off": errs[False][0], "median_error_px_on": errs[True][0],
                         "p90_error_px_off": errs[False][1], "p90_error_px_on": errs[True][1], "valid": errs[True][2]}
    print(json.dumps(out))


def run_child(args, lib=None):
    env = dict(os.environ)
    if lib:
        env["SID_LIBRARY"] = lib
    else:
        env.pop("SID_LIBRARY", None)
    r = subprocess.run([sys.executable, os.path.abspath(__file__)] + args, env=env, capture_output=True, text=True)
    if r.returncode:
        raise RuntimeError(r.stderr[-3000:])
    return json.loads(r.stdout.strip().splitlines()[-1])


def main():
    parent = os.path.abspath(sys.argv[1])
    arms = [("parent", ["--step", "0"], parent), ("new_off", ["--step", "0"], None), ("new_on", ["--step", "1"], None)]
    times = {a: [] for a, _, _ in arms}
    sha = {}
    print("1. cfg2 resident step, host clock around Context.run (40 calls per process, 6 rounds, arms alternating)")
    for rnd in range(6):
        for name, args, lib in arms:
            d = run_child(args, lib)
            times[name] += d["ms"]
            sha[name] = d["sha"]
            print("  round %d %-8s median %.3f ms  min %.3f ms  (%s)" % (rnd, name, np.median(d["ms"]), min(d["ms"]), d["kernel"]),
                  flush=True)
    for name in times:
        t = np.array(times[name])
        print("  %-8s median %.3f ms  p10 %.3f  p90 %.3f  (%d calls)" % (name, np.median(t), np.percentile(t, 10),
                                                                      np.percentile(t, 90), t.size))
    print("  table parent == new without flag (bytes): %s" % (sha["parent"] == sha["new_off"]))
    print("  table with flag differs (refined c2 / r2): %s" % (sha["new_on"] != sha["new_off"]))
    print("2. torch.profiler, cfg2 step, mean device time per kernel launch")
    prof = run_child(["--profile"])
    for arm, ks in prof.items():
        for k, v in sorted(ks.items()):
            print("  %-9s %-40s %3d launches  %9.1f us" % (arm, k[:40], v["calls"], v["mean_us"]))
    print("3./4. cfg1 (ORB first guess) and the drop-in EW call")
    d = run_child(["--cfg1-drop-in"])
    print(json.dumps(d, indent=1))


if __name__ == "__main__":
    if "--step" in sys.argv:
        child_step(int(sys.argv[sys.argv.index("--step") + 1]))
    elif "--profile" in sys.argv:
        child_profile()
    elif "--cfg1-drop-in" in sys.argv:
        cfg1_and_drop_in()
    else:
        main()
