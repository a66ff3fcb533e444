"""Cost and calibration of SID_UNCERT / uncertainty=True on one GPU.

    python scratch/time_uncert.py PARENT_TREE

PARENT_TREE: a checkout of the parent commit with its library built (its Python binds the parent's exports).

1. cfg2 resident step (39 425 points, 3 angles, s 35, b 20, subpixel): the parent, this library without SID_UNCERT and
   with it, each in its own process, alternating, 4 rounds of 40 timed calls (host clock around Context.run, which ends
   in the table's read-back); the three tables compared byte for byte.
2. torch.profiler, mean device time per launch of every kernel of a cfg2 resident call, with and without SID_UNCERT.
3. bench.py's drop_in_ew scene (cfg2's pair rotated by a known angle, 50 000 matches, 200 x 200 grid):
   pattern_matching(subpixel=True, uncertainty=True); median predicted sigma, median |error| against the known drift,
   per axis, and the share of errors inside 1 and 2 sigma."""
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
SUBPIXEL, UNCERT = 8, 64


def _root():
    root = sys.argv[sys.argv.index("--root") + 1] if "--root" in sys.argv else ROOT
    sys.path.insert(0, root)
    return root


def child_step(flag, n_calls=40):
    from sea_ice_drift_b200 import _lib, synthetic as syn
    img1, img2, c1, r1, c2, r2, b, cfg = syn.make_config("cfg2", seed=0)
    ctx = _lib.Context(0)
    ctx.set_pair(img1, img2)
    flags = _lib.SID_HES_NORM | SUBPIXEL | (UNCERT if flag else 0)
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
    for flag in (0, UNCERT):
        flags = _lib.SID_HES_NORM | SUBPIXEL | flag
        ctx.run(c1, r1, c2, r2, b, 35, cfg["angles"], 0.0, flags=flags)
        with profile(activities=[ProfilerActivity.CUDA]) as prof:
            for _ in range(20):
                ctx.run(c1, r1, c2, r2, b, 35, cfg["angles"], 0.0, flags=flags)
        res["uncert_%s" % ("on" if flag else "off")] = kernel_times(prof)
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


def child_drop_in_ew():
    from sea_ice_drift_b200 import pmlib, synthetic as syn
    n1, n2, kx, ky, k2x, k2y, lon, lat, m = ew_scene()
    ts = {False: [], True: []}
    res = {}
    for rnd in range(4):
        for unc in (False, True):
            t0 = time.perf_counter()
            with contextlib.redirect_stdout(io.StringIO()):
                res[unc] = pmlib.pattern_matching(lon, lat, n1, kx, ky, n2, k2x, k2y, angles=[-3, 0, 3], img_size=35,
                                                  subpixel=True, uncertainty=unc)
            if rnd:
                ts[unc].append(time.perf_counter() - t0)
    r = res[True]
    same = all(a.tobytes() == b.tobytes() for a, b in zip(res[False], r[:7]))
    sel = np.isfinite(r[0]) & np.isfinite(r[7]) & np.isfinite(r[8])
    c2, r2 = n2.transform_points(r[5][sel], r[6][sel], 1)
    c1g, r1g = n1.transform_points(lon[sel], lat[sel], 1)
    tx, ty = syn.apply_affine(m, c1g, r1g)
    ex, ey = c2 - (tx - 1), r2 - (ty - 1)
    fwd = n2._fwd[:, :2]                                     # pixel -> lon / lat: sigma in px from the grids
    sx, sy = r[7][sel] / abs(fwd[0, 0]), r[8][sel] / abs(fwd[1, 1])
    out = {"grid_points": int(lon.size), "valid": int(np.isfinite(r[0]).sum()), "with_sigma": int(sel.sum()),
           "grids_identical_to_call_without": same,
           "ms_median_off": 1e3 * float(np.median(ts[False])), "ms_median_on": 1e3 * float(np.median(ts[True]))}
    for name, e, s in (("column", ex, sx), ("row", ey, sy)):
        out[name] = {"median_sigma_px": float(np.median(s)), "median_abs_error_px": float(np.median(np.abs(e))),
                     "rms_error_px": float(np.sqrt(np.mean(e * e))), "mean_error_px": float(np.mean(e)),
                     "within_1sigma": float(np.mean(np.abs(e) <= s)), "within_2sigma": float(np.mean(np.abs(e) <= 2 * s)),
                     "within_1sigma_centred": float(np.mean(np.abs(e - np.mean(e)) <= s))}
    print(json.dumps(out))


def run_child(args, root=ROOT):
    p = subprocess.run([sys.executable, os.path.abspath(__file__)] + args + ["--root", root], cwd=root,
                       stdout=subprocess.PIPE, stderr=subprocess.PIPE, text=True)
    if p.returncode:
        sys.stderr.write(p.stderr)
        raise RuntimeError("child %s failed" % args)
    return json.loads(p.stdout.strip().splitlines()[-1])


def main():
    parent = os.path.abspath(sys.argv[1])
    arms = [("parent", ["--step", "0"], parent), ("new_off", ["--step", "0"], ROOT), ("new_on", ["--step", "1"], ROOT)]
    times = {a: [] for a, _, _ in arms}
    sha = {}
    print("1. cfg2 resident step with subpixel, host clock around Context.run (40 calls per process, 4 rounds, arms "
          "alternating)")
    for rnd in range(4):
        for name, args, root in arms:
            d = run_child(args, root)
            times[name] += d["ms"]
            sha[name] = d["sha"]
            print("  round %d %-8s median %.3f ms  min %.3f ms  (%s)" % (rnd, name, np.median(d["ms"]), min(d["ms"]),
                                                                    d["kernel"]), flush=True)
    for name in times:
        t = np.array(times[name])
        print("  %-8s median %.3f ms  p10 %.3f  p90 %.3f  (%d calls)" % (name, np.median(t), np.percentile(t, 10),
                                                                      np.percentile(t, 90), t.size))
    print("  tables parent == new without flag == new with flag (bytes): %s" % (sha["parent"] == sha["new_off"] == sha["new_on"]))
    print("2. torch.profiler, cfg2 resident call, mean device time per launch (20 calls each)", flush=True)
    for arm, ks in run_child(["--profile-step"]).items():
        for k, v in sorted(ks.items()):
            print("  %-11s %-60s %3d launches  %9.1f us" % (arm, k, v["launches"], v["mean_us"]))
    print("3. drop_in_ew: pattern_matching(subpixel=True) with and without uncertainty=True", flush=True)
    print(json.dumps(run_child(["--drop-in-ew"]), indent=1), flush=True)


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
    else:
        main()
