"""Cost and yield of SID_MASKED (masked=True) on one GPU.

    python scratch/time_masked.py PARENT_LIB.so

1. cfg2 resident step (39 425 points, 3 angles, s 35, b 20; no template holds a 0 pixel, so the flag only adds the
   search for candidates): the parent library, this library without the flag and with it, each in its own process,
   alternating, 4 rounds of 40 timed calls (host clock around Context.run, which ends in the table's read-back); the
   three tables compared byte for byte.
2. EW-sized scene with a coastline and a swath edge (cfg2's 10400 x 10400 pair, land fixed in both images, no-data beyond
   a slanted swath edge that differs between the images, 50 000 matches on ice, 200 x 200 grid): the whole get_drift_PM
   call with and without masked=True (alternating, 6 rounds), the vectors recovered and their error against the known
   drift; in a separate process torch.profiler's device times of pm_masked_kernel and masked_candidates_kernel."""
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
    flags = _lib.SID_HES_NORM | (16 if flag else 0)
    for _ in range(5):
        out = ctx.run(c1, r1, c2, r2, b, 35, cfg["angles"], 0.0, flags=flags)
    ts = []
    for _ in range(n_calls):
        t0 = time.perf_counter()
        out = ctx.run(c1, r1, c2, r2, b, 35, cfg["angles"], 0.0, flags=flags)
        ts.append(time.perf_counter() - t0)
    print(json.dumps({"ms": [t * 1e3 for t in ts], "sha": hashlib.sha256(out.tobytes()).hexdigest(),
                      "kernel": ctx.last_kernel_name}))


def coast_scene():
    from sea_ice_drift_b200 import synthetic as syn
    img1, img2, *_ = syn.make_config("cfg2", seed=0)
    side = img1.shape[0]
    m = syn.rotation_matrix(img1.shape, syn.CONFIGS["cfg2"]["warp"][1])
    img1, img2 = img1.copy(), img2.copy()
    for y0 in range(0, side, 1024):                       # in blocks: the full-size index grids would need 1.7 GB
        yy, xx = np.mgrid[y0:min(side, y0 + 1024), :side]
        land = xx > 0.72 * side + 400 * np.sin(yy / 700.0) + 150 * np.sin(yy / 173.0)
        img1[y0:y0 + 1024][land | (yy > 0.8 * side + 0.1 * xx)] = 0
        img2[y0:y0 + 1024][land | (yy > 0.82 * side + 0.08 * xx)] = 0
    rng = np.random.default_rng(7)
    nk, grid = 50000, 200
    kx, ky = rng.uniform(40, side - 40, 3 * nk), rng.uniform(40, side - 40, 3 * nk)
    k2x, k2y = syn.apply_affine(m, kx, ky)
    ice = (img1[ky.astype(int), kx.astype(int)] > 0) & \
        (img2[np.clip(k2y, 0, side - 1).astype(int), np.clip(k2x, 0, side - 1).astype(int)] > 0)
    sel = np.flatnonzero(ice)[:nk]
    kx, ky = kx[sel], ky[sel]
    k2x, k2y = k2x[sel] + rng.normal(0, 0.8, sel.size), k2y[sel] + rng.normal(0, 0.8, sel.size)
    n1, n2 = syn.ArrayDomain(img1), syn.ArrayDomain(img2)
    gx, gy = np.meshgrid(np.linspace(150, side - 150, grid), np.linspace(150, side - 150, grid))
    lon, lat = n2.transform_points(gx, gy)
    return n1, n2, kx, ky, k2x, k2y, lon, lat, m


def child_drop_in():
    from sea_ice_drift_b200 import synthetic as syn
    from sea_ice_drift_b200.seaicedrift import SeaIceDrift
    n1, n2, kx, ky, k2x, k2y, lon, lat, m = coast_scene()
    sid = SeaIceDrift(n1, n2)
    ll = (*n1.transform_points(kx, ky), *n2.transform_points(k2x, k2y))
    ts = {False: [], True: []}
    res = {}
    for rnd in range(6):
        for masked in (False, True):
            t0 = time.perf_counter()
            with contextlib.redirect_stdout(io.StringIO()):
                res[masked] = sid.get_drift_PM(lon, lat, *ll, angles=[-3, 0, 3], img_size=35, masked=masked)
            if rnd:
                ts[masked].append(time.perf_counter() - t0)

    def errors(r, sel):
        c2, r2 = n2.transform_points(r[5][sel], r[6][sel], 1)
        c1g, r1g = n1.transform_points(lon[sel], lat[sel], 1)
        tx, ty = syn.apply_affine(m, c1g, r1g)
        return np.hypot(c2 - (tx - 1), r2 - (ty - 1))
    was = np.isfinite(res[False][0])
    new = np.isfinite(res[True][0]) & ~was
    same = all(a[was].tobytes() == b[was].tobytes() for a, b in zip(res[False], res[True]))
    e_new, e_was = errors(res[True], new), errors(res[False], was)
    print(json.dumps({"keypoints": int(kx.size), "grid_points": int(lon.size),
                      "ms_median_off": 1e3 * float(np.median(ts[False])), "ms_median_on": 1e3 * float(np.median(ts[True])),
                      "ms_all_off": [1e3 * t for t in ts[False]], "ms_all_on": [1e3 * t for t in ts[True]],
                      "vectors_off": int(was.sum()), "vectors_recovered": int(new.sum()), "unmasked_vectors_identical": same,
                      "recovered_error_px": {"median": float(np.median(e_new)), "p90": float(np.percentile(e_new, 90)),
                                             "within_1px": float(np.mean(e_new <= 1.0)), "over_2px": int((e_new > 2).sum())},
                      "unmasked_error_px": {"median": float(np.median(e_was)), "p90": float(np.percentile(e_was, 90))}}))


def child_profile():
    from torch.profiler import profile, ProfilerActivity
    from sea_ice_drift_b200.seaicedrift import SeaIceDrift
    n1, n2, kx, ky, k2x, k2y, lon, lat, m = coast_scene()
    sid = SeaIceDrift(n1, n2)
    ll = (*n1.transform_points(kx, ky), *n2.transform_points(k2x, k2y))
    res = {}
    for masked in (False, True):
        with contextlib.redirect_stdout(io.StringIO()):
            sid.get_drift_PM(lon, lat, *ll, angles=[-3, 0, 3], img_size=35, masked=masked)
            with profile(activities=[ProfilerActivity.CUDA]) as prof:
                for _ in range(3):
                    sid.get_drift_PM(lon, lat, *ll, angles=[-3, 0, 3], img_size=35, masked=masked)
        tot = {}
        for ev in prof.events():
            if ev.device_type.name == "CUDA" and "kernel" in ev.name:
                tot.setdefault(ev.name, []).append(ev.device_time if hasattr(ev, "device_time") else ev.cuda_time)
        res["masked_%s" % ("on" if masked else "off")] = {k: {"calls": len(v), "mean_us": float(np.mean(v))}
                                                          for k, v in tot.items()}
    print(json.dumps(res))


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
    print("1. cfg2 resident step, host clock around Context.run (40 calls per process, 4 rounds, arms alternating)")
    for rnd in range(4):
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
    print("  tables parent == new without flag == new with flag (bytes): %s" % (sha["parent"] == sha["new_off"] == sha["new_on"]))
    print("2. EW-sized scene with a coastline and a swath edge: get_drift_PM with and without masked=True", flush=True)
    print(json.dumps(run_child(["--drop-in"]), indent=1), flush=True)
    print("   torch.profiler, mean device time per kernel launch (3 calls each)")
    prof = run_child(["--profile"])
    for arm, ks in prof.items():
        for k, v in sorted(ks.items()):
            print("  %-10s %-48s %3d launches  %9.1f us" % (arm, k[:48], v["calls"], v["mean_us"]))


if __name__ == "__main__":
    if "--step" in sys.argv:
        child_step(int(sys.argv[sys.argv.index("--step") + 1]))
    elif "--drop-in" in sys.argv:
        child_drop_in()
    elif "--profile" in sys.argv:
        child_profile()
    else:
        main()
