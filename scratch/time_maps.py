"""Cost of returning the winning maps and templates (Context.run_maps / sid_run_maps) at BASELINE cfg2 on one GPU.

    python scratch/time_maps.py [--rounds 10] [--per-point 300] > OUT

On a resident pair: run vs run_maps -- call time (host clock around the synchronous call), device time of the kernels,
memsets and copies of one call (torch.profiler, in a separate pass), and the bytes each call copies device -> host.
Then the per-point alternative: pmlib.rotate_and_match on the point's window, one call per point, for a sample of
points, extrapolated (and labelled so) to the whole grid.  Needs a CUDA device; there is no CPU path."""
import argparse
import os
import sys
import time

import numpy as np

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from sea_ice_drift_b200 import _lib, pmlib, synthetic as syn   # noqa: E402


def device_times(fn, calls):
    """Sum of CUDA kernel / memset / memcpy time per call, by kind, from torch.profiler."""
    import torch
    from torch.profiler import profile, ProfilerActivity
    torch.cuda.init()
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        for _ in range(calls):
            fn()
        torch.cuda.synchronize()
    kinds = {"kernels": 0.0, "memset": 0.0, "memcpy DtoH": 0.0, "memcpy HtoD": 0.0}
    for ev in prof.events():
        if ev.device_type.name != "CUDA":
            continue
        name = ev.name.lower()
        t = ev.device_time / 1000.0 if hasattr(ev, "device_time") else ev.cuda_time / 1000.0
        if "memset" in name:
            kinds["memset"] += t
        elif "memcpy" in name and "dtoh" in name:
            kinds["memcpy DtoH"] += t
        elif "memcpy" in name and "htod" in name:
            kinds["memcpy HtoD"] += t
        elif "memcpy" not in name:
            kinds["kernels"] += t
    return {k: v / calls for k, v in kinds.items()}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--rounds", type=int, default=10)
    ap.add_argument("--per-point", type=int, default=300)
    args = ap.parse_args()
    import subprocess
    print(subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv"],
                         capture_output=True, text=True).stdout.strip())
    img1, img2, c1, r1, c2, r2, b, cfg = syn.make_config("cfg2", seed=0)
    s, angles = cfg["img_size"], cfg["angles"]
    n = c1.size
    print("cfg2: %d x %d pair, %d points, img_size %d, border %s, angles %s" % (img1.shape[0], img1.shape[1], n, s,
                                                                              cfg["border"], angles))
    ctx = _lib.Context(0)
    ctx.set_pair(img1, img2)
    run = lambda: ctx.run(c1, r1, c2, r2, b, s, angles, 0.0, want_status=True)
    run_maps = lambda: ctx.run_maps(c1, r1, c2, r2, b, s, angles, 0.0, want_status=True)
    tab, st = run()
    tab_m, maps, tpls, st_m = run_maps()
    assert tab.tobytes() == tab_m.tobytes() and np.array_equal(st, st_m)
    packed = int(sum((m.size if m is not None else 0) for m in maps))
    shapes = np.zeros((n, 2), np.int32)
    import ctypes as C
    tot = C.c_int64(0)
    arrs = [np.ascontiguousarray(a, dtype=np.float64) for a in (c1, r1, c2, r2, b)]
    ctx._check(ctx._lib.sid_map_layout(ctx.handle, n, *[a.ctypes.data for a in arrs], s, shapes.ctypes.data, C.byref(tot)))
    print("valid rows %d of %d; layout total %d floats (%.1f MB of maps), valid maps %d floats, templates %.1f MB"
          % (int((st == 1).sum()), n, tot.value, tot.value * 4 / 1e6, packed, n * s * s / 1e6))
    d2h_run = n * 5 * 8 + n * 4
    d2h_maps = d2h_run + tot.value * 4 + n * s * s
    times = {"run": [], "run_maps": []}
    kms = {"run": [], "run_maps": []}
    for _ in range(args.rounds):
        for name, fn in (("run", run), ("run_maps", run_maps)):
            t0 = time.perf_counter()
            fn()
            times[name].append((time.perf_counter() - t0) * 1e3)
            kms[name].append(ctx.last_kernel_ms)
    print("\nresident pair, %d alternating rounds (host clock around the synchronous call; last_kernel_ms = the point "
          "kernel's CUDA events)" % args.rounds)
    for name in ("run", "run_maps"):
        t = np.array(times[name])
        print("  %-9s call  median %8.3f ms  (min %8.3f, max %8.3f)   point kernel median %.3f ms" %
              (name, np.median(t), t.min(), t.max(), float(np.median(kms[name]))))
    print("  bytes device -> host per call: run %.2f MB, run_maps %.2f MB" % (d2h_run / 1e6, d2h_maps / 1e6))
    print("\ndevice time per call by kind (torch.profiler, 3 calls each, separate pass):")
    for name, fn in (("run", run), ("run_maps", run_maps)):
        try:
            dt = device_times(fn, 3)
            print("  %-9s " % name + ", ".join("%s %.3f ms" % (k, v) for k, v in dt.items()))
        except Exception as e:          # the profiler's event API differs between torch versions
            print("  %-9s profiler pass failed: %r" % (name, e))

    # per-point alternative: rotate_and_match on each point's window, one call per point
    k = min(args.per_point, n)
    idx = np.linspace(0, n - 1, k).astype(int)
    hws = int(s / 2.)
    wins = [img2[int(r2[i] - hws - b[i]):int(r2[i] + hws + b[i] + 1), int(c2[i] - hws - b[i]):int(c2[i] + hws + b[i] + 1)]
            for i in idx]
    pmlib.rotate_and_match(img1, c1[idx[0]], r1[idx[0]], s, wins[0], 0.0, angles=angles, template_matcher=None)
    t0 = time.perf_counter()
    agree = 0
    for j, i in enumerate(idx):
        res = pmlib.rotate_and_match(img1, c1[i], r1[i], s, wins[j], 0.0, angles=angles, template_matcher=None)
        if st[i] == 1 and res[5].tobytes() == maps[i].tobytes() and np.array_equal(res[6], tpls[i]):
            agree += 1
    per = (time.perf_counter() - t0) / k
    print("\nper-point pmlib.rotate_and_match loop: %d points measured, %.2f ms per point (maps / templates equal to "
          "run_maps for %d of %d valid sampled rows)" % (k, per * 1e3, agree, int((st[idx] == 1).sum())))
    print("  EXTRAPOLATED to the %d-point grid (not measured): %.1f s per grid, against one run_maps call" % (n, per * n))
    ctx.close()


if __name__ == "__main__":
    main()
