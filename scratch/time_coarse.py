"""Cost and accuracy of drift without feature tracking (pmlib.coarse_tracking) on one GPU.

    python scratch/time_coarse.py

1. sid::downsample_kernel on the EW pair (10400 x 10400 each, 216 MB read: larger than the 126 MB L2): CUDA events around
   200 launches per factor on the context's stream, bytes read + written over the time, against 7.7 TB/s.
2. bench.py's drop_in_ew scene (the EW pair with cfg2's 2 degree rotation, 200 x 200 grid, angles [-3, 0, 3], img_size
   35): the coarse stage alone (coarse_tracking), the whole get_drift_PM(..., *get_drift_coarse()) call, and the ORB
   route (synthetic.orb_matches on the host cores, then get_drift_PM) -- median of 5 calls after one warm-up call each --
   with the median / p90 error of the final vectors against the known drift (minus the reference's -1 px template-centre
   bias, as bench.py measures it) and whether prepare_first_guess stayed on the device; for step 8, 12, 16, 24 and 32.
   Before that, the coarse stage at the default step 32 step by step (upload, downsampling, lattice, matching, selection).
3. Which kernels ran in one coarse route call (torch.profiler, its own pass after the timings)."""
import contextlib
import io
import json
import os
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)


def downsample_bandwidth(img1, img2):
    import torch
    from sea_ice_drift_b200 import _lib
    ctx = _lib.Context(0)
    stream = torch.cuda.current_stream()
    ctx.set_stream(stream.cuda_stream)
    ctx.set_pair(img1, img2)
    rows = []
    for k in (2, 4, 8, 16):
        shape = (img1.shape[0] // k, img1.shape[1] // k)
        pitch, nbytes = _lib.pair_layout(*shape)
        bufs = [torch.zeros(nbytes, dtype=torch.uint8, device="cuda:0") for _ in range(2)]
        args = [(b.data_ptr(), pitch, nbytes) for b in bufs]
        for _ in range(10):
            ctx.downsample_pair(k, *args)
        ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        n = 200
        ev0.record(stream)
        for _ in range(n):
            ctx.downsample_pair(k, *args)
        ev1.record(stream)
        torch.cuda.synchronize()
        us = ev0.elapsed_time(ev1) * 1e3 / n
        moved = 2 * (shape[0] * k) * (shape[1] * k) + 2 * shape[0] * shape[1]
        rows.append(dict(factor=k, us_per_launch=us, bytes=moved, tb_per_s=moved / us / 1e6,
                         share_of_7_7_tb_s=moved / us / 1e6 / 7.7))
    ctx.set_stream(None)
    ctx.close()
    return rows


def coarse_breakdown(img1, img2, n1, n2, step=32, reps=5):
    """coarse_tracking's steps one by one, each ended by a synchronise: upload of the pair, downsampling, lattice and
    first guess on the host, matching on the private context, selection and mapping (medians over ``reps``)."""
    import torch
    from sea_ice_drift_b200 import _lib, pmlib
    k, s = 4, 35
    ctx = _lib.default_context()
    coarse = _lib.Context(0)
    shapes = [(img1.shape[0] // k, img1.shape[1] // k), (img2.shape[0] // k, img2.shape[1] // k)]
    bufs = []
    for w, shape in enumerate(shapes):
        pitch, nbytes = _lib.pair_layout(*shape)
        b = pmlib._coarse_buffer(0, w, (shape, k), nbytes)
        bufs.append((b.data_ptr(), pitch, b.numel()))
    torch.cuda.synchronize()
    t = {"set_pair": [], "downsample": [], "lattice_first_guess": [], "match": [], "select": []}
    for _ in range(reps + 1):
        t0 = time.perf_counter()
        ctx.set_pair(img1, img2)
        ctx.synchronize()
        t1 = time.perf_counter()
        ctx.downsample_pair(k, *bufs)
        ctx.synchronize()
        t2 = time.perf_counter()
        c1, r1, c2fg, r2fg, border, alpha0 = pmlib.coarse_inputs(n1, n2, shapes[0], shapes[1], k, step, s, 100.0)
        t3 = time.perf_counter()
        coarse.adopt_pair_device(bufs[0][0], shapes[0], bufs[0][1], bufs[0][2], bufs[1][0], shapes[1], bufs[1][1], bufs[1][2])
        table, status = coarse.run(c1, r1, c2fg, r2fg, border, s, [-3, 0, 3], alpha0, 0, _lib.SID_HES_NORM, want_status=True)
        t4 = time.perf_counter()
        pmlib.coarse_matches(table, status, c1, r1, k, s, 4.0)
        t5 = time.perf_counter()
        for key, a, b in (("set_pair", t0, t1), ("downsample", t1, t2), ("lattice_first_guess", t2, t3),
                          ("match", t3, t4), ("select", t4, t5)):
            t[key].append((b - a) * 1e3)
    kname = coarse.last_kernel_name
    coarse.close()
    return {key: float(np.median(v[1:])) for key, v in t.items()}, int(c1.size), kname


def quiet(fn, *a, **k):
    with contextlib.redirect_stdout(io.StringIO()):
        return fn(*a, **k)


def timed(fn, n=5):
    quiet(fn)
    ts, res = [], None
    for _ in range(n):
        t0 = time.perf_counter()
        res = quiet(fn)
        ts.append(time.perf_counter() - t0)
    return float(np.median(ts)) * 1e3, res


def main():
    import torch
    from sea_ice_drift_b200 import pmlib, synthetic as syn
    from sea_ice_drift_b200.seaicedrift import SeaIceDrift
    out = {"gpu": torch.cuda.get_device_name(0)}
    img1, img2, _, _, _, _, _, cfg = syn.make_config("cfg2", seed=0)
    out["downsample"] = downsample_bandwidth(img1, img2)
    for r in out["downsample"]:
        print("downsample_kernel factor %2d: %7.1f us per launch (both images), %.3f GB moved, %.2f TB/s = %.0f %% of 7.7 TB/s"
              % (r["factor"], r["us_per_launch"], r["bytes"] / 1e9, r["tb_per_s"], 100 * r["share_of_7_7_tb_s"]), flush=True)

    side = img1.shape[0]
    n1, n2 = syn.ArrayDomain(img1), syn.ArrayDomain(img2)
    gx, gy = np.meshgrid(np.linspace(150, side - 150, 200), np.linspace(150, side - 150, 200))
    lon, lat = n2.transform_points(gx, gy)
    sid = SeaIceDrift(n1, n2)
    kw = dict(angles=[-3, 0, 3], img_size=35)

    def errors(res):
        ok = np.isfinite(res[0])
        c2, r2 = n2.transform_points(res[5][ok], res[6][ok], 1)
        c1g, r1g = n1.transform_points(lon[ok], lat[ok], 1)
        tx, ty = syn.apply_affine(cfg["matrix"], c1g, r1g)
        e = np.hypot(c2 - (tx - 1), r2 - (ty - 1))
        return int(ok.sum()), float(np.median(e)), float(np.percentile(e, 90))

    real_near = pmlib.interpolation_near
    host_calls = [0]

    def counting_near(*a, **k):
        host_calls[0] += 1
        return real_near(*a, **k)
    pmlib.interpolation_near = counting_near

    bd, n_pts, kname = coarse_breakdown(img1, img2, n1, n2)
    out["coarse_breakdown_ms_step32"] = bd
    print("coarse stage at step 32 (the default), factor 4 (%d lattice points, matched by %s), ms: %s" % (n_pts, kname, json.dumps(bd)),
          flush=True)

    routes = {}
    for step in (8, 12, 16, 24, 32):
        ms_coarse, ll = timed(lambda: sid.get_drift_coarse(step=step))
        host_calls[0] = 0
        ms_all, res = timed(lambda: sid.get_drift_PM(lon, lat, *sid.get_drift_coarse(step=step), **kw))
        valid, med, p90 = errors(res)
        routes["coarse_step%d" % step] = dict(matches=int(ll[0].size), ms_coarse_stage=ms_coarse, ms_whole_call=ms_all,
                                              valid=valid, median_error_px=med, p90_error_px=p90,
                                              first_guess_device=host_calls[0] == 0)
        print("coarse step %2d: %d matches, coarse stage %.1f ms, whole get_drift_PM(..., *get_drift_coarse()) %.1f ms, "
              "%d valid, error median %.3f p90 %.3f px, device first guess: %s"
              % (step, ll[0].size, ms_coarse, ms_all, valid, med, p90, host_calls[0] == 0), flush=True)

    t0 = time.perf_counter()
    x1, y1, x2, y2 = syn.orb_matches(img1, img2)
    orb_s = time.perf_counter() - t0
    ll = n1.transform_points(x1, y1) + n2.transform_points(x2, y2)
    host_calls[0] = 0
    ms_pm, res = timed(lambda: sid.get_drift_PM(lon, lat, *ll, **kw))
    valid, med, p90 = errors(res)
    routes["orb"] = dict(matches=int(x1.size), s_feature_tracking_host=orb_s, host_cores=os.cpu_count(),
                         ms_get_drift_PM=ms_pm, ms_whole=orb_s * 1e3 + ms_pm, valid=valid, median_error_px=med,
                         p90_error_px=p90, first_guess_device=host_calls[0] == 0)
    print("ORB route: %d matches, feature tracking %.2f s on %d host cores, get_drift_PM %.1f ms, %d valid, error median "
          "%.3f p90 %.3f px, device first guess: %s" % (x1.size, orb_s, os.cpu_count(), ms_pm, valid, med, p90,
                                                         host_calls[0] == 0), flush=True)
    out["drop_in_ew"] = routes
    pmlib.interpolation_near = real_near

    from torch.profiler import profile, ProfilerActivity
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        quiet(lambda: sid.get_drift_PM(lon, lat, *sid.get_drift_coarse(), **kw))
        torch.cuda.synchronize()
    kernels = {}
    for ev in prof.events():
        if ev.device_type.name == "CUDA" and "memcpy" not in ev.name.lower() and "memset" not in ev.name.lower():
            name = ev.name.split("(")[0].split("<")[0]
            n, t = kernels.get(name, (0, 0.0))
            kernels[name] = (n + 1, t + ev.device_time / 1e3)
    out["kernels"] = {k: dict(launches=n, ms=t) for k, (n, t) in sorted(kernels.items())}
    for k, (n, t) in sorted(kernels.items(), key=lambda kv: -kv[1][1]):
        print("  kernel %-40s %3d launches %8.3f ms" % (k, n, t))
    print(json.dumps(out))


if __name__ == "__main__":
    main()
