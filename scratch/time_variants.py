"""Time the fused kernel on a full workload under launch variants (env overrides read per launch)."""
import os, sys, time
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import numpy as np, torch
from sea_ice_drift_b200 import _lib, synthetic as syn

name = sys.argv[1] if len(sys.argv) > 1 else "cfg2"
kw = {}
if len(sys.argv) > 2: kw = dict(side=int(sys.argv[2]), grid=int(sys.argv[3]))
img1, img2, c1, r1, c2, r2, b, cfg = syn.make_config(name, seed=0, **kw)
n = len(c1); s = cfg["img_size"]; angles = cfg["angles"]
dev = torch.device("cuda", 0)
ctx = _lib.Context(0)
stream = torch.cuda.Stream()
ctx.set_stream(stream.cuda_stream)
ctx.set_pair(img1, img2)
d_pts = torch.from_numpy(np.stack([c1, r1, c2, r2, b])).to(dev)
d_out = torch.empty((n, 5), dtype=torch.float64, device=dev); d_st = torch.empty(n, dtype=torch.int32, device=dev)
ptrs = [d_pts[k].data_ptr() for k in range(5)]
flops = (len(angles) * 2.0 * s * s * (2 * b + 1 + (s % 2 == 0)) ** 2).sum()
ref = None
def run(label, env, reps=5):
    global ref
    for k in ("SID_PM_GLOBAL_SCRATCH", "SID_PM_PATH", "SID_PM_TMA", "SID_PM_SPLIT_TAIL"): os.environ.pop(k, None)
    os.environ.update(env)
    with torch.cuda.stream(stream):
        for _ in range(2): ctx.run_device(n, *ptrs, int(b.max()), s, angles, 0.0, d_out.data_ptr(), d_st.data_ptr())
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record(stream)
        for _ in range(reps): ctx.run_device(n, *ptrs, int(b.max()), s, angles, 0.0, d_out.data_ptr(), d_st.data_ptr())
        e1.record(stream)
    torch.cuda.synchronize()
    ms = e0.elapsed_time(e1) / reps
    out = d_out.cpu().numpy()
    same = True if ref is None else np.array_equal(out, ref, equal_nan=True)
    if ref is None: ref = out
    print("%-34s %8.3f ms  %7.2f Mvec/s  %6.1f TFLOP/s-eq  (%.0f%% of FP32-FMA peak 74.4)  same_as_first=%s" % (
        label, ms, n / ms / 1e3, flops / ms / 1e9, 100 * flops / ms / 1e9 / 74.45, same), flush=True)
print(name, "points", n, "angles", angles, "s", s, "border", cfg["border"])
run("imma, TMA, split tail", {})
run("imma, TMA, fused tail", {"SID_PM_SPLIT_TAIL": "0"})
run("dp4a, TMA, split tail", {"SID_PM_PATH": "dp4a"})
