"""Mixed borders at EW size (prepare_first_guess's distribution: 47 % at 20, the rest up to 50): device time of the resident
step with one launch, two border classes (default) and hand-made finer splits."""
import os, sys, time
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import numpy as np, torch
from sea_ice_drift_b200 import synthetic as syn, pmlib, _lib
img1, img2, c1, r1, c2, r2, b, cfg = syn.make_config("cfg2", seed=0)
rng = np.random.default_rng(7); side = img1.shape[0]; nk = 50000
m = syn.rotation_matrix(img1.shape, 2.0)
kx, ky = rng.uniform(40, side - 40, nk), rng.uniform(40, side - 40, nk)
k2x, k2y = syn.apply_affine(m, kx, ky); k2x, k2y = k2x + rng.normal(0, 0.8, nk), k2y + rng.normal(0, 0.8, nk)
pts = list(syn.orb_first_guess_inputs(img1, img2, 200, 35, inset=150, matches=(kx, ky, k2x, k2y)))
brd = pts[4]
print("points", len(brd), "at 20:", int((brd == 20).sum()), "max", brd.max())
ctx = _lib.Context(0); ctx.set_pair(img1, img2)
dev = torch.device("cuda", 0)
stream = torch.cuda.current_stream()
ctx.set_stream(stream.cuda_stream)
def timed(subsets, label, env=None):
    if env: os.environ.update(env)
    ds = []
    for sel in subsets:
        p = [x[sel] for x in pts]
        d = torch.from_numpy(np.stack(p)).to(dev)
        o = torch.empty((len(p[0]), 5), dtype=torch.float64, device=dev)
        ds.append((d, o, int(p[4].max()), len(p[0])))
    def step():
        for d, o, mb, n in ds:
            ctx.run_device(n, *[d[k].data_ptr() for k in range(5)], mb, 35, [-3, 0, 3], 0.0, o.data_ptr())
    for _ in range(3): step()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record(stream)
    for _ in range(10): step()
    e1.record(stream); torch.cuda.synchronize()
    print("%-60s %7.3f ms / step   (%s)" % (label, e0.elapsed_time(e1) / 10, ctx.last_kernel_name), flush=True)
    if env:
        for k in env: del os.environ[k]
    return torch.cat([o for _, o, _, _ in ds]).cpu().numpy()
allp = np.arange(len(brd))
a = timed([allp], "one launch (SID_PM_CLASSES=0)", {"SID_PM_CLASSES": "0"})
bres = timed([allp], "two classes (default)")
print("same table:", np.array_equal(a, bres, equal_nan=True))
for cut in (28, 32, 36, 40):
    timed([np.nonzero(brd <= 20)[0], np.nonzero((brd > 20) & (brd <= cut))[0], np.nonzero(brd > cut)[0]], "three hand-made classes: <=20 | <=%d | rest" % cut, {"SID_PM_CLASSES": "0"})
timed([np.nonzero(brd <= 20)[0], np.nonzero((brd > 20) & (brd <= 28))[0], np.nonzero((brd > 28) & (brd <= 38))[0], np.nonzero(brd > 38)[0]], "four hand-made classes: <=20 | <=28 | <=38 | rest", {"SID_PM_CLASSES": "0"})
for path in ("imma",):
    timed([np.nonzero(brd <= 20)[0]], "the <= 20 class alone", {"SID_PM_CLASSES": "0"})
    timed([np.nonzero(brd > 20)[0]], "the > 20 class alone", {"SID_PM_CLASSES": "0"})
    timed([np.nonzero(brd > 20)[0]], "the > 20 class alone, fused tail forced", {"SID_PM_CLASSES": "0", "SID_PM_SPLIT_TAIL": "0"})
