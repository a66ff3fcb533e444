"""Dispatch A/B of two library builds: python scratch/ab_dispatch.py old=path1.so new=path2.so [--quick]

Runs the same matching calls on each library (SID_LIBRARY, one subprocess per library) with SID_DEBUG=1 and compares,
byte for byte, everything a call leaves: return code and error text, launch count, sid_last_kernel_name, the SID_DEBUG
launch / tail / refuse lines, the result table, the status, the winning maps and the templates.  Cases: img_size x border
(1 up to one past the largest accepted) x angles x flag set x SID_PM_PATH, each through sid_run, sid_run_pair (pinned and
pageable images, three upload bands), sid_run_device and sid_run_maps; mixed-border point sets that split into border
classes; the largest border sid_run accepts.  Prints the differing lines and exits 1 when the libraries disagree."""
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))

CHILD = r'''
import hashlib, os, sys
sys.path.insert(0, %r)
import numpy as np
import torch
from sea_ice_drift_b200 import _lib, synthetic as syn

QUICK = "--quick" in sys.argv
SIDE = 1200
SIZES = [2, 3, 4, 21, 35, 50, 65, 80, 96, 112, 113, 128]
BORDERS = [1, 2, 3, 4, 8, 16, 20, 21, 22, 23, 24, 32, 48, 64, 100, 125, 144, 209, 212]
FEW_BORDERS = [1, 20, 24]             # flag sets that do not enter the dispatch (rot_order, hes_norm, mcc_norm)
ANGLES = {"a1": [3], "a3": [0, 3, -3], "a7": [-9, -6, -3, 0, 3, 6, 9], "a21": list(range(-10, 11))}
FLAGS = {"default": (0, _lib.flags_from_kwargs()), "rot_order1": (1, _lib.flags_from_kwargs()),
         "raw_hes": (0, _lib.flags_from_kwargs(hes_norm=False)), "mcc_norm": (0, _lib.flags_from_kwargs(mcc_norm=True)),
         "hes_smth": (0, _lib.flags_from_kwargs(hes_smth=True))}
PATH = sys.argv[sys.argv.index("--path") + 1]          # SID_PM_PATH of this run ("default": unset)
if QUICK:
    SIZES, BORDERS = [3, 35, 128], [1, 20, 24, 48, 144, 212]
    FLAGS = {k: FLAGS[k] for k in ("default", "hes_smth")}

m = syn.rotation_matrix((SIDE, SIDE), 3.0)
img1 = syn.speckle_image((SIDE, SIDE), seed=23)
img2 = syn.warp_pair(img1, m, seed=23)
img1 = img1.copy()
img1[299:302, 299:302] = 0                                   # a template of zeros: NaN row
pin1 = torch.empty(img1.shape, dtype=torch.uint8, pin_memory=True).numpy(); pin1[:] = img1
pin2 = torch.empty(img2.shape, dtype=torch.uint8, pin_memory=True).numpy(); pin2[:] = img2
ctx = _lib.Context(0)


def points(border):
    """3 x 3 grid around the centre, fractional first guess / border, a NaN row, rejected and clipped windows."""
    mid = SIDE / 2.
    gx, gy = np.meshgrid(mid + np.array([-30., 0., 30.]), mid + np.array([-25., 0., 25.]))
    c1, r1 = list(gx.ravel()), list(gy.ravel())
    c2, r2 = [list(np.round(v)) for v in syn.apply_affine(m, np.array(c1), np.array(r1))]
    b = [float(border)] * len(c1)
    for row in ((mid - 20, mid + 20, mid - 19.5, mid + 19.75, border - 0.5), (300.5, 300.5, 300.5, 300.5, border),
                (mid, mid, 5.0, mid, border), (np.nan, mid, mid, mid, border), (mid, mid, SIDE - 30.0, mid - 10, border)):
        for v, x in zip((c1, r1, c2, r2, b), row):
            v.append(x)
    return [np.asarray(v, dtype=np.float64) for v in (c1, r1, c2, r2, b)]


def mixed_points(n_side=25):
    """A grid with most borders at 20 and the rest 21 ... 45: the calls split into two border classes."""
    g = np.linspace(260, SIDE - 260, n_side)
    gx, gy = np.meshgrid(g, g)
    c1, r1 = gx.ravel(), gy.ravel()
    c2, r2 = [np.round(v) for v in syn.apply_affine(m, c1, r1)]
    rng = np.random.default_rng(5)
    b = np.where(rng.random(c1.size) < 0.8, 20.0, rng.integers(21, 46, c1.size).astype(np.float64))
    return [c1, r1, c2, r2, b]


def digest(*arrays):
    h = hashlib.sha256()
    for a in arrays:
        h.update(np.ascontiguousarray(a).tobytes())
    return h.hexdigest()[:20]


def call(tag, fn):
    sys.stderr.write("== %%s\n" %% tag)
    sys.stderr.flush()
    before = ctx.launch_count
    try:
        res = "ok " + fn()
    except Exception as e:                                   # SidError / ValueError: code and message
        res = "%%s: %%s" %% (type(e).__name__, e)
    sys.stderr.flush()
    print("%%s | %%s | launches %%d | %%s" %% (tag, res, ctx.launch_count - before, ctx.last_kernel_name), flush=True)


def entries(tag, pts, s, ang, rot, flags):
    def run():
        out, st = ctx.run(*pts, s, ang, 0.0, rot_order=rot, flags=flags, want_status=True)
        return digest(out, st)

    def run_pair(pinned):
        def f():
            os.environ["SID_BANDS"] = "3"
            try:
                a, b = (pin1, pin2) if pinned else (img1, img2)
                out, st = ctx.run_pair(a, b, *pts, s, ang, 0.0, rot_order=rot, flags=flags, want_status=True)
            finally:
                del os.environ["SID_BANDS"]
            return digest(out, st)
        return f

    def run_device():
        ctx.set_pair(img1, img2)
        d = [torch.from_numpy(np.ascontiguousarray(v)).cuda() for v in pts]
        out = torch.full((pts[0].size, 5), float("nan"), dtype=torch.float64, device="cuda")
        st = torch.zeros(pts[0].size, dtype=torch.int32, device="cuda")
        torch.cuda.synchronize()
        ctx.run_device(pts[0].size, *[t.data_ptr() for t in d], 0, s, ang, 0.0, out.data_ptr(), st.data_ptr(),
                       rot_order=rot, flags=flags)
        ctx.synchronize()
        return digest(out.cpu().numpy(), st.cpu().numpy())

    def run_maps():
        out, maps, tpl, st = ctx.run_maps(*pts, s, ang, 0.0, rot_order=rot, flags=flags, want_status=True)
        return digest(out, st, tpl, *[x for x in maps if x is not None])

    ctx.set_pair(img1, img2)
    call(tag + " run", run)
    call(tag + " run_pair_pinned", run_pair(True))
    call(tag + " run_pair_pageable", run_pair(False))
    call(tag + " run_device", run_device)
    ctx.set_pair(img1, img2)
    call(tag + " run_maps", run_maps)


def largest_accepted(s, ang):
    pts = points(1)
    lo, hi = 1, 1024
    ctx.set_pair(img1, img2)
    while hi - lo > 1:
        mid = (lo + hi) // 2
        try:
            ctx.run(*pts[:4], np.full(pts[0].size, float(mid)), s, ang, 0.0)
            lo = mid
        except Exception:
            hi = mid
    return lo


if PATH != "default":
    os.environ["SID_PM_PATH"] = PATH
for s in SIZES:
    for an, ang in ANGLES.items():
        top = largest_accepted(s, ang)
        print("largest %%s s%%d %%s %%d" %% (PATH, s, an, top), flush=True)
        borders = sorted(set(b for b in BORDERS if b <= top + 1) | {top, top + 1})
        for fn, (rot, flags) in FLAGS.items():
            few = fn not in ("default", "hes_smth")
            for b in [b for b in borders if b in FEW_BORDERS or b >= top] if few else borders:
                entries("%%s s%%d %%s %%s b%%d" %% (PATH, s, an, fn, b), points(b), s, ang, rot, flags)
for s in (21, 35, 50, 65):
    for an, ang in ANGLES.items():
        for fn, (rot, flags) in FLAGS.items():
            entries("%%s s%%d %%s %%s mixed" %% (PATH, s, an, fn), mixed_points(), s, ang, rot, flags)
''' % ROOT


def compare(libs, extra):
    """Both libraries on the same calls; returns the number of differing lines."""
    res = {}
    for name, path in libs:
        env = dict(os.environ, SID_LIBRARY=os.path.abspath(path), SID_DEBUG="1")
        for k in ("SID_PM_PATH", "SID_BANDS", "SID_BAND_PLAN", "SID_PM_CLASSES", "SID_PM_SPLIT_TAIL"):
            env.pop(k, None)
        p = subprocess.run([sys.executable, "-c", CHILD] + extra, env=env, capture_output=True, text=True)
        if p.returncode:
            sys.stderr.write(p.stderr[-4000:])
            raise SystemExit("%s: child exited with %d" % (name, p.returncode))
        res[name] = (p.stdout.splitlines(), p.stderr.splitlines())
    (na, (oa, ea)), (nb, (ob, eb)) = list(res.items())
    bad = 0
    for what, a, b in (("result", oa, ob), ("stderr", ea, eb)):
        if len(a) != len(b):
            print("%s: %d lines (%s) vs %d lines (%s)" % (what, len(a), na, len(b), nb))
            bad += 1
        for i, (x, y) in enumerate(zip(a, b)):
            if x != y:
                bad += 1
                if bad <= 40:
                    print("%s line %d differs:\n  %s: %s\n  %s: %s" % (what, i, na, x, nb, y))
    cases = sum(1 for x in oa if " | " in x)
    refused = sum(1 for x in oa if " | ok " not in x and " | " in x)
    print("%s: %d calls (%d refused), %d result lines, %d stderr lines: %s" %
          (" ".join(extra), cases, refused, len(oa), len(ea), "IDENTICAL" if bad == 0 else "%d DIFFERENCES" % bad), flush=True)
    return bad


def main():
    libs = [a.split("=", 1) for a in sys.argv[1:] if "=" in a]
    extra = [a for a in sys.argv[1:] if a.startswith("--")]
    assert len(libs) == 2, __doc__
    bad = sum(compare(libs, extra + ["--path", path]) for path in ("default", "ws", "tc", "imma", "dp4a"))
    raise SystemExit(1 if bad else 0)


if __name__ == "__main__":
    main()
