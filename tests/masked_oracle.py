"""TEST INFRASTRUCTURE ONLY -- ctypes front-end of the masked-correlation oracle (tests/masked_oracle.c, which includes
oracle/mcc_oracle.c unchanged).  Same calling conventions as oracle/c_oracle.py; the library is compiled on first use
into the temporary directory, keyed by the hash of both sources."""
import ctypes as C
import hashlib
import os
import subprocess
import tempfile
import threading

import numpy as np

from oracle.angle_table import angle_table

HERE = os.path.dirname(os.path.abspath(__file__))
SOURCES = [os.path.join(HERE, "masked_oracle.c"), os.path.join(os.path.dirname(HERE), "oracle", "mcc_oracle.c")]
_u8p, _f32p, _f64p, _i32p = C.POINTER(C.c_uint8), C.POINTER(C.c_float), C.POINTER(C.c_double), C.POINTER(C.c_int)
_lib = None
_lock = threading.Lock()


def lib():
    global _lib
    with _lock:
        if _lib is None:
            digest = hashlib.sha256(b"".join(open(p, "rb").read() for p in SOURCES)).hexdigest()[:16]
            path = os.path.join(tempfile.gettempdir(), "sid_masked_oracle_%s_%d.so" % (digest, os.getuid()))
            if not os.path.exists(path):
                tmp = "%s.tmp.%d" % (path, os.getpid())
                subprocess.check_call(["gcc", "-O2", "-fPIC", "-shared", "-std=c11", "-ffp-contract=off",
                                       "-fno-fast-math", "-o", tmp, SOURCES[0], "-lm"])
                os.replace(tmp, path)
            _lib = C.CDLL(path)
    return _lib


def _u8(a):
    a = np.asarray(a)
    if a.dtype != np.uint8 or a.ndim != 2 or a.strides[1] != 1:
        a = np.ascontiguousarray(a, dtype=np.uint8)
    return a


def _ptr(a, t):
    return a.ctypes.data_as(t)


def match_template_masked(image, templ):
    """The masked rule with mask = (templ > 0) on every position of ``image`` (sido_match_template_masked)."""
    image = _u8(image)
    templ = np.ascontiguousarray(templ, dtype=np.uint8)
    H, W = image.shape
    s = templ.shape[0]
    if templ.shape != (s, s):
        raise ValueError("square template only")
    out = np.zeros((H - s + 1, W - s + 1), np.float32)
    rc = lib().sido_match_template_masked(_ptr(image, _u8p), C.c_int(H), C.c_int(W), C.c_int64(image.strides[0]),
                                          _ptr(templ, _u8p), C.c_int(s), _ptr(out, _f32p))
    if rc:
        raise ValueError("sido_match_template_masked rc=%d" % rc)
    return out


def rotate_and_match(img1, c1, r1, img_size, image2, alpha0, angles=[-3, 0, 3], mcc_norm=False, rot_order=0,
                     hes_norm=True, hes_smth=False, **kwargs):
    """oracle.c_oracle.rotate_and_match with the masked rule: ``(dc, dr, angle, r, h, map, template, valid)``, valid 1
    for a row matched as the reference does, 2 for a masked row; seven NaNs and 0 for a NaN row."""
    img1, image2 = _u8(img1), _u8(image2)
    tab = angle_table(angles, alpha0, img_size)
    H, W = image2.shape
    res = np.zeros((H - img_size + 1, W - img_size + 1), np.float32)
    tpl = np.zeros((img_size, img_size), np.uint8)
    valid, ba = C.c_int(0), C.c_int(-1)
    dc, dr = C.c_double(0), C.c_double(0)
    br, bh = C.c_float(0), C.c_float(0)
    rc = lib().sido_rotate_and_match_ex(
        _ptr(img1, _u8p), C.c_int(img1.shape[0]), C.c_int(img1.shape[1]), C.c_int64(img1.strides[0]),
        C.c_double(c1), C.c_double(r1), C.c_int(img_size),
        _ptr(image2, _u8p), C.c_int(H), C.c_int(W), C.c_int64(image2.strides[0]),
        C.c_int(len(angles)), _ptr(tab, _f64p), C.c_int(rot_order),
        C.c_int(bool(hes_norm)), C.c_int(bool(hes_smth)), C.c_int(bool(mcc_norm)),
        C.byref(valid), C.byref(dc), C.byref(dr), C.byref(ba), C.byref(br), C.byref(bh),
        _ptr(res, _f32p), _ptr(tpl, _u8p), C.c_int(1))
    if rc:
        raise ValueError("sido_rotate_and_match_ex rc=%d" % rc)
    if not valid.value:
        return (np.nan,) * 7 + (0,)
    return (dc.value, dr.value, angles[ba.value], np.float32(br.value), np.float32(bh.value), res, tpl, valid.value)


def use_mcc_batch(c1, r1, c2fg, r2fg, border, img1, img2, img_size, alpha0, angles=[-3, 0, 3], mcc_norm=False,
                  rot_order=0, hes_norm=True, hes_smth=False, **kwargs):
    """oracle.c_oracle.use_mcc_batch with the masked rule -> (n, 5) float64, status (n,) with 2 for masked rows."""
    img1, img2 = _u8(img1), _u8(img2)
    arrs = [np.ascontiguousarray(np.atleast_1d(x), dtype=np.float64) for x in (c1, r1, c2fg, r2fg, border)]
    n = arrs[0].size
    tab = angle_table(angles, alpha0, img_size)
    ang = np.ascontiguousarray(np.asarray(angles, dtype=np.float64))
    out = np.full((n, 5), np.nan, np.float64)
    status = np.zeros(n, np.int32)
    rc = lib().sido_use_mcc_batch_ex(
        C.c_int64(n), *[_ptr(a, _f64p) for a in arrs],
        _ptr(img1, _u8p), C.c_int(img1.shape[0]), C.c_int(img1.shape[1]), C.c_int64(img1.strides[0]),
        _ptr(img2, _u8p), C.c_int(img2.shape[0]), C.c_int(img2.shape[1]), C.c_int64(img2.strides[0]),
        C.c_int(img_size), C.c_int(len(angles)), _ptr(ang, _f64p), _ptr(tab, _f64p),
        C.c_int(rot_order), C.c_int(bool(hes_norm)), C.c_int(bool(hes_smth)), C.c_int(bool(mcc_norm)),
        _ptr(out, _f64p), _ptr(status, _i32p), C.c_int(1))
    if rc:
        raise ValueError("sido_use_mcc_batch_ex rc=%d" % rc)
    return out, status
