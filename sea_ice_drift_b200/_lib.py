"""ctypes binding of the C ABI declared in include/sid_b200.h.

The CUDA library is the only compute path: there is no CPU fallback.  If the
shared object is missing it is built in-tree with nvcc; if that fails, or no CUDA
device is usable, every entry point raises.
"""
import ctypes as C
import os
import threading

import numpy as np

from . import _build

_u8p = C.POINTER(C.c_uint8)
_f32p = C.POINTER(C.c_float)
_f64p = C.POINTER(C.c_double)
_i32p = C.POINTER(C.c_int)

SID_TM_CCOEFF_NORMED = 5
SID_HES_NORM, SID_HES_SMTH, SID_MCC_NORM = 1, 2, 4
SID_SUBPIXEL = 8                # extension: sub-pixel c2 / r2 (include/sid_b200.h)
SID_MASKED = 16                 # extension: masked correlation for templates with 0 pixels (include/sid_b200.h)
SID_PEAKS = 32                  # extension: the secondary peaks of every row's winning map (include/sid_b200.h)
SID_N_PEAKS = 3                 # secondary peaks recorded per row
SID_UNCERT = 64                 # extension: covariance of every row's sub-pixel offsets (include/sid_b200.h)
SID_PT_VALID = 1                # point status of a valid row (sid_run*)
SID_PT_MASKED = 2               # point status of a row matched by the masked rule (SID_MASKED)

EXPORTS = [
    "sid_version", "sid_create", "sid_destroy", "sid_last_error", "sid_set_stream", "sid_synchronize",
    "sid_set_pair", "sid_set_pair_device", "sid_pair_layout", "sid_adopt_pair_device", "sid_upload_rows", "sid_pm_epilogue_affine", "sid_first_guess", "sid_run", "sid_run_pair", "sid_run_device", "sid_map_layout", "sid_run_maps", "sid_launch_count", "sid_last_kernel_ms", "sid_last_kernel_name",
    "sid_rotate_and_match", "sid_get_template", "sid_match_template", "sid_get_hessian", "sid_knn_hamming2",
    "sid_deformation", "sid_downsample_pair", "sid_get_peaks", "sid_filter_outliers", "sid_get_uncertainty",
]

_lib = None
_lock = threading.Lock()


class SidError(RuntimeError):
    pass


def load_library():
    """Load (building first if needed) libsid_b200.so and declare its prototypes."""
    global _lib
    with _lock:
        if _lib is not None:
            return _lib
        path = os.environ.get("SID_LIBRARY")          # an experimental build for A/B runs (scratch/ab_build.sh)
        if not path:
            path = _build.LIB
            if _build.is_stale():
                path = _build.build()
        lib = C.CDLL(path)
        lib.sid_version.restype = C.c_char_p
        lib.sid_last_error.restype = C.c_char_p
        lib.sid_last_error.argtypes = [C.c_void_p]
        lib.sid_create.argtypes = [C.POINTER(C.c_void_p), C.c_int]
        lib.sid_destroy.argtypes = [C.c_void_p]
        lib.sid_destroy.restype = None
        lib.sid_set_stream.argtypes = [C.c_void_p, C.c_void_p]
        lib.sid_synchronize.argtypes = [C.c_void_p]
        lib.sid_launch_count.argtypes = [C.c_void_p]
        lib.sid_launch_count.restype = C.c_int64
        lib.sid_last_kernel_ms.argtypes = [C.c_void_p]
        lib.sid_last_kernel_ms.restype = C.c_double
        lib.sid_last_kernel_name.argtypes = [C.c_void_p]
        lib.sid_last_kernel_name.restype = C.c_char_p
        pair = [C.c_void_p, C.c_void_p, C.c_int, C.c_int, C.c_int64, C.c_void_p, C.c_int, C.c_int, C.c_int64]
        lib.sid_set_pair.argtypes = pair
        lib.sid_set_pair_device.argtypes = pair
        lib.sid_pair_layout.argtypes = [C.c_int, C.c_int, C.POINTER(C.c_int64), C.POINTER(C.c_int64)]
        lib.sid_adopt_pair_device.argtypes = [C.c_void_p, C.c_void_p, C.c_int, C.c_int, C.c_int64, C.c_int64,
                                              C.c_void_p, C.c_int, C.c_int, C.c_int64, C.c_int64]
        lib.sid_pm_epilogue_affine.argtypes = [C.c_void_p, C.c_int64, C.c_void_p, C.c_int64] + [C.c_void_p] * 6
        lib.sid_first_guess.argtypes = [C.c_void_p, C.c_int] + [C.c_void_p] * 4 + [C.c_int] + [C.c_void_p] * 2 + \
            [C.c_int64] + [C.c_void_p] * 6
        lib.sid_downsample_pair.argtypes = [C.c_void_p, C.c_int, C.c_void_p, C.c_int64, C.c_int64,
                                            C.c_void_p, C.c_int64, C.c_int64]
        lib.sid_upload_rows.argtypes = [C.c_void_p, C.c_void_p, C.c_int64, C.c_void_p, C.c_int64, C.c_int, C.c_int]
        lib.sid_run.argtypes = [C.c_void_p, C.c_int64] + [C.c_void_p] * 5 + \
            [C.c_int, C.c_int, C.c_void_p, C.c_void_p, C.c_int, C.c_uint, C.c_int, C.c_void_p, C.c_void_p]
        lib.sid_run_pair.argtypes = pair + [C.c_int64] + [C.c_void_p] * 5 + \
            [C.c_int, C.c_int, C.c_void_p, C.c_void_p, C.c_int, C.c_uint, C.c_int, C.c_void_p, C.c_void_p]
        lib.sid_run_device.argtypes = [C.c_void_p, C.c_int64] + [C.c_void_p] * 5 + \
            [C.c_int, C.c_int, C.c_int, C.c_void_p, C.c_void_p, C.c_int, C.c_uint, C.c_int, C.c_void_p, C.c_void_p]
        lib.sid_map_layout.argtypes = [C.c_void_p, C.c_int64] + [C.c_void_p] * 5 + [C.c_int, C.c_void_p, C.POINTER(C.c_int64)]
        lib.sid_run_maps.argtypes = lib.sid_run.argtypes + [C.c_int64, C.c_void_p, C.c_void_p]
        lib.sid_rotate_and_match.argtypes = [
            C.c_void_p, C.c_void_p, C.c_int, C.c_int, C.c_int64, C.c_double, C.c_double, C.c_int,
            C.c_void_p, C.c_int, C.c_int, C.c_int64, C.c_int, C.c_void_p, C.c_int, C.c_uint, C.c_int,
            _i32p, _f64p, _f64p, _i32p, _f32p, _f32p, C.c_void_p, C.c_void_p]
        lib.sid_get_template.argtypes = [C.c_void_p, C.c_void_p, C.c_int, C.c_int, C.c_int64, C.c_double,
                                         C.c_double, C.c_void_p, C.c_int, C.c_int, C.c_void_p]
        lib.sid_match_template.argtypes = [C.c_void_p, C.c_void_p, C.c_int, C.c_int, C.c_int64, C.c_void_p,
                                           C.c_int, C.c_int, C.c_int64, C.c_int, C.c_void_p]
        lib.sid_knn_hamming2.argtypes = [C.c_void_p, C.c_void_p, C.c_int, C.c_void_p, C.c_int, C.c_int, C.c_void_p, C.c_void_p]
        lib.sid_get_hessian.argtypes = [C.c_void_p, C.c_void_p, C.c_int, C.c_int, C.c_uint, C.c_void_p]
        lib.sid_deformation.argtypes = [C.c_void_p, C.c_int] + [C.c_void_p] * 4 + [C.c_int] + [C.c_void_p] * 7
        lib.sid_get_peaks.argtypes = [C.c_void_p, C.c_int64, C.c_void_p]
        lib.sid_get_uncertainty.argtypes = [C.c_void_p, C.c_int64, C.c_void_p]
        lib.sid_filter_outliers.argtypes = [C.c_void_p, C.c_int, C.c_int, C.c_int64] + [C.c_void_p] * 5 + \
            [C.c_double, C.c_double, C.c_void_p, C.c_void_p]
        _lib = lib
        return lib


def as_u8_image(a):
    """uint8 2-D array with unit column stride (rows may be pitched); copies only if needed."""
    a = np.asarray(a)
    if a.ndim != 2:
        raise ValueError("image must be 2-D")
    if a.dtype != np.uint8 or a.strides[1] != 1 or a.strides[0] < a.shape[1]:
        a = np.ascontiguousarray(a, dtype=np.uint8)
    return a


def angle_table(angles, alpha0, img_size):
    """Per-angle rotation table the C ABI expects, evaluated with NumPy exactly the
    way the reference's get_template does (reference pmlib.py:105-110):
    cos a, sin a and [tc, tc] . [[cos a, -sin a], [sin a, cos a]]."""
    tc = int(img_size / 2.) + 1
    centre = np.array([tc, tc])
    tab = np.empty((len(angles), 4), dtype=np.float64)
    for k, angle in enumerate(angles):
        a = np.radians(angle - alpha0)
        rot = np.array([[np.cos(a), -np.sin(a)], [np.sin(a), np.cos(a)]])
        shift = centre.dot(rot)
        tab[k] = (rot[0, 0], rot[1, 0], shift[0], shift[1])
    return tab


def pair_layout(rows, cols):
    """(pitch, bytes) of a resident image of ``rows x cols`` in the library's layout (sid_pair_layout)."""
    pitch, nbytes = C.c_int64(), C.c_int64()
    rc = load_library().sid_pair_layout(int(rows), int(cols), C.byref(pitch), C.byref(nbytes))
    if rc:
        raise ValueError("sid_pair_layout(%r, %r) failed" % (rows, cols))
    return int(pitch.value), int(nbytes.value)


def flags_from_kwargs(hes_norm=True, hes_smth=False, mcc_norm=False, subpixel=False, masked=False, uncertainty=False):
    if uncertainty and not subpixel:
        raise ValueError("uncertainty=True needs subpixel=True: it is the covariance of the sub-pixel offsets")
    return (SID_HES_NORM if hes_norm else 0) | (SID_HES_SMTH if hes_smth else 0) | (SID_MCC_NORM if mcc_norm else 0) | \
        (SID_SUBPIXEL if subpixel else 0) | (SID_MASKED if masked else 0) | (SID_UNCERT if uncertainty else 0)


def flags_from_options(kwargs):
    """The sid_run* flags of a kwargs dict of the drop-in API: ``hes_norm`` (default True), ``hes_smth``, ``mcc_norm``
    and the extensions ``subpixel``, ``masked`` and ``uncertainty`` (default False), so every entry point maps its
    keyword arguments the same way.  ``uncertainty`` without ``subpixel`` raises ValueError."""
    return flags_from_kwargs(kwargs.get('hes_norm', True), kwargs.get('hes_smth', False), kwargs.get('mcc_norm', False),
                             kwargs.get('subpixel', False), kwargs.get('masked', False),
                             kwargs.get('uncertainty', False))


class Context(object):
    """One sid_ctx: one CUDA device, one stream, one resident image pair."""

    def __init__(self, device=0):
        self._lib = load_library()
        self._h = C.c_void_p()
        rc = self._lib.sid_create(C.byref(self._h), int(device))
        if rc:
            raise SidError("sid_create(device=%d) failed with code %d: no usable CUDA device "
                           "(this package has no CPU fallback)" % (device, rc))
        self.device = int(device)
        self._pair_key = None

    def close(self):
        if self._h:
            self._lib.sid_destroy(self._h)
            self._h = C.c_void_p()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def _check(self, rc):
        if rc:
            msg = self._lib.sid_last_error(self._h).decode("utf-8", "replace")
            if rc in (-1, -4):
                raise ValueError("sid_b200: %s (code %d)" % (msg, rc))
            raise SidError("sid_b200: %s (code %d)" % (msg, rc))

    @property
    def handle(self):
        return self._h

    @property
    def launch_count(self):
        return int(self._lib.sid_launch_count(self._h))

    @property
    def last_kernel_ms(self):
        return float(self._lib.sid_last_kernel_ms(self._h))

    @property
    def last_kernel_name(self):
        return self._lib.sid_last_kernel_name(self._h).decode()

    def set_stream(self, cuda_stream):
        """None -> the context's own stream; 0 -> CUDA's legacy default stream (what
        torch.cuda.current_stream().cuda_stream is unless a side stream is active);
        anything else -> that cudaStream_t."""
        if cuda_stream is None:
            handle = 0
        elif int(cuda_stream) == 0:
            handle = 1                      # cudaStreamLegacy
        else:
            handle = int(cuda_stream)
        self._check(self._lib.sid_set_stream(self._h, C.c_void_p(handle)))

    def synchronize(self):
        self._check(self._lib.sid_synchronize(self._h))

    def set_pair(self, img1, img2):
        img1, img2 = as_u8_image(img1), as_u8_image(img2)
        self._check(self._lib.sid_set_pair(
            self._h, img1.ctypes.data, img1.shape[0], img1.shape[1], img1.strides[0],
            img2.ctypes.data, img2.shape[0], img2.shape[1], img2.strides[0]))
        self._pair_key = None
        return self

    def set_pair_device(self, ptr1, shape1, pitch1, ptr2, shape2, pitch2):
        self._check(self._lib.sid_set_pair_device(
            self._h, C.c_void_p(ptr1), shape1[0], shape1[1], pitch1, C.c_void_p(ptr2), shape2[0], shape2[1], pitch2))
        self._pair_key = None
        return self

    def adopt_pair_device(self, ptr1, shape1, pitch1, bytes1, ptr2, shape2, pitch2, bytes2):
        """Use caller-owned device buffers (layout of :func:`pair_layout`) as the resident pair, no copy."""
        self._check(self._lib.sid_adopt_pair_device(
            self._h, C.c_void_p(ptr1), shape1[0], shape1[1], pitch1, bytes1,
            C.c_void_p(ptr2), shape2[0], shape2[1], pitch2, bytes2))
        self._pair_key = None
        return self

    def downsample_pair(self, factor, buf1, buf2):
        """k x k box downsampling (k = ``factor``) of the resident pair into caller-owned device buffers
        (sid_downsample_pair), asynchronous on the context's stream.  ``buf1`` / ``buf2`` are ``(device pointer, pitch,
        bytes)`` in the layout of ``pair_layout(rows // factor, cols // factor)`` of image 1 / 2."""
        (p1, pitch1, bytes1), (p2, pitch2, bytes2) = buf1, buf2
        self._check(self._lib.sid_downsample_pair(self._h, int(factor), C.c_void_p(int(p1)), int(pitch1), int(bytes1),
                                                  C.c_void_p(int(p2)), int(pitch2), int(bytes2)))
        return self

    def pm_epilogue_affine(self, gpi, c2pm1, r2pm1, xy, ll, results=None):
        """pattern_matching's post-processing for affine geolocation on the device (sid_pm_epilogue_affine): returns
        the seven flat grids u, v, a, r, h, lon2, lat2 (NaN outside ``gpi``).  ``results`` None: use the table the
        previous run left on the device."""
        gpi = np.asarray(gpi, dtype=bool).ravel()
        idx = np.ascontiguousarray(np.flatnonzero(gpi), dtype=np.int32)
        c = np.ascontiguousarray(c2pm1, dtype=np.float64).ravel()
        r = np.ascontiguousarray(r2pm1, dtype=np.float64).ravel()
        xy = np.ascontiguousarray(xy, dtype=np.float64).reshape(6)
        ll = np.ascontiguousarray(ll, dtype=np.float64).reshape(6)
        res = None if results is None else np.ascontiguousarray(results, dtype=np.float64).reshape(-1, 5)
        out = np.empty((7, gpi.size), dtype=np.float64)
        self._check(self._lib.sid_pm_epilogue_affine(
            self._h, idx.size, idx.ctypes.data, gpi.size, c.ctypes.data, r.ctypes.data,
            None if res is None else res.ctypes.data, xy.ctypes.data, ll.ctypes.data, out.ctypes.data))
        return out

    def peaks(self, n):
        """The SID_PEAKS records of the previous run (sid_get_peaks): an (n, SID_N_PEAKS, 4) float64 array of c2, r2,
        r, h per secondary peak, rank order, NaN where missing."""
        out = np.empty((int(n), SID_N_PEAKS, 4), dtype=np.float64)
        self._check(self._lib.sid_get_peaks(self._h, int(n), out.ctypes.data))
        return out

    def uncertainty(self, n):
        """The SID_UNCERT records of the previous run (sid_get_uncertainty): an (n, 3) float64 array of var_c, var_r,
        cov_cr, the covariance of every row's sub-pixel offsets in image-2 pixels^2, NaN where undefined."""
        out = np.empty((int(n), 3), dtype=np.float64)
        self._check(self._lib.sid_get_uncertainty(self._h, int(n), out.ctypes.data))
        return out

    def filter_outliers(self, grid_shape, gpi, c2pm1, r2pm1, results=None, peaks=None, eps=1.0, threshold=2.0,
                        in_place=False):
        """Normalised median test with secondary-peak replacement (sid_filter_outliers) on a ``grid_shape`` (rows,
        cols) grid whose valid points are ``gpi`` (flat or grid-shaped, table order = row-major order of the True
        positions).  ``results`` / ``peaks`` None: the table and peaks the previous run left on the device.  Returns
        ``(table, flags)``; with ``in_place`` (device-resident inputs only) the device table is updated and ``table`` is
        None."""
        rows, cols = (int(v) for v in grid_shape)
        gpi = np.asarray(gpi, dtype=bool).ravel()
        if gpi.size != rows * cols:
            raise ValueError("gpi must have grid_shape's number of elements")
        idx = np.ascontiguousarray(np.flatnonzero(gpi), dtype=np.int32)
        c = np.ascontiguousarray(c2pm1, dtype=np.float64).ravel()
        r = np.ascontiguousarray(r2pm1, dtype=np.float64).ravel()
        if c.size != gpi.size or r.size != gpi.size:
            raise ValueError("c2pm1 / r2pm1 must have one value per grid point")
        if (results is None) != (peaks is None):
            raise ValueError("pass both results and peaks, or neither")
        res = pk = None
        if results is not None:
            res = np.ascontiguousarray(results, dtype=np.float64).reshape(-1, 5)
            pk = np.ascontiguousarray(peaks, dtype=np.float64).reshape(-1, SID_N_PEAKS, 4)
            if res.shape[0] != idx.size or pk.shape[0] != idx.size:
                raise ValueError("results / peaks need one row per valid grid point")
        out = None if in_place else np.empty((idx.size, 5), dtype=np.float64)
        flags = np.empty(idx.size, dtype=np.int32)
        self._check(self._lib.sid_filter_outliers(
            self._h, rows, cols, idx.size, idx.ctypes.data, c.ctypes.data, r.ctypes.data,
            None if res is None else res.ctypes.data, None if pk is None else pk.ctypes.data, float(eps),
            float(threshold), None if out is None else out.ctypes.data, flags.ctypes.data))
        return out, flags

    def first_guess(self, sx, sy, vx, vy, kx, ky, qx, qy):
        """Delaunay-linear interpolation of (vx, vy) from the sources (sx, sy) onto (qx, qy) and the distance of every
        query point to the nearest (kx, ky) point (sid_first_guess).  Returns (vx_q, vy_q, dist, flag)."""
        f64 = lambda a: np.ascontiguousarray(np.asarray(a, dtype=np.float64).ravel())
        sx, sy, vx, vy, kx, ky, qx, qy = map(f64, (sx, sy, vx, vy, kx, ky, qx, qy))
        if not (sx.size == sy.size == vx.size == vy.size) or kx.size != ky.size or qx.size != qy.size:
            raise ValueError("coordinate / value arrays must have matching lengths")
        ovx, ovy, od = (np.empty(qx.size, dtype=np.float64) for _ in range(3))
        flag = np.zeros(qx.size, dtype=np.int32)
        self._check(self._lib.sid_first_guess(
            self._h, sx.size, sx.ctypes.data, sy.ctypes.data, vx.ctypes.data, vy.ctypes.data, kx.size, kx.ctypes.data,
            ky.ctypes.data, qx.size, qx.ctypes.data, qy.ctypes.data, ovx.ctypes.data, ovy.ctypes.data, od.ctypes.data,
            flag.ctypes.data))
        return ovx, ovy, od, flag

    def upload_rows(self, dst_ptr, dst_pitch, rows_array):
        """Asynchronous 2-D upload of image rows (uint8, unit column stride) to ``dst_ptr`` on the context's stream."""
        a = as_u8_image(rows_array) if rows_array.shape[0] else rows_array
        if a.shape[0]:
            self._check(self._lib.sid_upload_rows(self._h, C.c_void_p(dst_ptr), dst_pitch, a.ctypes.data, a.strides[0],
                                                  a.shape[1], a.shape[0]))
        return a.shape[0] * a.shape[1]

    def run(self, c1, r1, c2fg, r2fg, border, img_size, angles, alpha0, rot_order=0, flags=SID_HES_NORM,
            mtype=SID_TM_CCOEFF_NORMED, want_status=False, keep_on_device=False):
        arrs = [np.ascontiguousarray(np.atleast_1d(x), dtype=np.float64) for x in (c1, r1, c2fg, r2fg, border)]
        n = arrs[0].size
        if any(a.size != n for a in arrs):
            raise ValueError("point arrays must have equal length")
        ang = np.ascontiguousarray(np.asarray(angles, dtype=np.float64))
        tab = angle_table(angles, alpha0, img_size)
        out = np.full((n, 5), np.nan, dtype=np.float64)
        status = np.zeros(n, dtype=np.int32)
        self._check(self._lib.sid_run(
            self._h, n, *[a.ctypes.data for a in arrs], int(img_size), len(ang), ang.ctypes.data,
            tab.ctypes.data, int(rot_order), int(flags), int(mtype), None if keep_on_device else out.ctypes.data,
            status.ctypes.data))
        if keep_on_device:
            return status if want_status else None
        return (out, status) if want_status else out

    def run_maps(self, c1, r1, c2fg, r2fg, border, img_size, angles, alpha0, rot_order=0, flags=SID_HES_NORM,
                 mtype=SID_TM_CCOEFF_NORMED, want_status=False):
        """:meth:`run` on the resident pair that also returns every valid row's winning NCC map and template
        (``rotate_and_match(...)[5]`` / ``[6]``, sid_run_maps): ``(table, maps, templates[, status])``.  ``maps`` is a
        list of N float32 2-D views into one contiguous buffer (point order), None where the row is neither valid nor
        masked (SID_MASKED); ``templates`` an (N, img_size, img_size) uint8 array, 0 where the row is neither."""
        arrs = [np.ascontiguousarray(np.atleast_1d(x), dtype=np.float64) for x in (c1, r1, c2fg, r2fg, border)]
        n = arrs[0].size
        if any(a.size != n for a in arrs):
            raise ValueError("point arrays must have equal length")
        ang = np.ascontiguousarray(np.asarray(angles, dtype=np.float64))
        tab = angle_table(angles, alpha0, img_size)
        shape = np.zeros((n, 2), dtype=np.int32)
        total = C.c_int64(0)
        self._check(self._lib.sid_map_layout(self._h, n, *[a.ctypes.data for a in arrs], int(img_size),
                                             shape.ctypes.data, C.byref(total)))
        buf = np.empty(total.value, dtype=np.float32)
        templates = np.zeros((n, int(img_size), int(img_size)), dtype=np.uint8)
        out = np.full((n, 5), np.nan, dtype=np.float64)
        status = np.zeros(n, dtype=np.int32)
        self._check(self._lib.sid_run_maps(
            self._h, n, *[a.ctypes.data for a in arrs], int(img_size), len(ang), ang.ctypes.data,
            tab.ctypes.data, int(rot_order), int(flags), int(mtype), out.ctypes.data, status.ctypes.data,
            buf.size, buf.ctypes.data, templates.ctypes.data))
        ends = np.cumsum(shape[:, 0].astype(np.int64) * shape[:, 1])
        maps = [buf[e - h * w:e].reshape(h, w) if st in (SID_PT_VALID, SID_PT_MASKED) else None
                for (h, w), e, st in zip(shape.tolist(), ends.tolist(), status.tolist())]
        return (out, maps, templates, status) if want_status else (out, maps, templates)

    def run_pair(self, img1, img2, c1, r1, c2fg, r2fg, border, img_size, angles, alpha0, rot_order=0,
                 flags=SID_HES_NORM, mtype=SID_TM_CCOEFF_NORMED, want_status=False, keep_on_device=False):
        """Upload the pair and match all points in one call, copy overlapped with compute."""
        img1, img2 = as_u8_image(img1), as_u8_image(img2)
        arrs = [np.ascontiguousarray(np.atleast_1d(x), dtype=np.float64) for x in (c1, r1, c2fg, r2fg, border)]
        n = arrs[0].size
        if any(a.size != n for a in arrs):
            raise ValueError("point arrays must have equal length")
        ang = np.ascontiguousarray(np.asarray(angles, dtype=np.float64))
        tab = angle_table(angles, alpha0, img_size)
        out = np.full((n, 5), np.nan, dtype=np.float64)
        status = np.zeros(n, dtype=np.int32)
        self._check(self._lib.sid_run_pair(
            self._h, img1.ctypes.data, img1.shape[0], img1.shape[1], img1.strides[0],
            img2.ctypes.data, img2.shape[0], img2.shape[1], img2.strides[0],
            n, *[a.ctypes.data for a in arrs], int(img_size), len(ang), ang.ctypes.data,
            tab.ctypes.data, int(rot_order), int(flags), int(mtype), None if keep_on_device else out.ctypes.data,
            status.ctypes.data))
        self._pair_key = None
        if keep_on_device:
            return status if want_status else None
        return (out, status) if want_status else out

    def run_device(self, n, d_c1, d_r1, d_c2fg, d_r2fg, d_border, max_border, img_size, angles, alpha0,
                   d_out, d_status=0, rot_order=0, flags=SID_HES_NORM, mtype=SID_TM_CCOEFF_NORMED):
        ang = np.ascontiguousarray(np.asarray(angles, dtype=np.float64))
        tab = angle_table(angles, alpha0, img_size)
        self._check(self._lib.sid_run_device(
            self._h, int(n), C.c_void_p(d_c1), C.c_void_p(d_r1), C.c_void_p(d_c2fg), C.c_void_p(d_r2fg),
            C.c_void_p(d_border), int(max_border), int(img_size), len(ang), ang.ctypes.data, tab.ctypes.data,
            int(rot_order), int(flags), int(mtype), C.c_void_p(d_out), C.c_void_p(d_status)))

    def rotate_and_match(self, img1, c1, r1, img_size, image2, angles, alpha0, rot_order=0,
                         flags=SID_HES_NORM, mtype=SID_TM_CCOEFF_NORMED):
        img1, image2 = as_u8_image(img1), as_u8_image(image2)
        tab = angle_table(angles, alpha0, img_size)
        H, W = image2.shape
        if H < img_size or W < img_size:
            raise ValueError("search window smaller than the template")
        res = np.zeros((max(H - img_size + 1, 1), max(W - img_size + 1, 1)), np.float32)
        tpl = np.zeros((img_size, img_size), np.uint8)
        valid, ba = C.c_int(0), C.c_int(-1)
        dc, dr = C.c_double(0), C.c_double(0)
        br, bh = C.c_float(0), C.c_float(0)
        self._check(self._lib.sid_rotate_and_match(
            self._h, img1.ctypes.data, img1.shape[0], img1.shape[1], img1.strides[0], float(c1), float(r1),
            int(img_size), image2.ctypes.data, H, W, image2.strides[0], len(angles), tab.ctypes.data,
            int(rot_order), int(flags), int(mtype), C.byref(valid), C.byref(dc), C.byref(dr), C.byref(ba),
            C.byref(br), C.byref(bh), res.ctypes.data, tpl.ctypes.data))
        self._pair_key = None
        if not valid.value:
            return None
        return dc.value, dr.value, ba.value, np.float32(br.value), np.float32(bh.value), res, tpl

    def get_template(self, img, c, r, a, s, rot_order=0):
        img = as_u8_image(img)
        tab = angle_table([a], 0.0, s)
        out = np.zeros((s, s), np.uint8)
        self._check(self._lib.sid_get_template(self._h, img.ctypes.data, img.shape[0], img.shape[1], img.strides[0],
                                               float(c), float(r), tab.ctypes.data, int(s), int(rot_order),
                                               out.ctypes.data))
        self._pair_key = None
        return out

    def match_template(self, image, templ, method=SID_TM_CCOEFF_NORMED):
        image, templ = as_u8_image(image), as_u8_image(templ)
        H, W = image.shape
        th, tw = templ.shape
        if H < th or W < tw:
            raise ValueError("image smaller than template")
        out = np.zeros((H - th + 1, W - tw + 1), np.float32)
        self._check(self._lib.sid_match_template(self._h, image.ctypes.data, H, W, image.strides[0],
                                                 templ.ctypes.data, th, tw, templ.strides[0], int(method),
                                                 out.ctypes.data))
        self._pair_key = None
        return out

    def knn_hamming2(self, d1, d2):
        """Two nearest train descriptors per query (Hamming): (idx, dist) int32 arrays of shape (n1, 2)."""
        d1 = np.ascontiguousarray(d1, dtype=np.uint8)
        d2 = np.ascontiguousarray(d2, dtype=np.uint8)
        if d1.ndim != 2 or d2.ndim != 2 or d1.shape[1] != d2.shape[1]:
            raise ValueError("descriptors must be 2-D uint8 arrays with equal row length")
        idx = np.full((d1.shape[0], 2), -1, np.int32)
        dist = np.full((d1.shape[0], 2), -1, np.int32)
        self._check(self._lib.sid_knn_hamming2(self._h, d1.ctypes.data, d1.shape[0], d2.ctypes.data, d2.shape[0],
                                               d1.shape[1], idx.ctypes.data, dist.ctypes.data))
        return idx, dist

    def deformation(self, x, y, u, v, tri, area=None):
        """(e1, e2, e3, area, perimeter) of the m elements ``tri`` (m x 3 node indices) from node values."""
        x, y, u, v = [np.ascontiguousarray(np.ravel(k), dtype=np.float64) for k in (x, y, u, v)]
        n = x.size
        if any(k.size != n for k in (y, u, v)):
            raise ValueError("node arrays must have equal length")
        tri = np.ascontiguousarray(tri, dtype=np.int32)
        if tri.ndim != 2 or tri.shape[1] != 3:
            raise ValueError("triangulation must be an (m, 3) index array")
        m = tri.shape[0]
        ain = None
        if area is not None:
            ain = np.ascontiguousarray(np.ravel(area), dtype=np.float64)
            if ain.size != m:
                raise ValueError("one area per element expected")
        outs = [np.full(m, np.nan) for _ in range(5)]
        self._check(self._lib.sid_deformation(self._h, n, x.ctypes.data, y.ctypes.data, u.ctypes.data, v.ctypes.data,
                                              m, tri.ctypes.data, ain.ctypes.data if ain is not None else None,
                                              *[o.ctypes.data for o in outs]))
        return tuple(outs)

    def get_hessian(self, ccm, flags=SID_HES_NORM):
        ccm = np.ascontiguousarray(ccm, dtype=np.float32)
        if ccm.ndim != 2:
            raise ValueError("ccm must be 2-D")
        out = np.zeros_like(ccm)
        self._check(self._lib.sid_get_hessian(self._h, ccm.ctypes.data, ccm.shape[0], ccm.shape[1], int(flags),
                                              out.ctypes.data))
        return out


_default = {}


def default_context(device=None):
    """Process-wide context per device (created lazily, so nothing touches CUDA
    before a fork; device defaults to LOCAL_RANK or 0)."""
    if device is None:
        device = int(os.environ.get("SID_DEVICE", os.environ.get("LOCAL_RANK", "0")))
    key = (os.getpid(), int(device))
    ctx = _default.get(key)
    if ctx is None:
        ctx = Context(device)
        _default[key] = ctx
    return ctx
