"""ctypes binding of oracle/libcamcal_oracle.so.  TEST INFRASTRUCTURE ONLY.

Importable from tests/, __graft_entry__.smoke() and bench.py's cpu_baseline /
``--impl reference`` legs -- nowhere else (the product package never imports this).
"""
from __future__ import annotations

import ctypes as C
import os
import subprocess

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
_SO = os.path.join(_HERE, "libcamcal_oracle.so")

PER_VIEW = 66
SHARED = 21


class Intr(C.Structure):
    _fields_ = [(n, C.c_double) for n in ("frow", "fcol", "crow", "ccol", "k", "checker_size")]


class View(C.Structure):
    _fields_ = [("rvec", C.c_double * 3), ("tvec", C.c_double * 3)]


class ChainS(C.Structure):
    _fields_ = [("R", C.c_double * 9), ("t", C.c_double * 3), ("Rinv", C.c_double * 9),
                ("tinv", C.c_double * 3)] + [(n, C.c_double) for n in (
                    "a_row", "b_row", "a_col", "b_col", "frow", "fcol", "crow", "ccol", "k",
                    "inv_cs", "cs_back")]


def build(force: bool = False) -> str:
    src = os.path.join(_HERE, "camcal_oracle.c")
    if force or not os.path.exists(_SO) or os.path.getmtime(_SO) < os.path.getmtime(src):
        if os.path.exists(src):
            subprocess.check_call(["make", "-C", _HERE, "-s"])
    return _SO


_lib = None


def lib():
    global _lib
    if _lib is None:
        if not os.path.exists(_SO):
            build()
        L = C.CDLL(_SO)
        dp = C.POINTER(C.c_double)
        L.cco_cubic_root.restype = C.c_double
        L.cco_cubic_root.argtypes = [C.c_double]
        L.cco_get_ratio.restype = C.c_double
        L.cco_get_ratio.argtypes = [dp, dp, C.c_int, C.c_int, C.c_double]
        _lib = L
    return _lib


def _dp(a):
    return a.ctypes.data_as(C.POINTER(C.c_double))


def _f64(a):
    return np.ascontiguousarray(a, dtype=np.float64)


def make_intr(intr) -> Intr:
    return Intr(*[float(x) for x in intr])


def make_view(rvec, tvec) -> View:
    v = View()
    v.rvec[:] = [float(x) for x in rvec]
    v.tvec[:] = [float(x) for x in tvec]
    return v


def make_views(views):
    arr = (View * len(views))()
    for i, (rv, tv) in enumerate(views):
        arr[i].rvec[:] = [float(x) for x in rv]
        arr[i].tvec[:] = [float(x) for x in tv]
    return arr


def chain(intr, rvec, tvec) -> ChainS:
    ch = ChainS()
    i, v = make_intr(intr), make_view(rvec, tvec)
    lib().cco_chain_build(C.byref(i), C.byref(v), C.byref(ch))
    return ch


def cubic_root(c: float) -> float:
    return lib().cco_cubic_root(float(c))


def world2img(ch, xyz, nthreads=0):
    xyz = _f64(xyz).reshape(-1, 3)
    x, y, z = [np.ascontiguousarray(xyz[:, i]) for i in range(3)]
    n = len(x)
    row, col = np.empty(n), np.empty(n)
    lib().cco_world2img_batch(C.byref(ch), _dp(x), _dp(y), _dp(z), _dp(row), _dp(col),
                              C.c_size_t(n), C.c_int(nthreads))
    return row, col


def world2img_soa(ch, x, y, z=None, nthreads=0):
    x, y = _f64(x), _f64(y)
    n = len(x)
    row, col = np.empty(n), np.empty(n)
    zp = _dp(_f64(z)) if z is not None else None
    lib().cco_world2img_batch(C.byref(ch), _dp(x), _dp(y), zp, _dp(row), _dp(col),
                              C.c_size_t(n), C.c_int(nthreads))
    return row, col


def img2world_soa(ch, row, col, want_z=True, nthreads=0):
    row, col = _f64(row), _f64(col)
    n = len(row)
    x, y = np.empty(n), np.empty(n)
    z = np.empty(n) if want_z else None
    lib().cco_img2world_batch(C.byref(ch), _dp(row), _dp(col), _dp(x), _dp(y),
                              _dp(z) if want_z else None, C.c_size_t(n), C.c_int(nthreads))
    return x, y, z


def get_ratio(imgpoints, checker_size):
    """imgpoints: (n1, n2, 2) with [a, b] = corner (a, b)."""
    ip = np.asarray(imgpoints, dtype=np.float64)
    n1, n2 = ip.shape[:2]
    rows = np.ascontiguousarray(ip[:, :, 0].T).ravel()  # a fastest
    cols = np.ascontiguousarray(ip[:, :, 1].T).ravel()
    return lib().cco_get_ratio(_dp(rows), _dp(cols), n1, n2, float(checker_size))


def get_axes(ratio, checker_size, n_corners, sz):
    out = (C.c_longlong * 2)()
    lib().cco_get_axes(C.c_double(ratio), C.c_double(checker_size), int(n_corners[0]),
                       int(n_corners[1]), int(sz[0]), int(sz[1]), out)
    return int(out[0]), int(out[1])


def _axs(axs_min):
    return (C.c_longlong * 2)(int(axs_min[0]), int(axs_min[1]))


def rectify_map(ch, inv_ratio, axs_min, sz, nthreads=0):
    """returns (map_row, map_col) arrays of shape (sz2, sz1) = memory order (r contiguous)."""
    sz1, sz2 = sz
    mr, mc = np.empty((sz2, sz1)), np.empty((sz2, sz1))
    lib().cco_rectify_map(C.byref(ch), C.c_double(inv_ratio), _axs(axs_min), _dp(mr), _dp(mc),
                          sz1, sz2, C.c_size_t(sz1), C.c_int(nthreads))
    return mr, mc


def rectify_f32c1(ch, inv_ratio, axs_min, src, fill=np.nan, nthreads=0):
    """src: float32 (nframes, sz2, sz1) C-order == Julia (sz1, sz2) frames, r contiguous."""
    src = np.ascontiguousarray(src, dtype=np.float32)
    nf, sz2, sz1 = src.shape
    dst = np.empty_like(src)
    lib().cco_rectify_f32c1(C.byref(ch), C.c_double(inv_ratio), _axs(axs_min),
                            src.ctypes.data_as(C.POINTER(C.c_float)),
                            dst.ctypes.data_as(C.POINTER(C.c_float)), sz1, sz2,
                            C.c_size_t(sz1), C.c_size_t(sz1 * sz2), nf, C.c_float(fill),
                            C.c_int(nthreads))
    return dst


def rectify_u8c3(ch, inv_ratio, axs_min, src, fill=(0, 0, 0), nthreads=0):
    """src: uint8 (nframes, sz2, sz1, 3) C-order."""
    src = np.ascontiguousarray(src, dtype=np.uint8)
    nf, sz2, sz1, _ = src.shape
    dst = np.empty_like(src)
    f = (C.c_uint8 * 3)(*[int(v) for v in fill])
    lib().cco_rectify_u8c3(C.byref(ch), C.c_double(inv_ratio), _axs(axs_min),
                           src.ctypes.data_as(C.POINTER(C.c_uint8)),
                           dst.ctypes.data_as(C.POINTER(C.c_uint8)), sz1, sz2,
                           C.c_size_t(sz1), C.c_size_t(sz1 * sz2), nf, f, C.c_int(nthreads))
    return dst


def reproj_jtj(intr, aspect, views, obj, img, want_jac=False, nthreads=0):
    """views: list of (rvec, tvec); obj (nc,3); img (nv,nc,2)."""
    obj, img = _f64(obj), _f64(img)
    nv, nc = img.shape[0], img.shape[1]
    pv = np.empty((nv, PER_VIEW))
    sh = np.empty(SHARED)
    jac = np.empty((nv, nc, 2, 10)) if want_jac else None
    i = make_intr(intr)
    va = make_views(views) if not isinstance(views, C.Array) else views
    lib().cco_reproj_jtj(C.byref(i), C.c_double(aspect), va, nv, _dp(obj), _dp(img), nc,
                         _dp(pv), _dp(sh), _dp(jac) if want_jac else None, C.c_int(nthreads))
    return pv, sh, jac


def calculate_errors(intr, views, obj, imgs, n_corners, inv_samples, raw_sums=False):
    """the reference's four errors; raw_sums: the four sums over all views they normalise"""
    obj, imgs, inv_samples = _f64(obj), _f64(imgs), _f64(inv_samples)
    nv, S = inv_samples.shape[0], inv_samples.shape[1]
    ir = np.ascontiguousarray(inv_samples[:, :, 0])
    ic = np.ascontiguousarray(inv_samples[:, :, 1])
    out = (C.c_double * 4)()
    i = make_intr(intr)
    fn = lib().cco_calculate_error_sums if raw_sums else lib().cco_calculate_errors
    fn(C.byref(i), make_views(views), nv, _dp(obj), _dp(imgs), int(n_corners[0]), int(n_corners[1]),
       _dp(ir), _dp(ic), S, out)
    return tuple(out)
