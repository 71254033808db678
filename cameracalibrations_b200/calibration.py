"""Host-side mirror of the reference's calibration object (src/meta.jl, src/io.jl,
src/buildcalibrations.jl, src/plot_calibration.jl) over the C ABI of libcamcal_b200.

Same names and argument meaning as the Julia package; differences forced by the host
language are listed in INTEGRATION.md:
  * view indices are 0-based here (Julia: 1-based);
  * `c(points, idx)` takes a BATCH: an (n, 2) array is RowCol -> returns (n, 3) XYZ, an
    (n, 3) array is XYZ -> returns (n, 2) RowCol (Julia dispatches on SVector{2}/{3} and
    is applied by broadcast, src/buildcalibrations.jl:29,46).  The points stay interleaved, as
    the reference keeps them: the cc_*_aos entry points read and write that layout directly;
  * numpy arrays take the `*_host` entry points (chunked H2D -> kernel -> D2H), CUDA
    torch tensors take the device entry points on torch's current stream.
Every numeric result comes from the CUDA kernels; there is no Python/numpy fallback.
"""
from __future__ import annotations

import ctypes as C
import functools
import json
import math
import re
from typing import Sequence

import numpy as np

from . import _lib
from ._lib import lib, check

try:  # torch is plumbing only: device memory + streams
    import torch
except Exception:  # pragma: no cover
    torch = None


def _is_torch(x) -> bool:
    return torch is not None and isinstance(x, torch.Tensor)


def _stream_ptr(device_index: int):
    return C.c_void_p(torch.cuda.current_stream(device_index).cuda_stream)


def _np_ptr(a: np.ndarray):
    return C.c_void_p(a.ctypes.data)


def _t_ptr(t):
    return C.c_void_p(t.data_ptr())


def _device(t) -> int:
    """The device of a CUDA tensor."""
    return t.device.index if t.device.index is not None else torch.cuda.current_device()


def _where(x):
    """(context, pointer of an array, entry point suffix, stream argument) of a call on x: a CUDA tensor runs on
    its own device, on torch's current stream there; a numpy array takes the `_host` entry point on the default
    device."""
    if _is_torch(x):
        dev = _device(x)
        return _lib.context(dev), _t_ptr, "", (_stream_ptr(dev),)
    return _lib.context(_default_device()), _np_ptr, "_host", ()


def _check_points(t) -> None:
    if not t.is_cuda:
        raise TypeError("torch inputs must be CUDA tensors (numpy arrays take the host path)")
    if t.dtype not in (torch.float32, torch.float64):
        raise TypeError("float32 or float64 points only")


def _points(pts):
    """Interleaved points as the point maps take them: a tensor as it is, anything else as a numpy array that
    stays float32 or becomes float64."""
    if _is_torch(pts):
        return pts
    pts = np.asarray(pts)
    return pts if pts.dtype in (np.float32, np.float64) else pts.astype(np.float64)


class Calibration:
    """`Calibration` of src/meta.jl:17-33: intrinsic (frow, fcol, crow, ccol), one
    extrinsic (rotation vector, translation) per image, scale = 1/checker_size, the
    radial coefficient k and the file names."""

    def __init__(self, intrinsic, extrinsics, scale, k, files: Sequence[str]):
        frow, fcol, crow, ccol = [float(v) for v in intrinsic]
        self.intrinsic = (frow, fcol, crow, ccol)
        self.extrinsics = [(tuple(float(v) for v in r), tuple(float(v) for v in t)) for r, t in extrinsics]
        self.scale = float(scale)              # diag of LinearMap(I/checker_size)
        self.k = float(k)
        self.files = list(files)
        self._intr = _lib.make_intr(frow, fcol, crow, ccol, self.k, 1.0 / self.scale)
        self._views = [_lib.make_view(r, t) for r, t in self.extrinsics]
        self._view_rows = np.array([r + t for r, t in self.extrinsics], dtype=np.float64).reshape(-1, 6)

    # -- construction from fit results: obj2img, src/buildcalibrations.jl:1-6
    @classmethod
    def from_fit(cls, Rs, ts, frow, fcol, crow, ccol, checker_size, k, files):
        return cls((frow, fcol, crow, ccol), list(zip(Rs, ts)), 1.0 / checker_size, k, files)

    @property
    def checker_size(self) -> float:
        return 1.0 / self.scale

    def _index(self, extrinsic) -> int:
        if extrinsic is None:      # src/meta.jl:90-93: first file whose name contains "extrinsic"
            for i, f in enumerate(self.files):
                if re.search("extrinsic", f):
                    return i
            raise IndexError("no file name contains 'extrinsic'")
        if isinstance(extrinsic, str):
            return self.files.index(extrinsic)
        i = int(extrinsic)
        if not 0 <= i < len(self._views):
            raise IndexError(f"extrinsic index {i} out of range 0:{len(self._views)}")  # BoundsError
        return i

    # -- SoA entry points ---------------------------------------------------------
    def img2world(self, row, col, extrinsic=None, want_z: bool = True):
        """(c::Calibration)(i::RowCol, idx), src/meta.jl:82; want_z=False is
        rectification(c, idx), src/meta.jl:99."""
        vi = self._index(extrinsic)
        return _point_call("img2world", self, vi, (row, col), 3 if want_z else 2)

    def world2img(self, x, y, z=None, extrinsic=None):
        """(c::Calibration)(xyz::XYZ, idx), src/meta.jl:88; z=None means z = 0."""
        vi = self._index(extrinsic)
        ins = (x, y) if z is None else (x, y, z)
        return _point_call("world2img", self, vi, ins, 2)

    # -- points of many views in one call: c.(pts_v, v) over views v ----------------
    def img2world_views(self, row, col, extrinsics, counts, want_z: bool = True):
        """Pixel -> world for consecutive segments of points with their own views: points
        [sum(counts[:s]), sum(counts[:s+1])) use extrinsics[s] (view indices or file names, as
        warp_views takes them).  One call (one launch for CUDA tensors); every point's result is
        bit-identical to img2world with its segment's view."""
        return _point_call("img2world", self, self._segments(extrinsics, counts), (row, col), 3 if want_z else 2)

    def world2img_views(self, x, y, z, extrinsics, counts):
        """World -> pixel over segments of views, as img2world_views; z=None means z = 0."""
        ins = (x, y) if z is None else (x, y, z)
        return _point_call("world2img", self, self._segments(extrinsics, counts), ins, 2)

    def _segments(self, extrinsics, counts):
        """(views, nviews, offsets) of cc_*_views as numpy arrays: cc_view rows [rvec | tvec] and size_t
        offsets.  Built without a Python loop when the extrinsics are integers (10 000 views are common)."""
        vis = np.asarray(extrinsics)
        if vis.dtype.kind not in "iu":                    # file names or None: one at a time
            vis = np.asarray([self._index(e) for e in extrinsics], dtype=np.int64)
        elif vis.size and (vis.min() < 0 or vis.max() >= len(self._views)):
            bad = int(vis[(vis < 0) | (vis >= len(self._views))][0])
            raise IndexError(f"extrinsic index {bad} out of range 0:{len(self._views)}")  # BoundsError
        counts = np.asarray(counts, dtype=np.int64).reshape(-1)
        if vis.ndim != 1 or len(vis) != len(counts) or not len(vis):
            raise ValueError("need one count per extrinsic, and at least one")
        if counts.min() < 0:
            raise ValueError("counts must be non-negative")
        offsets = np.zeros(len(counts) + 1, dtype=np.uint64)
        np.cumsum(counts, out=offsets[1:], dtype=np.uint64)
        return np.ascontiguousarray(self._view_rows[vis]), len(vis), offsets

    # -- the reference's callable: dispatch on RowCol (.., 2) vs XYZ (.., 3) -------
    def __call__(self, pts, extrinsic=None):
        if isinstance(extrinsic, (list, tuple)):
            return self._call_views(pts, extrinsic)
        pts = _points(pts)
        if pts.shape[-1] == 2:
            return _aos_call("img2world", self, self._index(extrinsic), pts, 3)
        if pts.shape[-1] == 3:
            return _aos_call("world2img", self, self._index(extrinsic), pts, 2)
        raise TypeError("points must be RowCol (.., 2) or XYZ (.., 3)")

    def _call_views(self, pts, extrinsics):
        """c(list of (n_i, 2 | 3) arrays, list of extrinsics): one call over all of them, the list of
        per-view results back (slices of one output)."""
        if len(pts) != len(extrinsics):
            raise ValueError("need one point array per extrinsic")
        is_t = bool(pts) and _is_torch(pts[0])
        if is_t:
            pts = [p.reshape(-1, p.shape[-1]) for p in pts]
        else:
            pts = [np.asarray(p) for p in pts]
            dt = np.float32 if pts and all(p.dtype == np.float32 for p in pts) else np.float64
            pts = [p.astype(dt, copy=False).reshape(-1, p.shape[-1]) for p in pts]
        dims = {p.shape[-1] for p in pts}
        if len(dims) != 1 or not dims <= {2, 3}:
            raise TypeError("points must all be RowCol (n, 2) or all XYZ (n, 3)")
        d = dims.pop()
        counts = [int(p.shape[0]) for p in pts]
        segs = self._segments(extrinsics, counts)
        cat = torch.cat(pts) if is_t else np.concatenate(pts)
        out = _aos_call("img2world" if d == 2 else "world2img", self, segs, cat, 5 - d)
        bounds = np.cumsum([0] + counts)
        return [out[int(a):int(b)] for a, b in zip(bounds[:-1], bounds[1:])]


def rectification(c: Calibration, extrinsic=None):
    """rectification(c, idx) = pop o image2real[idx], src/meta.jl:99-103."""
    vi = c._index(extrinsic)

    def f(rc):
        rc = _points(rc)
        if rc.shape[-1] != 2:                  # (row, col) are the first two coordinates
            rc = rc[..., :2]
            if rc.shape[-1] != 2:
                raise IndexError("points need a row and a column coordinate")
        return _aos_call("img2world", c, vi, rc, 2)

    return f


def _aos_call(kind, c: Calibration, vi, pts, out_dim: int):
    """One cc_{kind}_{f64|f32}_aos[_host] call on interleaved points pts (..., 2 | 3); returns (..., out_dim)
    in pts' dtype.  vi: a view index, or the (views, nviews, offsets) of Calibration._segments.  A
    C-contiguous input is passed as is; any other is copied once."""
    segs = isinstance(vi, tuple)
    views = (_np_ptr(vi[0]), vi[1], _np_ptr(vi[2])) if segs else (C.byref(c._views[vi]), 1, None)
    lead, in_dim = tuple(pts.shape[:-1]), int(pts.shape[-1])
    if _is_torch(pts):
        _check_points(pts)
        pts = pts.contiguous()
        out = torch.empty(lead + (out_dim,), dtype=pts.dtype, device=pts.device)
    else:
        pts = np.ascontiguousarray(pts, dtype=np.float32 if pts.dtype == np.float32 else np.float64)
        out = np.empty(lead + (out_dim,), dtype=pts.dtype)
    ctx, ptr, host, tail = _where(pts)
    n = math.prod(lead)
    _check_total(vi, n, segs)
    fn = getattr(lib, f"cc_{kind}_{'f32' if pts.itemsize == 4 else 'f64'}_aos{host}")
    io = (ptr(pts), ptr(out), out_dim) if kind == "img2world" else (ptr(pts), in_dim, ptr(out))
    check(fn(ctx.handle, C.byref(c._intr), *views, *io, C.c_size_t(n), *tail))
    return out


def _point_call(kind, c: Calibration, vi, ins, nout: int):
    """kind: img2world (ins=row,col; outs x,y[,z]) or world2img (ins=x,y[,z]; outs row,col).
    vi: a view index, or the (views, nviews, offsets) of Calibration._segments for cc_*_views."""
    segs = isinstance(vi, tuple)     # the views form takes its point count from the offsets
    views = (_np_ptr(vi[0]), vi[1], _np_ptr(vi[2])) if segs else (C.byref(c._views[vi]),)
    first = ins[0]
    if _is_torch(first):
        _check_points(first)
        ins = [t.contiguous() for t in ins]
        n = ins[0].numel()
        if any(t.dtype != first.dtype or t.numel() != n or t.device != first.device for t in ins):
            raise ValueError("coordinate arrays must share dtype, length and device")
        outs = [torch.empty(n, dtype=first.dtype, device=first.device) for _ in range(nout)]
    else:
        dt = np.float32 if np.asarray(first).dtype == np.float32 else np.float64
        ins = [np.ascontiguousarray(a, dtype=dt).reshape(-1) for a in ins]
        n = ins[0].size
        if any(a.size != n for a in ins):
            raise ValueError("coordinate arrays must have the same length")
        outs = [np.empty(n, dtype=dt) for _ in range(nout)]
    ctx, ptr, host, tail = _where(ins[0])
    _check_total(vi, n, segs)
    fn = getattr(lib, f"cc_{kind}_{'f32' if ins[0].itemsize == 4 else 'f64'}{'_views' if segs else ''}{host}")

    def slots(arrs, k):              # a missing z is a NULL pointer
        return [ptr(a) for a in arrs] + [None] * (k - len(arrs))
    io = slots(ins, 2) + slots(outs, 3) if kind == "img2world" else slots(ins, 3) + slots(outs, 2)
    check(fn(ctx.handle, C.byref(c._intr), *views, *io, *(() if segs else (C.c_size_t(n),)), *tail))
    return tuple(outs)


def _check_total(vi, n: int, segs: bool) -> None:
    """The library takes the point count from the offsets: they must cover the arrays exactly."""
    if segs and int(vi[2][-1]) != n:
        raise ValueError(f"counts sum to {int(vi[2][-1])}, the point arrays hold {n}")


def _default_device() -> int:
    if torch is not None and torch.cuda.is_available():
        return torch.cuda.current_device()
    return 0


# ---------------------------------------------------------------------------------
# rectification of frames: src/plot_calibration.jl
# ---------------------------------------------------------------------------------
def get_ratio(imgpoints, checker_size, n_corners=None) -> float:
    """src/plot_calibration.jl:8-13.  imgpoints: (n1, n2, 2) array, [a, b] = corner (a, b); or,
    with n_corners = (n1, n2), the flat (n1*n2, 2) layout detect_fit returns (corner a fastest,
    the memory of the reference's n1 x n2 Julia matrix)."""
    ip = np.asarray(imgpoints, dtype=np.float64)
    if ip.ndim == 2:
        if n_corners is None:
            raise ValueError("flat (n1*n2, 2) image points need n_corners=(n1, n2)")
        n1, n2 = int(n_corners[0]), int(n_corners[1])
        if ip.shape != (n1 * n2, 2):
            raise ValueError(f"expected {n1 * n2} corners, got array of shape {ip.shape}")
        ip = ip.reshape(n2, n1, 2).transpose(1, 0, 2)
    n1, n2 = ip.shape[:2]
    rows = np.ascontiguousarray(ip[:, :, 0].T).ravel()
    cols = np.ascontiguousarray(ip[:, :, 1].T).ravel()
    out = C.c_double()
    check(lib.cc_get_ratio(_np_ptr(rows), _np_ptr(cols), n1, n2, float(checker_size), C.byref(out)))
    return float(out.value)


def get_axes(ratio, checker_size, n_corners, sz):
    """src/plot_calibration.jl:1-6 -> (min of first axis, min of second axis); each axis has
    the input's length."""
    out = (C.c_int64 * 2)()
    check(lib.cc_get_axes(float(ratio), float(checker_size), int(n_corners[0]), int(n_corners[1]),
                          int(sz[0]), int(sz[1]), out))
    return int(out[0]), int(out[1])


def image_transformations(c: Calibration, extrinsic_index, imgpointss, checker_size, n_corners, sz):
    """src/plot_calibration.jl:15-22: (ratio, axs_min) that drive `warp`."""
    vi = c._index(extrinsic_index)
    ratio = get_ratio(imgpointss[vi], checker_size, n_corners)   # (n1, n2, 2) or detect_fit's flat layout
    return ratio, get_axes(ratio, checker_size, n_corners, sz)


def _frames(frames, fill, coord: str, gather: str, out, single: bool):
    """What warp and warp_views share: the frames as the library reads them, C-contiguous (a numpy array that is
    not uint8 becomes float32), whether they are uint8 RGB, the output buffer, the fill value and the flags.
    single: a frame without the leading axis is a batch of one, and the last value returned says so."""
    flags = {"f64": _lib.COORD_F64, "f32": _lib.COORD_F32}[coord] | {
        "auto": _lib.GATHER_AUTO, "direct": _lib.GATHER_DIRECT, "tma": _lib.GATHER_TMA}[gather]
    if _is_torch(frames):
        if not frames.is_cuda:
            raise TypeError("torch frames must be CUDA tensors (numpy arrays take the host path)")
        u8 = frames.dtype == torch.uint8
        frames = frames.contiguous()
    else:
        u8 = np.asarray(frames).dtype == np.uint8
        frames = np.ascontiguousarray(frames, dtype=np.uint8 if u8 else np.float32)
    one = single and frames.ndim == (3 if u8 else 2)
    if one:
        frames = frames.reshape((1,) + tuple(frames.shape))
    if frames.ndim != (4 if u8 else 3) or (u8 and frames.shape[-1] != 3):
        raise ValueError("frames must be (nframes, sz2, sz1) float32 or (nframes, sz2, sz1, 3) uint8")
    if out is None:
        out = torch.empty_like(frames) if _is_torch(frames) else np.empty_like(frames)
    if u8:
        fv = (C.c_uint8 * 3)(*([0, 0, 0] if fill is None else [int(v) for v in fill]))
    else:
        fv = C.c_float(float("nan") if fill is None else float(fill))
    return frames, u8, out, fv, flags, one


def warp(c: Calibration, extrinsic, frames, ratio: float, axs_min, fill=None, coord: str = "f64",
         gather: str = "auto", out=None):
    """warp(img, tform, axs), src/plot_calibration.jl:40, for a batch of frames of one view.

    frames: float32 (nframes, sz2, sz1) or uint8 (nframes, sz2, sz1, 3), C-contiguous -- i.e.
    the memory of Julia arrays of size (sz1, sz2) (first RowCol axis contiguous).  A single
    frame may omit the leading axis.  numpy -> host pipeline; CUDA torch tensor -> device.
    fill defaults to the reference's: NaN for float frames, black for RGB{N0f8}.
    coord: "f64" (reference precision, bit-exact index/weight selection) | "f32" (fast path).
    """
    vi = c._index(extrinsic)
    frames, u8, out, fv, flags, one = _frames(frames, fill, coord, gather, out, single=True)
    nframes, sz2, sz1 = int(frames.shape[0]), int(frames.shape[1]), int(frames.shape[2])
    axs = (C.c_int64 * 2)(int(axs_min[0]), int(axs_min[1]))
    ctx, ptr, host, tail = _where(frames)
    fn = getattr(lib, f"cc_rectify_{'u8c3' if u8 else 'f32c1'}{host}")
    check(fn(ctx.handle, C.byref(c._intr), C.byref(c._views[vi]), float(ratio), axs, ptr(frames), ptr(out),
             sz1, sz2, C.c_size_t(sz1), C.c_size_t(sz1 * sz2), nframes, fv, flags, *tail))
    return out[0] if one else out


def warp_views(c: Calibration, extrinsics, frames, ratios, axs_mins, fill=None, coord: str = "f64",
               gather: str = "auto", out=None):
    """Rectify frames that belong to DIFFERENT views in one call -- the loop of the reference's plot
    (src/plot_calibration.jl:36-42: every calibration image with its own extrinsic, ratio, axes).

    extrinsics: view indices / file names, one per group; frames: (nviews * k, sz2, sz1) float32 or
    (nviews * k, sz2, sz1, 3) uint8 -- frames [v*k, (v+1)*k) belong to extrinsics[v]; ratios[v], axs_mins[v]
    as returned by image_transformations for that view.  A CUDA tensor is rectified on its stream; a numpy
    array takes the host pipeline over all views in one call (cc_rectify_views_*_host) and returns numpy."""
    vis = [c._index(e) for e in extrinsics]
    nv = len(vis)
    frames, u8, out, fv, flags, _ = _frames(frames, fill, coord, gather, out, single=False)
    if nv == 0 or frames.shape[0] % nv:
        raise ValueError("frames must be (nviews * k, sz2, sz1) float32 or (nviews * k, sz2, sz1, 3) uint8")
    k, sz2, sz1 = int(frames.shape[0]) // nv, int(frames.shape[1]), int(frames.shape[2])
    views = (_lib.View * nv)(*[c._views[i] for i in vis])
    rat = (C.c_double * nv)(*[float(r) for r in ratios])
    axs = (C.c_int64 * (2 * nv))(*[int(a) for am in axs_mins for a in am])
    ctx, ptr, host, tail = _where(frames)
    kern = "u8c3" if u8 else "f32c1"
    fn = getattr(lib, f"cc_rectify_views_{kern}_host" if host else f"cc_rectify_{kern}_views")
    check(fn(ctx.handle, C.byref(c._intr), views, nv, rat, axs, ptr(frames), ptr(out), sz1, sz2, C.c_size_t(sz1),
             C.c_size_t(sz1 * sz2), k, fv, flags, *tail))
    return out


def jpeg_info(data: bytes):
    """(sz1, sz2, channels) = (rows, columns, components) of a JPEG stream; header parse only."""
    buf = (C.c_uint8 * len(data)).from_buffer_copy(data)
    a, b, ch = C.c_int(), C.c_int(), C.c_int()
    check(lib.cc_jpeg_info(buf, C.c_size_t(len(data)), C.byref(a), C.byref(b), C.byref(ch)))
    return a.value, b.value, ch.value


def load_jpegs(datas, device=None, out=None):
    """Device-side `RGB.(FileIO.load(file))` for a list of JPEG files (src/plot_calibration.jl:37):
    the compressed bytes go to the GPU, the decoded frames never come back.  datas: list of bytes
    objects (or file names), all the same size.  Returns a CUDA uint8 tensor (n, sz2, sz1, 3) -- the
    u8c3 frame layout that warp() / warp_views() take."""
    blobs = []
    for d in datas:
        if isinstance(d, str):                       # a file name
            with open(d, "rb") as f:
                d = f.read()
        blobs.append(bytes(d))
    if not blobs:
        raise ValueError("no images")
    sz1, sz2, _ = jpeg_info(blobs[0])
    dev = _default_device() if device is None else int(device)
    if out is None:
        out = torch.empty((len(blobs), sz2, sz1, 3), dtype=torch.uint8, device=f"cuda:{dev}")
    bufs = [(C.c_uint8 * len(b)).from_buffer_copy(b) for b in blobs]
    ptrs = (C.c_void_p * len(bufs))(*[C.addressof(b) for b in bufs])
    lens = (C.c_size_t * len(bufs))(*[len(b) for b in blobs])
    check(lib.cc_jpeg_decode_u8c3(_lib.context(dev).handle, ptrs, lens, len(bufs), _t_ptr(out), sz1, sz2,
                                  C.c_size_t(sz1), C.c_size_t(sz1 * sz2), _stream_ptr(dev)))
    torch.cuda.current_stream(dev).synchronize()      # the compressed host buffers die with this frame
    return out


def rectify_map(c: Calibration, extrinsic, ratio: float, axs_min, sz, device=None, coord: str = "f64"):
    """Source (row, col) sampled by every output pixel as two (sz2, sz1) CUDA tensors: FP64 (the
    reference's map) or, coord="f32", the FP32 map of the fast path."""
    vi = c._index(extrinsic)
    dev = _default_device() if device is None else int(device)
    ctx = _lib.context(dev)
    sz1, sz2 = int(sz[0]), int(sz[1])
    mr = torch.empty((sz2, sz1), dtype=torch.float64 if coord == "f64" else torch.float32, device=f"cuda:{dev}")
    mc = torch.empty_like(mr)
    axs = (C.c_int64 * 2)(int(axs_min[0]), int(axs_min[1]))
    fn = lib.cc_rectify_map_f64 if coord == "f64" else lib.cc_rectify_map_f32
    check(fn(ctx.handle, C.byref(c._intr), C.byref(c._views[vi]), float(ratio), axs,
                                 _t_ptr(mr), _t_ptr(mc), sz1, sz2, C.c_size_t(sz1), _stream_ptr(dev)))
    return mr, mc


# ---------------------------------------------------------------------------------
# residual / Jacobian / errors: src/buildcalibrations.jl:28-67
# ---------------------------------------------------------------------------------
def views_tensor(extrinsics, device):
    """(nviews, 6) float64 CUDA tensor with the cc_view layout [rvec | tvec]."""
    a = np.asarray([list(r) + list(t) for r, t in extrinsics], dtype=np.float64).reshape(-1, 6)
    return torch.from_numpy(a).to(device)


def _dist_world(group=None) -> int:
    d = torch.distributed if torch is not None else None
    return d.get_world_size(group) if d is not None and d.is_available() and d.is_initialized() else 1


def allreduce_shared(t, group=None):
    """The exchange step of the path: in-place sum of a small float64 CUDA tensor over the ranks,
    through cc_allreduce_shared (raw NCCL inside libcamcal_b200, csrc/comm.cu).  torch.distributed
    is only the bootstrap that carries the NCCL unique id to the other ranks, once per context."""
    if _dist_world(group) > 1:
        ctx = _lib.context(_device(t))
        ctx.comm_init_from_torch(group)
        ctx.allreduce(t)
    return t


def reproj_jtj(intr, aspect, views, obj, img, group=None):
    """Residual sum, Jacobian and normal-equation blocks of this rank's views.

    intr: (frow, fcol, crow, ccol, k, checker_size); views: (nviews, 6) [rvec|tvec];
    obj: (ncorners, 3); img: (nviews, ncorners, 2).  numpy -> host entry point; CUDA torch
    tensors -> device entry point.  Returns (per_view (nviews, 66), shared (21,)).
    With torch.distributed initialised (or `group` given) the shared block is all-reduced
    (NCCL sum through cc_allreduce_shared) so every rank holds the global J'J_ii, J'r_i and sum r^2.
    """
    ci = _lib.make_intr(*[float(v) for v in intr])
    on_device = _is_torch(img)
    if on_device:
        views, obj, img = (t.contiguous().to(torch.float64) for t in (views, obj, img))
        new = functools.partial(torch.empty, dtype=torch.float64, device=img.device)
    else:
        views = np.ascontiguousarray(views, dtype=np.float64).reshape(-1, 6)
        obj, img = (np.ascontiguousarray(a, dtype=np.float64) for a in (obj, img))
        new = np.empty
    nv, nc = int(img.shape[0]), int(img.shape[1])
    pv, sh = new((nv, _lib.PER_VIEW)), new(_lib.SHARED)
    ctx, ptr, host, tail = _where(img)
    fn = getattr(lib, f"cc_reproj_jtj_f64{host}")
    check(fn(ctx.handle, C.byref(ci), float(aspect), ptr(views), nv, ptr(obj), ptr(img), nc, ptr(pv), ptr(sh), *tail))
    if on_device:
        allreduce_shared(sh, group)
    return pv, sh


def calculate_errors(c: Calibration, imgpointss, objpoints, checker_size, sz, files, n_corners,
                     inverse_samples: int = 100, rng=None, group=None):
    """calculate_errors, src/buildcalibrations.jl:37-67, fused on the device.

    imgpointss: (nviews, n1*n2, 2) with corner a fastest; objpoints: (n1*n2, 3) already
    multiplied by checker_size (src/buildcalibrations.jl:15).  Returns the reference's
    NamedTuple as a dict: n, reprojection, projection, distance, inverse.
    """
    rng = np.random.default_rng() if rng is None else rng
    nv = len(c.extrinsics)
    n1, n2 = int(n_corners[0]), int(n_corners[1])
    samples = rng.random((nv, max(1, inverse_samples), 2)) * (np.asarray(sz, dtype=np.float64) - 1) + 1
    dev = _default_device()
    device = f"cuda:{dev}"
    views = views_tensor(c.extrinsics, device)
    obj = torch.as_tensor(np.ascontiguousarray(objpoints, dtype=np.float64)).reshape(-1, 3).to(device)
    img = torch.as_tensor(np.ascontiguousarray(imgpointss, dtype=np.float64)).reshape(nv, -1, 2).to(device)
    ir = torch.from_numpy(np.ascontiguousarray(samples[:, :, 0])).to(device)
    ic = torch.from_numpy(np.ascontiguousarray(samples[:, :, 1])).to(device)
    sums = torch.empty(4, dtype=torch.float64, device=device)
    check(lib.cc_calculate_errors_f64(_lib.context(dev).handle, C.byref(c._intr), _t_ptr(views), nv,
                                      _t_ptr(obj), _t_ptr(img), n1, n2, _t_ptr(ir), _t_ptr(ic),
                                      int(inverse_samples), _t_ptr(sums), _stream_ptr(dev)))
    n_files = nv
    if _dist_world(group) > 1:                      # one all-reduce: the four sums and the view count
        both = torch.cat([sums, torch.tensor([float(nv)], dtype=torch.float64, device=device)])
        allreduce_shared(both, group)
        sums, n_files = both[:4], int(round(float(both[4].item())))
    s = sums.cpu().numpy()
    n = n1 * n2 * n_files
    return dict(n=n_files,
                reprojection=math.sqrt(s[0] / n),
                projection=math.sqrt(s[1] / n),
                distance=math.sqrt(s[2] / ((n1 - 1) * (n2 - 1)) / n_files),
                inverse=math.sqrt(s[3] / max(1, inverse_samples) / n_files))


# ---------------------------------------------------------------------------------
# JSON save / load: src/io.jl:9-32 (CalibrationIO field names and nesting)
# ---------------------------------------------------------------------------------
def save(file, c: Calibration) -> None:
    frow, fcol, crow, ccol = c.intrinsic
    doc = {
        "intrinsic": {"linear": [frow, fcol], "translation": [crow, ccol]},
        "extrinsics": [{"linear": {"sx": r[0], "sy": r[1], "sz": r[2]}, "translation": list(t)}
                       for r, t in c.extrinsics],
        "scale": {"linear": [c.scale] * 3},
        "k": c.k,
        "files": c.files,
    }
    with open(file, "w") as f:
        json.dump(doc, f)


def _rvec_from_json(lin):
    if isinstance(lin, dict):
        return (lin["sx"], lin["sy"], lin["sz"])
    a = np.asarray(lin, dtype=np.float64)
    if a.size == 3:
        return tuple(a.ravel())
    if a.size == 9:  # a rotation matrix (column-major, as JSON3 writes AbstractMatrix): log map
        R = a.reshape(3, 3).T
        th = math.acos(max(-1.0, min(1.0, (np.trace(R) - 1) / 2)))
        if th < 1e-12:
            return (0.0, 0.0, 0.0)
        w = np.array([R[2, 1] - R[1, 2], R[0, 2] - R[2, 0], R[1, 0] - R[0, 1]]) / (2 * math.sin(th))
        return tuple(w * th)
    raise ValueError("unrecognised rotation encoding")


def load(file) -> Calibration:
    with open(file) as f:
        d = json.load(f)
    lin, tr = d["intrinsic"]["linear"], d["intrinsic"]["translation"]
    ext = [(_rvec_from_json(e["linear"]), tuple(e["translation"])) for e in d["extrinsics"]]
    return Calibration((lin[0], lin[1], tr[0], tr[1]), ext, d["scale"]["linear"][0], d["k"], d["files"])
