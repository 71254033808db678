"""Levenberg-Marquardt fit of the camera model on the device (SURVEY 8f rank 2).

The reference fits by calling OpenCV.calibrateCamera (src/detect_fit.jl:47) with
CALIB_ZERO_TANGENT_DIST + FIX_K2 + FIX_K3 + FIX_ASPECT_RATIO (+ FIX_K1 when
with_distortion == false) (:40) and CRITERIA = (EPS + MAX_ITER, 30, 1e-3)
(src/CameraCalibrations.jl:16).  Here the same model is fitted by an LM loop whose every
numerical step runs in hand-written kernels:

    cc_reproj_jtj_f64   residuals, analytic Jacobian, normal-equation blocks  (csrc/residual.cu)
    cc_lm_schur_f64     per-view 6x6 Cholesky + Schur complement on (f, crow, ccol, k)
    cc_lm_update_f64    4x4 solve, back-substitution, candidate parameters     (csrc/lm.cu)

The host only compares two scalars per iteration (accept / reject, stopping rule) and, when
views are sharded over ranks, all-reduces 21 + 21 + 2 doubles (NCCL).  Starting values follow
OpenCV's calibrateCamera: principal point at the image centre, focal length from the
homographies' vanishing-point constraints (cvInitIntrinsicParams2D), extrinsics from the
homography decomposition.
"""
from __future__ import annotations

import ctypes as C

import numpy as np

from . import _lib
from ._lib import check, lib
from .calibration import _device, _t_ptr, _stream_ptr, reproj_jtj, allreduce_shared, torch

FREE_ALL = 0b1111
FREE_NO_K = 0b0111          # CALIB_FIX_K1


# ------------------------------------------------------------------ starting values (host, tiny)
def _homographies(xy, rcs):
    """DLT with Hartley normalisation, all views at once: (x, y, 1) -> (row, col, 1).
    xy (n, 2) board corners, rcs (nv, n, 2) detections.  The 9x9 normal matrices are
    eigen-decomposed in one batched call (starting values only: the LM refines them)."""
    def norm(p):                                   # p (..., n, 2) -> normalised points, T (..., 3, 3)
        m = p.mean(-2, keepdims=True)
        s = np.sqrt(2.0) / np.maximum(np.sqrt(((p - m) ** 2).sum(-1)).mean(-1), 1e-300)
        T = np.zeros(p.shape[:-2] + (3, 3))
        T[..., 0, 0] = T[..., 1, 1] = s
        T[..., 0, 2], T[..., 1, 2] = -s * m[..., 0, 0], -s * m[..., 0, 1]
        T[..., 2, 2] = 1.0
        return (p - m) * s[..., None, None], T
    a, Ta = norm(np.asarray(xy, float))
    b, Tb = norm(np.asarray(rcs, float))
    nv, n = b.shape[0], b.shape[1]
    A = np.zeros((nv, 2 * n, 9))
    A[:, 0::2, 0:2], A[:, 0::2, 2] = a, 1.0
    A[:, 0::2, 6:8], A[:, 0::2, 8] = -b[:, :, :1] * a, -b[:, :, 0]
    A[:, 1::2, 3:5], A[:, 1::2, 5] = a, 1.0
    A[:, 1::2, 6:8], A[:, 1::2, 8] = -b[:, :, 1:] * a, -b[:, :, 1]
    _, vecs = np.linalg.eigh(np.einsum("vij,vik->vjk", A, A))
    h = vecs[:, :, 0].reshape(nv, 3, 3)            # eigenvector of the smallest eigenvalue
    H = np.linalg.inv(Tb) @ h @ Ta
    return H / H[:, 2:3, 2:3]


def _rodrigues_inv(R):
    U, _, Vt = np.linalg.svd(R)
    R = U @ Vt
    if np.linalg.det(R) < 0:
        R = U @ np.diag([1, 1, -1.0]) @ Vt
    th = np.arccos(np.clip((np.trace(R) - 1) / 2, -1, 1))
    w = np.array([R[2, 1] - R[1, 2], R[0, 2] - R[2, 0], R[1, 0] - R[0, 1]])
    if th < 1e-12:
        return 0.5 * w
    if np.pi - th < 1e-6:       # near pi: axis from the symmetric part
        B = (R + np.eye(3)) / 2
        ax = np.sqrt(np.maximum(np.diag(B), 0))
        i = int(np.argmax(ax))
        ax = B[i] / ax[i]
        return th * ax / np.linalg.norm(ax)
    return th * w / (2 * np.sin(th))


def initial_guess(obj, imgs, sz, aspect=1.0):
    """obj (nc, 3) in world units with z == 0; imgs (nv, nc, 2) (row, col); sz = (sz1, sz2).
    Returns (intr (frow, fcol, crow, ccol, k), views (nv, 6))."""
    obj, imgs = np.asarray(obj, float), np.asarray(imgs, float)
    c = np.array([(sz[0] - 1) / 2.0, (sz[1] - 1) / 2.0])
    Hs = _homographies(obj[:, :2], imgs)
    # cvInitIntrinsicParams2D: with the principal point removed, each homography gives two
    # linear equations in (1/frow^2, 1/fcol^2)
    A, b = [], []
    for H in Hs:
        Hc = H.copy()
        Hc[0] -= Hc[2] * c[0]
        Hc[1] -= Hc[2] * c[1]
        h, v = Hc[:, 0], Hc[:, 1]
        d1, d2 = (h + v) / 2, (h - v) / 2
        n = [1 / np.linalg.norm(x) for x in (h, v, d1, d2)]
        h, v, d1, d2 = h * n[0], v * n[1], d1 * n[2], d2 * n[3]
        A += [[h[0] * v[0], h[1] * v[1]], [d1[0] * d2[0], d1[1] * d2[1]]]
        b += [-h[2] * v[2], -d1[2] * d2[2]]
    f = np.linalg.lstsq(np.array(A), np.array(b), rcond=None)[0]
    fr, fc = np.sqrt(abs(1 / f[0])), np.sqrt(abs(1 / f[1]))
    if aspect:
        tf = (fr + fc) / (aspect + 1.0)
        fr, fc = aspect * tf, tf
    Kinv = np.linalg.inv(np.array([[fr, 0, c[0]], [0, fc, c[1]], [0, 0, 1.0]]))
    views = []
    for H in Hs:
        M = Kinv @ H
        lam = 2.0 / (np.linalg.norm(M[:, 0]) + np.linalg.norm(M[:, 1]))
        if M[2, 2] * lam < 0:
            lam = -lam                              # board in front of the camera
        r1, r2, t = M[:, 0] * lam, M[:, 1] * lam, M[:, 2] * lam
        views.append(np.concatenate([_rodrigues_inv(np.stack([r1, r2, np.cross(r1, r2)], 1)), t]))
    return (fr, fc, c[0], c[1], 0.0), np.array(views)


# ------------------------------------------------------------------ device steps
def lm_schur(per_view, lam):
    """phase 1 on this rank's views: returns (yz (nv, 30), schur (21,)) device tensors"""
    dev = _device(per_view)
    nv = int(per_view.shape[0])
    yz = torch.empty((max(nv, 1), _lib.LM_YZ), dtype=torch.float64, device=per_view.device)
    schur = torch.empty(_lib.LM_SCHUR, dtype=torch.float64, device=per_view.device)
    check(lib.cc_lm_schur_f64(_lib.context(dev).handle, _t_ptr(per_view), nv, float(lam), _t_ptr(yz),
                              _t_ptr(schur), _stream_ptr(dev)))
    return yz, schur


def lm_update(shared, schur, lam, free_mask, yz, views):
    """phase 2: returns (candidate views (nv, 6), delta (8,)) device tensors"""
    dev = _device(views)
    nv = int(views.shape[0])
    out = torch.empty_like(views)
    delta = torch.empty(_lib.LM_DELTA, dtype=torch.float64, device=views.device)
    check(lib.cc_lm_update_f64(_lib.context(dev).handle, _t_ptr(shared), _t_ptr(schur), float(lam),
                               int(free_mask), _t_ptr(yz), _t_ptr(views), nv, _t_ptr(out), _t_ptr(delta),
                               _stream_ptr(dev)))
    return out, delta


def _dist_on(group):
    return torch.distributed.is_available() and torch.distributed.is_initialized()


def lm_fit(intr0, views0, obj, imgs, checker_size=1.0, aspect=1.0, with_distortion=True, max_iter=30,
           eps=1e-3, device=None, group=None, history=None):
    """Minimise the reprojection error over (f, crow, ccol[, k]) and every view's (rvec, tvec).

    intr0: (frow, fcol, crow, ccol, k); views0: (nv, 6) THIS rank's views; obj (nc, 3) board
    corners (already in world units); imgs (nv, nc, 2) detected (row, col).  With
    torch.distributed initialised the views may be sharded over ranks: the shared blocks are
    all-reduced and every rank takes the same accept/reject decisions.
    Returns dict(intr=(frow, fcol, crow, ccol, k), views=(nv, 6) ndarray, rms, iterations, lam).
    max_iter / eps default to the reference's CRITERIA (30, 1e-3: relative parameter step)."""
    assert torch is not None and torch.cuda.is_available(), "lm_fit runs on the GPU: no CPU fallback"
    dev = torch.device("cuda", torch.cuda.current_device() if device is None else device)
    f64 = dict(dtype=torch.float64, device=dev)
    views = torch.as_tensor(np.asarray(views0, float).reshape(-1, 6), **f64).contiguous()
    obj_t = torch.as_tensor(np.asarray(obj, float), **f64).contiguous()
    img_t = torch.as_tensor(np.asarray(imgs, float), **f64).contiguous()
    nv, nc = int(img_t.shape[0]), int(obj_t.shape[0])
    img_t = img_t.reshape(max(nv, 0), nc, 2)
    n_res = torch.tensor([1.0 * nv * nc], **f64)        # cv2 reports sqrt(sum |r|^2 / number of points)
    dist = _dist_on(group)
    if dist:
        allreduce_shared(n_res, group)
    n_res = float(n_res.item())
    f, crow, ccol, k = float(intr0[1]), float(intr0[2]), float(intr0[3]), float(intr0[4])
    if not with_distortion:
        k = 0.0
    mask = FREE_ALL if with_distortion else FREE_NO_K

    def blocks(f, crow, ccol, k, v):
        return reproj_jtj((aspect * f, f, crow, ccol, k, checker_size), aspect, v, obj_t, img_t, group=group)

    pv, sh = blocks(f, crow, ccol, k, views)
    sse = float(sh[20].item())
    lam, it, accepted = 1e-3, 0, 0
    while it < max_iter:
        it += 1
        yz, schur = lm_schur(pv, lam)
        if dist:
            allreduce_shared(schur, group)
        cand, delta = lm_update(sh, schur, lam, mask, yz, views)
        if dist:
            norms = delta[4:6].clone()
            allreduce_shared(norms, group)
            delta[4:6] = norms
        d = delta.cpu().numpy()
        bad = float(schur[20].item()) > 0 or d[6] == 0.0 or not np.all(np.isfinite(d))
        if not bad:
            fc, crc, ccc, kc = f + d[0], crow + d[1], ccol + d[2], k + d[3]
            pv_c, sh_c = blocks(fc, crc, ccc, kc, cand)
            sse_c = float(sh_c[20].item())
            bad = not np.isfinite(sse_c) or sse_c >= sse
        if history is not None:
            history.append(dict(it=it, lam=lam, sse=sse, accepted=not bad))
        if bad:
            lam = min(lam * 10.0, 1e16)
            continue
        step = np.sqrt(d[4] + float(np.sum(d[:4] ** 2)))
        size = np.sqrt(d[5] + f * f + crow * crow + ccol * ccol + k * k)
        f, crow, ccol, k, views, pv, sh, sse = fc, crc, ccc, kc, cand, pv_c, sh_c, sse_c
        lam = max(lam / 10.0, 1e-16)
        accepted += 1
        if step < eps * size:
            break
    return dict(intr=(aspect * f, f, crow, ccol, k), views=views.cpu().numpy(), rms=float(np.sqrt(sse / n_res)),
                iterations=it, accepted=accepted, lam=lam, sse=sse)


def _f64(a, dev):
    """a as a C-contiguous float64 tensor on dev; a tensor already so is returned as it is."""
    if torch.is_tensor(a):
        return a.to(dtype=torch.float64, device=dev).contiguous()
    return torch.as_tensor(np.asarray(a, float), dtype=torch.float64, device=dev).contiguous()


def _fit_intr(intr0, aspect, with_distortion, checker_size):
    """The starting cc_intr of a whole fit: frow = aspect * fcol, and k = 0 without distortion."""
    return _lib.make_intr(aspect * intr0[1], intr0[1], intr0[2], intr0[3], intr0[4] if with_distortion else 0.0,
                          checker_size)


def _fit_result(ci, views, rms, its, **device):
    """The result dict of a whole fit from the cc_intr, rms and iteration count the library wrote."""
    return dict(intr=(ci.frow, ci.fcol, ci.crow, ci.ccol, ci.k), views=views, **device, rms=rms.value,
                iterations=its.value)


def lm_fit_device(intr0, views0, obj, imgs, checker_size=1.0, aspect=1.0, with_distortion=True, max_iter=30,
                  eps=1e-3, device=None, group=None):
    """cc_lm_fit_f64: the whole fit as ONE device-resident loop (csrc/lm.cu) over THIS rank's
    views; damping, accept/reject and the stopping rule live in device memory, an iteration costs
    two small NCCL all-reduces and no host synchronisation.  Same arguments and result as lm_fit;
    device tensors may be passed for views0 / obj / imgs.  views0 itself is never written: the fit
    runs on a copy, returned as views_device."""
    assert torch is not None and torch.cuda.is_available(), "lm_fit_device runs on the GPU: no CPU fallback"
    dev = torch.device("cuda", torch.cuda.current_device() if device is None else device)
    views = _f64(views0, dev).reshape(-1, 6)
    if views.data_ptr() == (views0.data_ptr() if torch.is_tensor(views0) else 0):
        views = views.clone()
    obj_t, img_t = _f64(obj, dev), _f64(imgs, dev)
    nv, nc = int(views.shape[0]), int(obj_t.shape[0])
    ctx = _lib.context(dev.index)
    if _dist_on(group):
        ctx.comm_init_from_torch(group)
    ci = _fit_intr(intr0, aspect, with_distortion, checker_size)
    rms, its = C.c_double(), C.c_int()
    check(lib.cc_lm_fit_f64(ctx.handle, C.byref(ci), float(aspect), FREE_ALL if with_distortion else FREE_NO_K,
                            _t_ptr(views), nv, _t_ptr(obj_t), _t_ptr(img_t), nc, int(max_iter), float(eps),
                            C.byref(rms), C.byref(its), _stream_ptr(dev.index)))
    return _fit_result(ci, views.cpu().numpy(), rms, its, views_device=views)


def initial_guess_device(obj, imgs, sz, aspect=1.0, device=None, group=None):
    """cc_lm_initial_guess_f64: the starting values of initial_guess computed on the device for this
    rank's views (batched DLT + pose kernels, csrc/init.cu).  Returns (intr 5-tuple, views (nv, 6)
    CUDA tensor)."""
    dev = torch.device("cuda", torch.cuda.current_device() if device is None else device)
    obj_t, img_t = _f64(obj, dev), _f64(imgs, dev)
    nc = int(obj_t.shape[0])
    img_t = img_t.reshape(-1, nc, 2)
    nv = int(img_t.shape[0])
    views = torch.empty((nv, 6), dtype=torch.float64, device=dev)
    ctx = _lib.context(dev.index)
    if _dist_on(group):
        ctx.comm_init_from_torch(group)
    ci = _lib.make_intr(1.0, 1.0, 0.0, 0.0, 0.0, 1.0)
    check(lib.cc_lm_initial_guess_f64(ctx.handle, _t_ptr(obj_t), _t_ptr(img_t), nv, nc, int(sz[0]), int(sz[1]),
                                      float(aspect), C.byref(ci), _t_ptr(views), _stream_ptr(dev.index)))
    return (ci.frow, ci.fcol, ci.crow, ci.ccol, ci.k), views


def lm_fit_host(intr0, views0, obj, imgs, checker_size=1.0, aspect=1.0, with_distortion=True, max_iter=30,
                eps=1e-3, device=0):
    """cc_lm_fit_f64_host: the same fit in ONE call of the C ABI (host arrays in and out; what the
    Julia shim calls instead of OpenCV.calibrateCamera).  Single device."""
    views = np.ascontiguousarray(np.asarray(views0, float).reshape(-1, 6))
    obj = np.ascontiguousarray(obj, dtype=np.float64)
    imgs = np.ascontiguousarray(imgs, dtype=np.float64)
    nv, nc = int(imgs.shape[0]), int(obj.shape[0])
    ci = _fit_intr(intr0, aspect, with_distortion, checker_size)
    rms, its = C.c_double(), C.c_int()
    vp = lambda a: a.ctypes.data_as(C.c_void_p)
    check(lib.cc_lm_fit_f64_host(_lib.context(device).handle, C.byref(ci), float(aspect),
                                 FREE_ALL if with_distortion else FREE_NO_K, vp(views), nv, vp(obj), vp(imgs), nc,
                                 int(max_iter), float(eps), C.byref(rms), C.byref(its)))
    return _fit_result(ci, views, rms, its)
