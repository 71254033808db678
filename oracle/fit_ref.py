"""An independent reference of the fit path: residual, Jacobian and normal-equation blocks.
TEST INFRASTRUCTURE ONLY.

It shares no arithmetic with oracle/camcal_oracle.c or csrc/residual.cu, whose Jacobians are
the same closed formula: here
  * R = I + a [r]x + b [r]x^2 with a = sin(theta)/theta and b = (1 - cos theta)/theta^2 =
    2 sin^2(theta/2)/theta^2 (Taylor series for |theta^2| < 1e-8), theta^2 = r.r without a
    conjugate, so the residual is analytic in every parameter;
  * the Jacobian is taken by complex step (one complex evaluation per parameter, step 1e-200):
    no difference of nearby numbers is formed, so every column is accurate to a few ulps at any
    rotation angle;
  * every block entry is summed with math.fsum.
The same residual code runs on mpmath numbers, which is how tests/test_fit_reference.py checks
the complex-step Jacobian itself.

Parameters of one view: p = (rvec[3], tvec[3], f, crow, ccol, k), frow = aspect * f, fcol = f,
the layout of the kernel's Jacobian columns.
"""
from __future__ import annotations

import math

import numpy as np

STEP = 1e-200
U = 2.0 ** -53
NPAR = 10
PER_VIEW = 66
SHARED = 21


class _Numpy:
    sin, cos, sqrt = np.sin, np.cos, np.sqrt

    @staticmethod
    def select(cond, x, y):
        return np.where(cond, x, y)

    @staticmethod
    def small(t2):
        return np.abs(t2) < 1e-8


class _Mp:
    def __init__(self, mp):
        self.sin, self.cos, self.sqrt = mp.sin, mp.cos, mp.sqrt

    @staticmethod
    def select(cond, x, y):
        return x if cond else y

    @staticmethod
    def small(t2):
        return abs(t2) < 1e-8


def rotation(r, m=_Numpy):
    """R (3 x 3 nested lists) of the rotation vector r = (r0, r1, r2): numbers or arrays."""
    t2 = r[0] * r[0] + r[1] * r[1] + r[2] * r[2]
    small = m.small(t2)
    ts = m.select(small, 1.0, t2)              # keeps the direct branch finite where it is not used
    th = m.sqrt(ts)
    hs = m.sin(th / 2)
    a = m.select(small, 1 - t2 / 6 * (1 - t2 / 20 * (1 - t2 / 42)), m.sin(th) / th)
    b = m.select(small, (1 - t2 / 12 * (1 - t2 / 30 * (1 - t2 / 56))) / 2, 2 * hs * hs / ts)
    K = [[0, -r[2], r[1]], [r[2], 0, -r[0]], [-r[1], r[0], 0]]
    K2 = [[sum(K[i][l] * K[l][j] for l in range(3)) for j in range(3)] for i in range(3)]
    return [[(1 if i == j else 0) + a * K[i][j] + b * K2[i][j] for j in range(3)] for i in range(3)]


def project(p, checker_size, aspect, X, m=_Numpy):
    """(row, col) of the world points X = (x, y, z) under the view / intrinsics p."""
    R = rotation(p[0:3], m)
    q = [X[j] / checker_size for j in range(3)]
    P = [R[i][0] * q[0] + R[i][1] * q[1] + R[i][2] * q[2] + p[3 + i] for i in range(3)]
    u, v = P[0] / P[2], P[1] / P[2]
    radial = 1 + p[9] * (u * u + v * v)
    return aspect * p[6] * radial * u + p[7], p[6] * radial * v + p[8]


def _params(views, intr):
    """(10, nv, 1) float array: per view rvec, tvec, then the shared (f, crow, ccol, k)."""
    views = np.asarray(views, dtype=np.float64).reshape(-1, 6)
    nv = views.shape[0]
    p = np.empty((NPAR, nv, 1))
    p[:6, :, 0] = views.T
    p[6:, :, 0] = np.asarray(intr, dtype=np.float64)[:, None]
    return p


def residual(views, intr, checker_size, aspect, obj, img):
    """(nv, nc, 2) predicted minus observed.  views (nv, 6); intr = (f, crow, ccol, k) with
    frow = aspect * f; obj (nc, 3); img (nv, nc, 2)."""
    obj, img = np.asarray(obj, np.float64), np.asarray(img, np.float64)
    row, col = project(_params(views, intr), checker_size, aspect, obj.T)
    return np.stack([row - img[..., 0], col - img[..., 1]], -1)


def jacobian(views, intr, checker_size, aspect, obj):
    """(nv, nc, 2, 10) Jacobian of the residual by complex step."""
    obj = np.asarray(obj, np.float64)
    p = _params(views, intr).astype(np.complex128)
    nv, nc = p.shape[1], obj.shape[0]
    J = np.empty((nv, nc, 2, NPAR))
    for j in range(NPAR):
        pc = p.copy()
        pc[j] += 1j * STEP
        row, col = project(pc, checker_size, aspect, obj.T)
        J[:, :, 0, j] = np.broadcast_to(row.imag, (nv, nc)) / STEP
        J[:, :, 1, j] = np.broadcast_to(col.imag, (nv, nc)) / STEP
    return J


# entry (a, b) of the per-view block and of the shared block, in the kernel's layout
_PV_PAIRS = [(a, b) for a in range(6) for b in range(6)] + [(a, 6 + b) for a in range(6) for b in range(4)] \
    + [(a, NPAR) for a in range(6)]
_SH_PAIRS = [(6 + a, 6 + b) for a in range(4) for b in range(4)] + [(6 + a, NPAR) for a in range(4)] \
    + [(NPAR, NPAR)]


def blocks(views, intr, checker_size, aspect, obj, img):
    """The normal-equation blocks of reproj_jtj and the error scale of every entry.

    Returns a dict:
      per_view (nv, 66): A (6 x 6 full) | B (6 x 4 row-major) | g (6), fsum over the view's corners
      shared (21,):      C (4 x 4 full) | g_i (4) | sum of squared residuals, fsum over all views
      E_pv, E_sh:        the same entries over |J_a| |J_b|, |J_a| |r| and r^2 (plain sums)
      T_pv, T_sh:        the part of a computed entry's error that comes from errors of J and r
                         themselves (see tolerance)
      m_pv, m_sh:        number of terms summed per entry
      J (nv, nc, 2, 10), r (nv, nc, 2)."""
    obj, img = np.asarray(obj, np.float64), np.asarray(img, np.float64)
    nv, nc = img.shape[0], img.shape[1]
    J = jacobian(views, intr, checker_size, aspect, obj)
    r = residual(views, intr, checker_size, aspect, obj, img)
    # columns 0..9: J, column 10: r; rows: (corner, row/col) of each view
    Z = np.concatenate([J, r[..., None]], -1).reshape(nv, 2 * nc, NPAR + 1)
    # error model of the inputs of the sums: a Jacobian column is right to ETA_J * (its largest
    # magnitude in the view) -- the normwise criterion the oracle meets -- and a residual to
    # ETA_R * (|frow u_d| + |crow| + |observed|), the magnitudes its last subtraction cancels
    pred = np.abs(r + img)
    rho = ETA_R * (pred + np.abs(img) + np.abs(np.asarray(intr)[[1, 2]])).reshape(nv, 2 * nc)
    absZ = np.abs(Z)
    M = absZ.max(1) * ETA_J                       # (nv, 11): error of each column, per view
    M[:, NPAR] = 0.0
    S = absZ.sum(1)                               # (nv, 11)
    Srho = np.einsum("vka,vk->va", absZ, rho)     # (nv, 11): sum |Z_a| rho

    def entry_err(a, b):                          # per view: error of sum Z_a Z_b from the inputs' errors
        ea = M[:, a] * S[:, b] + M[:, b] * S[:, a] + 2 * nc * M[:, a] * M[:, b]
        if b == NPAR:
            ea = ea + Srho[:, a] + (Srho[:, NPAR] if a == NPAR else 0.0)
        return ea

    pv = np.empty((nv, PER_VIEW))
    E_pv, T_pv = np.empty((nv, PER_VIEW)), np.empty((nv, PER_VIEW))
    for e, (a, b) in enumerate(_PV_PAIRS):
        prod = Z[:, :, a] * Z[:, :, b]
        pv[:, e] = [math.fsum(row) for row in prod]
        E_pv[:, e] = np.abs(prod).sum(1)
        T_pv[:, e] = entry_err(a, b)
    sh = np.empty(SHARED)
    E_sh, T_sh = np.empty(SHARED), np.empty(SHARED)
    for e, (a, b) in enumerate(_SH_PAIRS):
        prod = (Z[:, :, a] * Z[:, :, b]).ravel()
        sh[e] = math.fsum(prod)
        E_sh[e] = np.abs(prod).sum()
        T_sh[e] = entry_err(a, b).sum()
    return dict(per_view=pv, shared=sh, E_pv=E_pv, E_sh=E_sh, T_pv=T_pv, T_sh=T_sh, m_pv=2 * nc,
                m_sh=2 * nc * nv, J=J, r=r)


ETA_J = 32 * U
ETA_R = 8 * U


def gamma(m):
    """gamma_m = m u / (1 - m u): the relative bound of a sum of m rounded terms, in any order."""
    return m * U / (1 - m * U)


def tolerance(ref, which):
    """Entry-wise bound |computed - reference| for a block computed in float64 from the same data:
    gamma_m E (rounding of the products and the sum) + T (errors of J and r, carried into the sum
    by both sides).  which: "per_view" or "shared"."""
    if which == "per_view":
        return gamma(ref["m_pv"] + 1) * ref["E_pv"] + 2 * ref["T_pv"]
    return gamma(ref["m_sh"] + 1) * ref["E_sh"] + 2 * ref["T_sh"]


# rotation angles where a closed-form Rodrigues derivative goes wrong: zero, below and around the
# point where cos(theta) rounds to 1 (~1.5e-8), and up to pi
THETAS = (0.0, 1e-15, 1e-13, 1e-12, 1e-11, 1e-10, 1e-8, 3e-8, 1e-7, 1e-6, 1e-4, 1e-2, 0.5, 2.0,
          math.pi - 1e-6, math.pi)


def board(nc, planar=True, seed=0):
    """(nc, 3) corners of a board centred near the origin (none on it), within |x|, |y| <= 6, rows of
    round(sqrt(nc)) corners (so no 3 of 4 or 5 corners are collinear); planar: z = 0, else z drawn in
    [-1, 1]."""
    n1 = max(1, int(round(math.sqrt(nc))))
    a, b = np.arange(nc) % n1, np.arange(nc) // n1
    n2 = int(b.max()) + 1
    step = 12.0 / max(n1, n2, 2)
    obj = np.zeros((nc, 3))
    obj[:, 0] = (a - (n1 - 1) / 2 + 0.3) * step
    obj[:, 1] = (b - (n2 - 1) / 2 + 0.2) * step
    if not planar:
        obj[:, 2] = np.random.default_rng(seed).uniform(-1.0, 1.0, nc)
    return obj


def case(nc, nv, k=-0.12, aspect=1.0, checker_size=1.0, planar=True, seed=0, thetas=THETAS, noise=0.25):
    """A synthetic problem: view v rotated by thetas[v % len] about a random axis, the board's
    centre 30 to 35 units in front of the camera; image points projected by this module plus Gaussian noise (pixels).
    Returns (intr, views (nv, 6), obj (nc, 3) in world units, img (nv, nc, 2)) with
    intr = (frow, fcol, crow, ccol, k, checker_size), the library's argument."""
    rng = np.random.default_rng(seed)
    axes = rng.normal(size=(nv, 3))
    axes /= np.linalg.norm(axes, axis=1, keepdims=True)
    th = np.array([thetas[v % len(thetas)] for v in range(nv)])
    views = np.concatenate([axes * th[:, None],
                            np.stack([rng.normal(0, 1, nv), rng.normal(0, 1, nv), rng.uniform(30, 35, nv)], 1)], 1)
    obj = board(nc, planar, seed) * checker_size
    f, crow, ccol = 1400.0, 540.0, 960.0
    clean = residual(views, (f, crow, ccol, k), checker_size, aspect, obj, np.zeros((nv, nc, 2)))
    img = clean + rng.normal(0, noise, clean.shape) if noise else clean
    return (aspect * f, f, crow, ccol, k, checker_size), views, obj, img


def mp_jacobian(mp, p, checker_size, aspect, X, h=None):
    """(2, 10) Jacobian of (row, col) at one corner by central differences in mpmath; p: 10 numbers,
    X: (x, y, z).  Run it at mp.dps >= 50: step 1e-20 leaves truncation and rounding below 1e-38."""
    m = _Mp(mp)
    h = mp.mpf("1e-20") if h is None else h
    P = [mp.mpf(float(x)) for x in p]
    Xm = [mp.mpf(float(x)) for x in X]
    J = np.empty((2, NPAR))
    for j in range(NPAR):
        lo, hi = list(P), list(P)
        lo[j] -= h
        hi[j] += h
        a, b = project(hi, checker_size, aspect, Xm, m), project(lo, checker_size, aspect, Xm, m)
        J[0, j] = float((a[0] - b[0]) / (2 * h))
        J[1, j] = float((a[1] - b[1]) / (2 * h))
    return J
