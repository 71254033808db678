"""An independent reference of the rectification map and per-pixel bounds on the error of the two
device pipelines that compute it.  TEST INFRASTRUCTURE ONLY.

The map (src/plot_calibration.jl:17-18): output pixel (I1, I2) samples the source image at
  real2image[i] o push(., 0) o inv(LinearMap(ratio*I)),
i.e. with q = (I1, I2) / (ratio * cs) and the rotation R of the view's rotation vector,
  P = R[:, 0] q1 + R[:, 1] q2 + t,  (u, v) = (P1, P2) / P3,  radial = 1 + k (u^2 + v^2),
  (row, col) = (frow radial u + crow, fcol radial v + ccol).
It is evaluated here in np.longdouble (64-bit significand or more; elsewhere mpmath on a subsample)
and, on a few thousand pixels, in mpmath at 50 digits.  R comes from fit_ref.rotation; nothing is
shared with oracle/camcal_oracle.c or the kernels.

The bounds are first order: every rounding z -> z (1 + e), |e| <= u, of the kernel's own sequence,
propagated to (row, col) through the partial derivatives of the rest of the chain,
  |d row| <= SAFETY * u * sum_z |d row / d z| * |z|,
with u = 2^-24 for the fast path (CC_COORD_F32, rectify_device.cuh: RectFast) and 2^-53 for the exact
path (RectExact).  For the fast path |z| is taken as the power of two at or below it (half an ulp of z
is u times that), and the host fold's roundings of A, C, T and of the camera constants to float enter
with their actual values (every float a rounding may give, where the doubles are not known to the last
bit): both keep the bound within ~7 % of the worst error it covers.  The derivatives that matter are
1/|P3| (on the sums of |terms| of each P_i) and the slope of the lens, 1 + 3 k r^2 along the radius: past the fold of the distortion polynomial
(r^2 > 1/(3|k|)) it magnifies the rounding of u and v by up to ~1e4 at in-frame pixels, which is why the
FP32 map is held to 1e-3 px only where the lens is monotone and the point is in front of the camera.
"""
from __future__ import annotations

import itertools
from dataclasses import dataclass

import numpy as np

from oracle.fit_ref import _Mp, rotation

U32 = 2.0 ** -24
U64 = 2.0 ** -53
# the first-order terms are evaluated at the exact intermediates and the bound is used only where the
# relative perturbation of P3 is below LINEAR, so the second-order rest is a few LINEAR of it; the factor
# also covers the double rounding (FP64, then FP32) of the emulation below, 2^-29 relative per step
SAFETY = 1.0625
# rcp.approx.ftz.f32 is within 1 ulp (2^-23); one Newton step squares that and adds one rounding
RCP32 = U32 * (1.0 + 2.0 ** -20)
# the exact path's R, from sin / cos in double: |dR_ij| <= 8 u (checked against mpmath by the tests)
R_ABS64 = 8.0
# the first-order bound is reported only where it linearises: |dP3 / P3| below this
LINEAR = 2.0 ** -10
CHUNK = 1 << 20                      # pixels per longdouble chunk
LONGDOUBLE_OK = np.finfo(np.longdouble).nmant >= 63


@dataclass(frozen=True)
class Geom:
    intr: tuple        # (frow, fcol, crow, ccol, k, checker_size)
    view: tuple        # (rvec, tvec)
    ratio: float
    axs: tuple         # axs_min (first, second axis)
    sz: tuple          # (sz1, sz2): sz1 contiguous


def board_ratio(intr, view, n=(20, 14)):
    """get_ratio of the board's own projected corners (src/plot_calibration.jl:1-6)."""
    a, b = np.meshgrid(np.arange(n[0], dtype=np.float64), np.arange(n[1], dtype=np.float64), indexing="ij")
    row, col = _world2img(intr, view, a * intr[5], b * intr[5], np.float64)
    d1 = np.hypot(np.diff(row, axis=0), np.diff(col, axis=0)).mean()
    d2 = np.hypot(np.diff(row, axis=1), np.diff(col, axis=1)).mean()
    return float((d1 + d2) / 2.0 / intr[5])


def axes(ratio, cs, n, sz):
    w = [np.rint(ratio * cs * (m - 1)) for m in n]
    return tuple(int(np.rint((w[i] - sz[i]) / 2.0)) for i in range(2))


def geom(intr, view, sz, ratio_scale=1.0, ratio=None, axs=None, n=(20, 14)):
    """A Geom with the board's ratio (times ratio_scale) and centred axes unless given."""
    if ratio is None:
        ratio = board_ratio(intr, view, n) * ratio_scale
    if axs is None:
        axs = axes(ratio, intr[5], n, sz)
    return Geom(tuple(float(x) for x in intr), (tuple(map(float, view[0])), tuple(map(float, view[1]))),
                float(ratio), tuple(int(x) for x in axs), tuple(int(x) for x in sz))


def _world2img(intr, view, x, y, dt):
    R = rotation([dt(c) for c in view[0]])
    cs = dt(intr[5])
    t = [dt(c) for c in view[1]]
    P = [R[i][0] * (x / cs) + R[i][1] * (y / cs) + t[i] for i in range(3)]
    u, v = P[0] / P[2], P[1] / P[2]
    radial = 1 + dt(intr[4]) * (u * u + v * v)
    return dt(intr[0]) * radial * u + dt(intr[2]), dt(intr[1]) * radial * v + dt(intr[3])


# ------------------------------------------------------------------ reference values
def _chain_ld(g: Geom, a, b):
    """Every intermediate of the map at output pixels (a, b) (0-based), in np.longdouble."""
    ld = np.longdouble
    R = rotation([ld(c) for c in g.view[0]])
    den = ld(g.ratio) * ld(g.intr[5])
    q1 = (ld(g.axs[0]) + a.astype(ld)) / den
    q2 = (ld(g.axs[1]) + b.astype(ld)) / den
    P = [R[i][0] * q1 + (R[i][1] * q2 + ld(g.view[1][i])) for i in range(3)]
    u, v = P[0] / P[2], P[1] / P[2]
    r2 = u * u + v * v
    radial = ld(g.intr[4]) * r2 + 1
    row = (ld(g.intr[0]) * u) * radial + ld(g.intr[2])
    col = (ld(g.intr[1]) * v) * radial + ld(g.intr[3])
    return dict(q1=q1, q2=q2, P=P, u=u, v=v, r2=r2, radial=radial, row=row, col=col, R=R)


def mp_map(g: Geom, a, b, dps=50):
    """(row, col) at pixels (a, b) in mpmath at dps digits, as lists of mpf."""
    import mpmath
    with mpmath.workdps(dps):
        mp = mpmath.mp
        R = rotation([mp.mpf(c) for c in g.view[0]], _Mp(mp))
        den = mp.mpf(g.ratio) * mp.mpf(g.intr[5])
        t = [mp.mpf(c) for c in g.view[1]]
        frow, fcol, crow, ccol, k = (mp.mpf(c) for c in g.intr[:5])
        rows, cols = [], []
        for ai, bi in zip(np.asarray(a).tolist(), np.asarray(b).tolist()):
            q1, q2 = (g.axs[0] + ai) / den, (g.axs[1] + bi) / den
            P = [R[i][0] * q1 + R[i][1] * q2 + t[i] for i in range(3)]
            u, v = P[0] / P[2], P[1] / P[2]
            radial = 1 + k * (u * u + v * v)
            rows.append(frow * radial * u + crow)
            cols.append(fcol * radial * v + ccol)
        return rows, cols


def _chain_mp(g: Geom, a, b):
    """_chain_ld's fields from mpmath, for platforms whose longdouble is a double."""
    import mpmath
    with mpmath.workdps(40):
        mp = mpmath.mp
        R = rotation([mp.mpf(c) for c in g.view[0]], _Mp(mp))
        den = mp.mpf(g.ratio) * mp.mpf(g.intr[5])
        out = {n: [] for n in ("q1", "q2", "P0", "P1", "P2", "u", "v", "r2", "radial", "row", "col")}
        for ai, bi in zip(a.tolist(), b.tolist()):
            q1, q2 = (g.axs[0] + ai) / den, (g.axs[1] + bi) / den
            P = [R[i][0] * q1 + R[i][1] * q2 + mp.mpf(g.view[1][i]) for i in range(3)]
            u, v = P[0] / P[2], P[1] / P[2]
            r2 = u * u + v * v
            radial = 1 + mp.mpf(g.intr[4]) * r2
            for n, x in (("q1", q1), ("q2", q2), ("P0", P[0]), ("P1", P[1]), ("P2", P[2]), ("u", u), ("v", v),
                         ("r2", r2), ("radial", radial), ("row", mp.mpf(g.intr[0]) * radial * u + mp.mpf(g.intr[2])),
                         ("col", mp.mpf(g.intr[1]) * radial * v + mp.mpf(g.intr[3]))):
                out[n].append(float(x) if n not in ("row", "col") else x)
        f = {n: np.array(out[n], dtype=np.float64) for n in out if n not in ("row", "col")}
        f["P"] = [f.pop("P0"), f.pop("P1"), f.pop("P2")]
        f["row"] = np.array([float(x) for x in out["row"]])
        f["col"] = np.array([float(x) for x in out["col"]])
        f["R"] = [[float(x) for x in r] for r in R]
        return f


# ------------------------------------------------------------------ the fast path's host fold
def fast_params(g: Geom):
    """make_fast (rectify.cu) in double: A, C, T rounded to float, the output centre (c1, c2)."""
    R = np.array(rotation([np.float64(c) for c in g.view[0]]), dtype=np.float64)
    sc = (1.0 / g.ratio) * (1.0 / g.intr[5])
    c1 = float(np.rint(g.axs[0] + 0.5 * (g.sz[0] - 1)))
    c2 = float(np.rint(g.axs[1] + 0.5 * (g.sz[1] - 1)))
    A, C = R[:, 0] * sc, R[:, 1] * sc
    T = np.asarray(g.view[1], dtype=np.float64) + A * c1 + C * c2
    f = np.float32
    return dict(A=A.astype(f), C=C.astype(f), T=T.astype(f), c1=f(c1), c2=f(c2),
                k=f(g.intr[4]), frow=f(g.intr[0]), fcol=f(g.intr[1]), crow=f(g.intr[2]), ccol=f(g.intr[3]))


def _fmaf(a, b, c):
    """fmaf emulated: the product of two floats is exact in double, the sum is rounded twice (double, float)"""
    return (a.astype(np.float64) * b + c).astype(np.float32)


def emulate_fast(g: Geom, a, b, newton=True, recentre=True, round_t=False):
    """rect_row_term + rect_coord(RectFast) in numpy: FP32 throughout, fused multiply-adds as _fmaf, the
    reciprocal correctly rounded (standing in for rcp.approx + one Newton step; newton=False: 1 ulp off,
    the worst rcp.approx allows).  recentre=False / round_t=True emulate make_fast without the output-centre
    shift, and with t rounded to float before the fold."""
    p = fast_params(g)
    if not recentre or round_t:
        R = np.array(rotation([np.float64(c) for c in g.view[0]]), dtype=np.float64)
        sc = (1.0 / g.ratio) * (1.0 / g.intr[5])
        c1 = float(p["c1"]) if recentre else 0.0
        c2 = float(p["c2"]) if recentre else 0.0
        t = np.asarray(g.view[1], dtype=np.float64)
        if round_t:
            t = t.astype(np.float32).astype(np.float64)
        p["T"] = (t + R[:, 0] * sc * c1 + R[:, 1] * sc * c2).astype(np.float32)
        p["c1"], p["c2"] = np.float32(c1), np.float32(c2)
    f = np.float32
    i1 = (np.asarray(a) + g.axs[0]).astype(f) - p["c1"]
    i2 = (np.asarray(b) + g.axs[1]).astype(f) - p["c2"]
    B = [_fmaf(p["A"][i], i1, p["T"][i]) for i in range(3)]
    P = [_fmaf(p["C"][i], i2, B[i]) for i in range(3)]
    with np.errstate(divide="ignore", invalid="ignore", over="ignore"):
        s = (1.0 / P[2].astype(np.float64)).astype(f)
        if not newton:                       # one ulp away from the correctly rounded reciprocal
            s = np.nextafter(s, np.where(s > 0, f(np.inf), f(-np.inf)))
        u, v = P[0] * s, P[1] * s
        if p["k"] != 0:
            r2 = _fmaf(v, v, u * u)
            radial = _fmaf(np.broadcast_to(p["k"], r2.shape), r2, f(1))
            u, v = u * radial, v * radial
        row = _fmaf(np.broadcast_to(p["frow"], u.shape), u, p["crow"])
        col = _fmaf(np.broadcast_to(p["fcol"], v.shape), v, p["ccol"])
    return row, col


# ------------------------------------------------------------------ the bounds
def _p2(x, d):
    """2^floor(log2(|x| + d)): half an ulp of any float within d of x is u times this"""
    m, e = np.frexp(np.abs(x) + d)
    return np.ldexp(np.where(m > 0, 0.5, 0.0), e)


def _bound(g: Geom, ch, a, b, fast):
    """(row, col) error bounds at pixels (a, b) for the fast (fast=True) or the exact path, first order in the
    roundings of the kernel's sequence, evaluated at the exact intermediates ch."""
    f8 = np.float64
    U = U32 if fast else U64
    frow, fcol, crow, ccol, k = (f8(x) for x in g.intr[:5])
    q1, q2 = ch["q1"].astype(f8), ch["q2"].astype(f8)
    P = [x.astype(f8) for x in ch["P"]]
    u, v, r2, radial = (ch[n].astype(f8) for n in ("u", "v", "r2", "radial"))
    row, col = ch["row"].astype(f8), ch["col"].astype(f8)
    R = np.array([[f8(x) for x in r] for r in ch["R"]])
    t = np.asarray(g.view[1], dtype=f8)
    with np.errstate(divide="ignore", invalid="ignore", over="ignore"):
        # the exact path's P_i: q = (I * fl(1/ratio)) * fl(1/cs) (four roundings), R within R_ABS64 u,
        # B_i = fma(R_i0, q1, t_i), P_i = fma(R_i1, q2, B_i)
        dP64 = [U64 * (R_ABS64 * (np.abs(q1) + np.abs(q2)) + 4 * (np.abs(R[i, 0] * q1) + np.abs(R[i, 1] * q2))
                       + np.abs(R[i, 0] * q1 + t[i]) + np.abs(P[i])) for i in range(3)]
        if fast:
            # make_fast: A, C and T = t + A c1 + C c2 in double, rounded to float; B_i = fmaf(A_i, I1 - c1, T_i),
            # P_i = fmaf(C_i, I2 - c2, B_i).  The float roundings of A, C, T enter with their actual values: the
            # library's doubles lie within dA, dC, dT of those computed here (its R within R_ABS64 u of the
            # rotation, this one within u), and where that interval straddles a float rounding boundary every
            # float it can round to is tried and the worst taken
            fp = fast_params(g)
            sc = (1.0 / g.ratio) * (1.0 / g.intr[5])
            A, C = R[:, 0] * sc, R[:, 1] * sc
            c1, c2 = f8(fp["c1"]), f8(fp["c2"])
            T = t + A * c1 + C * c2
            dA = (2 * R_ABS64 + 1) * U64 * sc + 4 * U64 * np.abs(A)
            dC = (2 * R_ABS64 + 1) * U64 * sc + 4 * U64 * np.abs(C)
            dT = dA * abs(c1) + dC * abs(c2) + 4 * U64 * (np.abs(t) + np.abs(A * c1) + np.abs(C * c2))
            i1, i2 = a + (g.axs[0] - c1), b + (g.axs[1] - c2)

            def floats(x, d):
                return sorted({f8(np.float32(x - d)), f8(np.float32(x + d))})

            dP = []
            for i in range(3):
                fold = 0.0
                for fa, fc, ft in itertools.product(floats(A[i], dA[i]), floats(C[i], dC[i]), floats(T[i], dT[i])):
                    fold = np.maximum(fold, np.abs((fa - A[i]) * i1 + (fc - C[i]) * i2 + (ft - T[i])))
                fold = fold + dP64[i] + dA[i] * np.abs(i1) + dC[i] * np.abs(i2) + dT[i]
                B = T[i] + A[i] * i1
                d = fold + U * (np.abs(B) + np.abs(P[i]))           # margin for the binades below
                dP.append(fold + U * (_p2(B, 2 * d) + _p2(P[i], 2 * d)))
            dk, dfrow, dfcol = f8(fp["k"]) - k, f8(fp["frow"]) - frow, f8(fp["fcol"]) - fcol
            dcrow, dccol = abs(f8(fp["crow"]) - crow), abs(f8(fp["ccol"]) - ccol)
            rnd = _p2
            rcp = RCP32                                              # the reciprocal, relative
        else:
            dP, dk, dfrow, dfcol, dcrow, dccol = dP64, 0.0, 0.0, 0.0, 0.0, 0.0
            rnd = lambda x, d: np.abs(x) + d                         # noqa: E731
            rcp = U64                                                # 1.0 / P3 is correctly rounded
        aP3 = np.abs(P[2])
        s = 1.0 / P[2]
        es = U * rnd(s, 2 * np.abs(s) * (dP[2] / aP3 + 2 * U)) / np.abs(s) + (rcp - U)
        # first-order errors of the intermediates: only used to pick the binade of the value a rounding sees
        du = 2 * ((dP[0] + np.abs(u) * dP[2]) / aP3 + 2 * U * np.abs(u))
        dv = 2 * ((dP[1] + np.abs(v) * dP[2]) / aP3 + 2 * U * np.abs(v))
        dr2 = 2 * np.abs(u) * du + 2 * np.abs(v) * dv + 2 * U * r2
        drad = np.abs(k) * dr2 + 2 * U + np.abs(r2 * dk)
        # slopes of the lens: d(radial u, radial v) / d(u, v); along the radius it is 1 + 3 k r^2
        gu, gv = 1 + k * (3 * u * u + v * v), 2 * k * u * v
        hu, hv = gv, 1 + k * (u * u + 3 * v * v)
        out = []
        for f, df, dc, x, w, dw, su, sv in ((frow, dfrow, dcrow, row, u, du, gu, gv),
                                            (fcol, dfcol, dccol, col, v, dv, hu, hv)):
            # P_i, the reciprocal, u = P1 s and v = P2 s
            e = (np.abs(su) * dP[0] + np.abs(sv) * dP[1] + np.abs(su * u + sv * v) * dP[2]) / aP3 \
                + np.abs(su * u + sv * v) * es + U * (np.abs(su) * rnd(u, du) + np.abs(sv) * rnd(v, dv))
            if k != 0:
                # u*u, the r2 fma, radial (and k rounded to float), the product radial * u
                e = e + np.abs(k * w) * U * (rnd(u * u, 2 * np.abs(u) * du) + rnd(r2, dr2)) \
                    + np.abs(w) * (U * rnd(radial, drad) + np.abs(r2 * dk)) \
                    + U * rnd(w * radial, np.abs(radial) * dw + np.abs(w) * drad)
            wr = w * radial if k != 0 else w
            e = f * e + np.abs(df * wr) + dc                         # frow, crow rounded to float
            e = e + U * rnd(x, 2 * f * (np.abs(e / f)) + 2 * U * np.abs(x))   # the last fma
            ok = dP[2] / aP3 <= LINEAR
            out.append(np.where(ok, SAFETY * e, np.inf))
    return out


@dataclass
class Chunk:
    a: np.ndarray            # first-axis output index (0-based)
    b: np.ndarray            # second-axis output index (0-based)
    row: np.ndarray          # reference map: np.longdouble (or float64 from mpmath)
    col: np.ndarray
    b32_row: np.ndarray      # per-pixel bounds, px
    b32_col: np.ndarray
    b64_row: np.ndarray
    b64_col: np.ndarray
    monotone: np.ndarray     # 1 + 3 k r^2 > 0
    front: np.ndarray        # P3 > 0

    def inframe(self, sz):
        """the reference map is inside the frame: 1 <= row <= sz1, 1 <= col <= sz2"""
        return (self.row >= 1) & (self.row <= sz[0]) & (self.col >= 1) & (self.col <= sz[1])


def evaluate(g: Geom, a, b) -> Chunk:
    a, b = np.asarray(a, dtype=np.int64).ravel(), np.asarray(b, dtype=np.int64).ravel()
    ch = _chain_ld(g, a, b) if LONGDOUBLE_OK else _chain_mp(g, a, b)
    af, bf = a.astype(np.float64), b.astype(np.float64)
    (b32r, b32c), (b64r, b64c) = _bound(g, ch, af, bf, True), _bound(g, ch, af, bf, False)
    mono = 1 + 3 * g.intr[4] * ch["r2"].astype(np.float64) > 0
    return Chunk(a, b, ch["row"], ch["col"], b32r, b32c, b64r, b64c, mono, ch["P"][2] > 0)


def sweep(g: Geom, sample=20000, seed=0):
    """Chunks covering every output pixel, whole lines at a time; where np.longdouble is a double, one
    chunk of `sample` random pixels evaluated in mpmath instead."""
    sz1, sz2 = g.sz
    if not LONGDOUBLE_OK:
        rng = np.random.default_rng(seed)
        n = min(sample, sz1 * sz2)
        flat = rng.choice(sz1 * sz2, size=n, replace=False)
        yield evaluate(g, flat % sz1, flat // sz1)
        return
    lines = max(1, CHUNK // sz1)
    for b0 in range(0, sz2, lines):
        b1 = min(sz2, b0 + lines)
        bb, aa = np.meshgrid(np.arange(b0, b1), np.arange(sz1), indexing="ij")
        yield evaluate(g, aa, bb)


# ------------------------------------------------------------------ geometries
C2 = (1400.0, 1400.0, 540.0, 960.0, -0.12, 1.0)          # 1080 x 1920
C3 = (2800.0, 2800.0, 1080.0, 1920.0, -0.12, 1.0)        # 2160 x 3840
SYN_VIEW = ((0.15, -0.1, 0.02), (-8.0, -12.0, 30.0))
HORIZON_VIEW = ((1.45, 0.1, 0.0), (-3.0, -2.0, 2.0))


def camera_for(sz, k=-0.12):
    f = 1400.0 / 1080.0 * sz[0]
    return (f, f, sz[0] / 2.0, sz[1] / 2.0, k, 1.0)


def _tilted(rx, rz=0.3):
    return ((rx, 0.1, rz), (-8.0, -12.0, 30.0))


def _k(intr, k):
    return intr[:4] + (k, intr[5])


def geometries():
    """name -> Geom: the two cameras; boards tilted by rx = 0.6, 0.9, 1.3 and a negative rz; ratios of 0.4,
    1 and 2.5 times the board's; k = -0.12, 0, 0.3; a view with a horizon inside the output; output axes
    thousands of pixels from the origin (where the fast path's re-centring matters); odd small frames."""
    C2sz, C3sz = (1080, 1920), (2160, 3840)
    return {
        "c2_syn": geom(C2, SYN_VIEW, C2sz),
        "c3_syn": geom(C3, SYN_VIEW, C3sz),
        "c3_rx0.6_r0.4": geom(C3, _tilted(0.6), C3sz, 0.4),
        "c2_rx0.9_r1": geom(C2, _tilted(0.9), C2sz, 1.0),
        "c3_rx1.3_r1": geom(C3, _tilted(1.3), C3sz, 1.0),
        "c3_rx1.3_r0.4": geom(C3, _tilted(1.3), C3sz, 0.4),
        "c3_rx1.3_r0.4_k0": geom(_k(C3, 0.0), _tilted(1.3), C3sz, 0.4),
        "c2_rx0.6_r2.5": geom(C2, _tilted(0.6), C2sz, 2.5),
        "c2_rx0.9_r2.5_k0.3": geom(_k(C2, 0.3), _tilted(0.9), C2sz, 2.5),
        "c2_rx1.3_r0.4_k0.3": geom(_k(C2, 0.3), _tilted(1.3), C2sz, 0.4),
        "c2_rx0.6_rz-0.5_r1": geom(C2, _tilted(0.6, -0.5), C2sz, 1.0),
        "horizon_r6": geom(camera_for((256, 192)), HORIZON_VIEW, (256, 192), ratio=6.0, axs=(-40, -30)),
        "horizon_r1.5": geom(camera_for((256, 192)), HORIZON_VIEW, (256, 192), ratio=1.5, axs=(-200, -400)),
        "c2_far_axes": geom(C2, ((0.15, -0.1, 0.02), (-24.5, 13.7, 12.0)), C2sz, ratio=120.0, axs=(2400, -2600)),
        "odd_131x77": geom(camera_for((131, 77)), _tilted(0.9), (131, 77), 0.4),
        "odd_33x17_k0.3": geom(camera_for((33, 17), 0.3), _tilted(0.6, -0.5), (33, 17), 1.0),
        "odd_5x3": geom(camera_for((5, 3)), SYN_VIEW, (5, 3)),
    }
