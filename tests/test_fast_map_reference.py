"""The rectification map against an independent high-precision reference (oracle/map_ref.py), on the CPU.

  * the np.longdouble reference agrees with mpmath at 50 digits, at random in-frame pixels and at the
    pixels where the FP32 error is largest;
  * the C oracle's FP64 map -- which the exact kernels equal bit for bit -- is within the FP64 bound of
    the reference at every pixel;
  * a numpy restatement of the fast path's arithmetic is within the FP32 bound at every in-frame pixel,
    the bound is at most 8 times the worst error it covers, and where the lens is monotone
    (1 + 3 k r^2 > 0) and the point is in front of the camera the bound itself is <= 1e-3 px;
  * the bound sees each of three plausible slips in the fast path's host fold and reciprocal.
tests/test_gpu_fast_map_reference.py holds the kernels to the same bounds."""
import functools

import numpy as np
import pytest

from oracle import map_ref as mr
from oracle import oracle_c as oc

GEOMS = mr.geometries()
TOL32_PX = 1e-3


def _err(fr, fc, ch):
    return np.abs(fr - ch.row).astype(np.float64), np.abs(fc - ch.col).astype(np.float64)


@functools.lru_cache(maxsize=None)
def _scan(name):
    """Sweep one geometry: the emulated fast map against the reference and the bounds.  Returns the largest
    emulated error and bound over in-frame pixels, the largest bound where the FP32 map is held to 1e-3 px,
    the number of pixels outside their bound, and the in-frame pixels with the largest emulated errors."""
    g = GEOMS[name]
    s = dict(err=0.0, bound=0.0, bound_mono=0.0, over=0, inframe=0, worst=[])
    for ch in mr.sweep(g):
        inf = ch.inframe(g.sz)
        er, ec = _err(*mr.emulate_fast(g, ch.a, ch.b), ch)
        s["over"] += int(np.sum(inf & ((er > ch.b32_row) | (ec > ch.b32_col))))
        s["inframe"] += int(inf.sum())
        if not inf.any():
            continue
        e = np.where(inf, np.maximum(er, ec), -1.0)
        b = np.maximum(ch.b32_row, ch.b32_col)
        s["err"] = max(s["err"], e.max())
        s["bound"] = max(s["bound"], b[inf].max())
        good = inf & ch.monotone & ch.front
        if good.any():
            s["bound_mono"] = max(s["bound_mono"], b[good].max())
        top = np.argsort(e)[-8:]
        s["worst"] += [(e[i], int(ch.a[i]), int(ch.b[i])) for i in top if e[i] >= 0]
    s["worst"] = sorted(s["worst"])[-16:]
    return s


@pytest.mark.parametrize("name", list(GEOMS))
def test_emulated_fast_map_within_its_bound(name):
    s = _scan(name)
    assert s["inframe"] > 0
    assert s["over"] == 0, s
    assert s["bound_mono"] <= TOL32_PX, s                 # the bound proves the contract there
    assert s["bound"] <= 8 * s["err"], s                  # and is tight


@pytest.mark.parametrize("name", list(GEOMS))
def test_reference_matches_mpmath(name):
    """50-digit mpmath at 2000 random in-frame pixels and at the 16 with the largest FP32 error."""
    pytest.importorskip("mpmath")
    g = GEOMS[name]
    rng = np.random.default_rng(len(name))
    a = rng.integers(0, g.sz[0], 20000)
    b = rng.integers(0, g.sz[1], 20000)
    ch = mr.evaluate(g, a, b)
    keep = np.flatnonzero(ch.inframe(g.sz))[:2000]
    a = np.concatenate([a[keep], [w[1] for w in _scan(name)["worst"]]]).astype(np.int64)
    b = np.concatenate([b[keep], [w[2] for w in _scan(name)["worst"]]]).astype(np.int64)
    ch = mr.evaluate(g, a, b)
    mrow, mcol = mr.mp_map(g, a, b)
    import mpmath
    with mpmath.workdps(50):
        dr = max(abs(mpmath.mpf(float(x)) + mpmath.mpf(float(x - np.longdouble(float(x)))) - m)
                 for x, m in zip(ch.row, mrow))
        dc = max(abs(mpmath.mpf(float(x)) + mpmath.mpf(float(x - np.longdouble(float(x)))) - m)
                 for x, m in zip(ch.col, mcol))
    assert dr <= 1e-12 and dc <= 1e-12, (dr, dc)


@pytest.mark.parametrize("name", list(GEOMS))
def test_oracle_map_within_fp64_bound(name):
    """The FP64 map of the C oracle (and so of the exact kernels, which equal it bit for bit) is accurate,
    not just equal to the oracle: within the FP64 bound of the reference at every pixel."""
    g = GEOMS[name]
    ch0 = oc.chain(g.intr, *g.view)
    omr, omc = oc.rectify_map(ch0, 1.0 / g.ratio, g.axs, g.sz)
    n = 0
    for ch in mr.sweep(g):
        o_r, o_c = omr[ch.b, ch.a], omc[ch.b, ch.a]
        fin = np.isfinite(ch.row.astype(np.float64)) & np.isfinite(ch.col.astype(np.float64))
        assert np.all(np.isfinite(ch.b64_row[fin]) & np.isfinite(ch.b64_col[fin]))
        er, ec = _err(o_r.astype(np.longdouble), o_c.astype(np.longdouble), ch)
        assert np.all(er[fin] <= ch.b64_row[fin]) and np.all(ec[fin] <= ch.b64_col[fin]), name
        n += int(fin.sum())
    assert n == g.sz[0] * g.sz[1] or not mr.LONGDOUBLE_OK


def test_rotation_within_the_assumed_fp64_error():
    """The bounds take the library's rotation matrix (the oracle's, which it equals), expanded in double from
    sin and cos, to within R_ABS64 u of the true rotation: the FP64 path through its P_i, the fast path through
    the doubles its host fold rounds to float.  Checked against mpmath for every geometry's rotation vector."""
    mpmath = pytest.importorskip("mpmath")
    from oracle.fit_ref import _Mp, rotation
    with mpmath.workdps(40):
        for g in GEOMS.values():
            Rm = rotation([mpmath.mpf(c) for c in g.view[0]], _Mp(mpmath.mp))
            R = np.array(oc.chain(g.intr, *g.view).R).reshape(3, 3)
            d = max(abs(mpmath.mpf(float(R[i, j])) - Rm[i][j]) for i in range(3) for j in range(3))
            assert d <= mr.R_ABS64 * mr.U64, (g.view, d)


@pytest.mark.parametrize("name,slip", [("c2_far_axes", dict(recentre=False)),
                                       ("c2_far_axes", dict(round_t=True)),
                                       ("c2_syn", dict(newton=False))])
def test_bound_sees_a_slip_in_the_fast_path(name, slip):
    """The FP32 bound is tight enough to see make_fast without its output-centre shift, with t rounded to
    float before the fold, and a reciprocal one ulp off (rcp.approx without its Newton step at its worst)."""
    g = GEOMS[name]
    over = 0
    for ch in mr.sweep(g):
        inf = ch.inframe(g.sz)
        er, ec = _err(*mr.emulate_fast(g, ch.a, ch.b, **slip), ch)
        over += int(np.sum(inf & ((er > ch.b32_row) | (ec > ch.b32_col))))
    assert over > 0
