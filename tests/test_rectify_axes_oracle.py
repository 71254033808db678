"""Rectification into output axes of any size (cc_rectify_axes_*): the reference of tests/rectify_axes_ref.py and the
Python layer's out_size, on the CPU.

- With the output geometry equal to the source's the reference is the oracle's cco_rectify_*, pixel for pixel.
- A pixel's value does not depend on the output window that holds it: a crop equals the same window of a larger
  output, bit for bit (f32 and u8).
- Downscaled and upscaled outputs are pinned to scipy.ndimage.map_coordinates(order=1), as the same-size rule is in
  test_oracle.py.
- warp / warp_views with out_size call cc_rectify_axes_* with the expected arguments; without it they call what
  they called before (the recorder of test_python_calls.py).
"""
import numpy as np
import pytest

from cameracalibrations_b200 import calibration as cal
from oracle import oracle_c as oc
import rectify_axes_ref as axref
from test_python_calls import INTR, VIEW, NAN, Buf, _cal, _expect, _frames, _rejects, _ret, mode, rec  # noqa: F401

# a tilted view whose output is partly out of frame (test_oracle.py's warp case)
RV, TV = (0.21, -0.17, 0.35), (-3.4, -1.2, 7.0)
CAM = (55.0, 55.0, 30.0, 24.0, 0.06, 1.0)
SZ, AXS, INV_RATIO = (61, 47), (-5, -9), 1.0 / 8.0


def _case(seed=3, nframes=2):
    ch = oc.chain(CAM, RV, TV)
    rng = np.random.default_rng(seed)
    f32 = rng.random((nframes, SZ[1], SZ[0])).astype(np.float32)
    u8 = rng.integers(0, 256, (nframes, SZ[1], SZ[0], 3), dtype=np.uint8)
    return ch, f32, u8


def _same(a, b):
    return np.array_equal(a, b, equal_nan=a.dtype.kind == "f")


def test_axes_reference_equals_same_size_oracle():
    ch, f32, u8 = _case()
    for axs in (AXS, (0, 0), (17, -30)):
        assert _same(axref.rectify_f32c1(ch, INV_RATIO, axs, f32, SZ, fill=np.nan),
                     oc.rectify_f32c1(ch, INV_RATIO, axs, f32, fill=np.nan))
        assert _same(axref.rectify_u8c3(ch, INV_RATIO, axs, u8, SZ, fill=(4, 5, 6)),
                     oc.rectify_u8c3(ch, INV_RATIO, axs, u8, fill=(4, 5, 6)))


@pytest.mark.parametrize("win", [((0, 0), (61, 47)), ((7, 11), (20, 9)), ((33, 2), (1, 40)), ((60, 46), (1, 1))])
def test_axes_reference_crop_identity(win):
    """A window of a larger output (here 2x the source extent, one ratio) equals a call with that window's axes."""
    ch, f32, u8 = _case()
    big_sz = (2 * SZ[0], 2 * SZ[1])
    (o1, o2), (n1, n2) = win
    axs_w = (AXS[0] + o1, AXS[1] + o2)
    big = axref.rectify_f32c1(ch, INV_RATIO, AXS, f32, big_sz, fill=np.nan)
    crop = axref.rectify_f32c1(ch, INV_RATIO, axs_w, f32, (n1, n2), fill=np.nan)
    assert crop.shape == (2, n2, n1)
    assert _same(crop, big[:, o2:o2 + n2, o1:o1 + n1])
    big8 = axref.rectify_u8c3(ch, INV_RATIO, AXS, u8, big_sz, fill=(1, 2, 3))
    crop8 = axref.rectify_u8c3(ch, INV_RATIO, axs_w, u8, (n1, n2), fill=(1, 2, 3))
    assert _same(crop8, big8[:, o2:o2 + n2, o1:o1 + n1])


@pytest.mark.parametrize("scale", [0.5, 2.0, 3.0])
def test_axes_reference_scaled_vs_scipy_map_coordinates(scale):
    """The same world window at another resolution: ratio * scale, axes axs_min * scale, extent sz * scale."""
    ndi = pytest.importorskip("scipy.ndimage")
    ch, f32, u8 = _case(seed=11, nframes=1)
    inv_ratio = INV_RATIO / scale
    axs = (int(round(AXS[0] * scale)), int(round(AXS[1] * scale)))
    out_sz = (int(SZ[0] * scale), int(SZ[1] * scale))
    mr, mc = oc.rectify_map(ch, inv_ratio, axs, out_sz)              # (out_sz2, out_sz1), 1-based source coordinates
    out = axref.rectify_f32c1(ch, inv_ratio, axs, f32, out_sz, fill=np.nan)[0].astype(np.float64)
    assert out.shape == (out_sz[1], out_sz[0])
    ref = ndi.map_coordinates(f32[0].astype(np.float64), [mc - 1.0, mr - 1.0], order=1, mode="constant", cval=np.nan)
    inb = (mr >= 1) & (mr <= SZ[0]) & (mc >= 1) & (mc <= SZ[1])
    assert 0.05 < inb.mean() < 0.95
    assert np.array_equal(np.isnan(out), ~inb) and np.array_equal(np.isnan(ref), ~inb)
    assert np.max(np.abs(out[inb] - ref[inb])) < 1e-7
    out8 = axref.rectify_u8c3(ch, inv_ratio, axs, u8, out_sz, fill=(1, 2, 3))[0]
    for c3 in range(3):
        r8 = ndi.map_coordinates(u8[0, :, :, c3].astype(np.float64), [mc - 1.0, mr - 1.0], order=1,
                                 mode="constant", cval=-1.0)
        assert np.all(out8[:, :, c3][~inb] == (1, 2, 3)[c3])
        frac = np.abs(r8[inb] - np.floor(r8[inb]) - 0.5)
        sure = frac > 1e-9
        assert np.array_equal(out8[:, :, c3][inb][sure], np.rint(r8[inb][sure]).astype(np.uint8))
        assert sure.mean() > 0.99


# ---------------------------------------------------------------- the Python layer's calls
@pytest.mark.parametrize("coord, gather, flags", [("f64", "auto", 0), ("f32", "tma", 33)])
@pytest.mark.parametrize("u8", [False, True])
@pytest.mark.parametrize("single", [False, True])
def test_warp_out_size(rec, mode, coord, gather, flags, u8, single):
    dt, kern = (np.uint8, "u8c3") if u8 else (np.float32, "f32c1")
    shape = ((6, 8) if single else (2, 6, 8)) + ((3,) if u8 else ())
    oshape = ((3, 10) if single else (2, 3, 10)) + ((3,) if u8 else ())
    f = mode.to(_frames(shape, dt))
    y = cal.warp(_cal(), "b_extrinsic.png", f, 0.5, (-3, 4), coord=coord, gather=gather, out_size=(10, 3))
    _ret(y, mode, oshape, dt)
    _expect(rec, mode.name(f"cc_rectify_axes_{kern}"), [
        mode.h, INTR, [VIEW[1]], 1, [0.5], [-3, 4], 10, 3, Buf(dt, shape, own=f), 8, 6, 8, 48,
        Buf(dt, ((1,) if single else ()) + oshape, own=y), 10, 30, 1 if single else 2, [0, 0, 0] if u8 else NAN,
        flags] + mode.tail)


@pytest.mark.parametrize("u8", [False, True])
@pytest.mark.parametrize("single", [False, True])
def test_warp_out_size_with_out(rec, mode, u8, single):
    dt, kern = (np.uint8, "u8c3") if u8 else (np.float32, "f32c1")
    shape = (1 if single else 3, 5, 7) + ((3,) if u8 else ())
    oshape = (1 if single else 3, 9, 4) + ((3,) if u8 else ())
    f = mode.to(_frames(shape[1:] if single else shape, dt))
    out = mode.to(np.zeros(oshape[1:] if single else oshape, dt))
    y = cal.warp(_cal(), 2, f, 1.25, np.array([2, -1]), fill=(1, 2, 3) if u8 else 0.25, out=out, out_size=(4, 9))
    if single:
        _ret(y, mode, oshape[1:], dt)
    else:
        _ret(y, mode, oshape, dt)
    _expect(rec, mode.name(f"cc_rectify_axes_{kern}"), [
        mode.h, INTR, [VIEW[2]], 1, [1.25], [2, -1], 4, 9, Buf(dt, shape[1:] if single else shape, own=f),
        7, 5, 7, 35, Buf(dt, oshape, own=out), 4, 36, shape[0], [1, 2, 3] if u8 else 0.25, 0] + mode.tail)


@pytest.mark.parametrize("u8", [False, True])
def test_warp_views_out_size(rec, mode, u8):
    dt, kern = (np.uint8, "u8c3") if u8 else (np.float32, "f32c1")
    shape = (4, 6, 8) + ((3,) if u8 else ())
    oshape = (4, 12, 5) + ((3,) if u8 else ())
    f = mode.to(_frames(shape, dt))
    y = cal.warp_views(_cal(), [2, "a.png"], f, [0.5, 0.75], [(-3, 4), (1, -2)], coord="f32", out_size=(5, 12))
    _ret(y, mode, oshape, dt)
    _expect(rec, mode.name(f"cc_rectify_axes_{kern}"), [
        mode.h, INTR, [VIEW[2], VIEW[0]], 2, [0.5, 0.75], [-3, 4, 1, -2], 5, 12, Buf(dt, shape, own=f), 8, 6, 8, 48,
        Buf(dt, oshape, own=y), 5, 60, 2, [0, 0, 0] if u8 else NAN, 1] + mode.tail)


def test_warp_without_out_size_calls_the_same_size_symbols(rec, mode):
    f = mode.to(_frames((2, 6, 8), np.float32))
    y = cal.warp(_cal(), 0, f, 1.0, (0, 0), out_size=None)
    _ret(y, mode, (2, 6, 8), np.float32)
    _expect(rec, mode.name("cc_rectify_f32c1"), [mode.h, INTR, VIEW[0], 1.0, [0, 0], Buf(np.float32, (2, 6, 8), own=f),
                                                 Buf(np.float32, (2, 6, 8), own=y), 8, 6, 8, 48, 2, NAN, 0] + mode.tail)
    y = cal.warp_views(_cal(), [0, 1], f, [1.0, 1.0], [(0, 0), (0, 0)])
    name = "cc_rectify_f32c1_views" if mode.cuda else "cc_rectify_views_f32c1_host"
    _expect(rec, name, [mode.h, INTR, [VIEW[0], VIEW[1]], 2, [1.0, 1.0], [0, 0, 0, 0], Buf(np.float32, (2, 6, 8), own=f),
                        Buf(np.float32, (2, 6, 8), own=y), 8, 6, 8, 48, 1, NAN, 0] + mode.tail)


def test_warp_out_size_rejects_a_wrong_out(rec, mode):
    c = _cal()
    f = mode.to(_frames((2, 6, 8), np.float32))
    _rejects(rec, ValueError, lambda: cal.warp(c, 0, f, 1.0, (0, 0), out=mode.to(np.zeros((2, 6, 8), np.float32)),
                                               out_size=(4, 3)))
    _rejects(rec, ValueError, lambda: cal.warp(c, 0, f, 1.0, (0, 0), out=mode.to(np.zeros((2, 3, 4), np.uint8)),
                                               out_size=(4, 3)))
    _rejects(rec, ValueError, lambda: cal.warp_views(c, [0, 1], f, [1.0, 1.0], [(0, 0), (0, 0)],
                                                     out=mode.to(np.zeros((2, 4, 3), np.float32)), out_size=(4, 3)))
