"""GPU parity tests: the CUDA path (through the C ABI) against the CPU oracle on the same
seeded inputs.  Tolerances (BASELINE.json north_star):
  FP64 kernels            <= 1e-9 px / world units
  FP32 fast path          <= 1e-3 px (round trip / map error)
  FP64 remap              bit-exact map, indices, weights and output
"""
import os
import ctypes as C

import numpy as np
import pytest

torch = pytest.importorskip("torch")

from conftest import BENCH_VIEW, C2_INTR, C3_INTR, SYN_VIEW, camera_for, load_golden
from oracle import oracle_c as oc

pytestmark = pytest.mark.gpu

TOL64 = 1e-9
TOL32_PX = 1e-3


@pytest.fixture(scope="module")
def cc():
    import cameracalibrations_b200 as m
    assert torch.cuda.is_available(), "GPU tests need a CUDA device"
    m.context(0)  # raises if the extension cannot run: no fallback
    return m


def _calib(cc, intr, views, files=None):
    files = files or [f"{i}.png" for i in range(len(views))]
    return cc.Calibration(intr[:4], views, 1.0 / intr[5], intr[4], files)


def _dev(a, dtype=None):
    t = torch.from_numpy(np.ascontiguousarray(a))
    if dtype is not None:
        t = t.to(dtype)
    return t.cuda()


# ------------------------------------------------------------------ point maps
def test_config1_every_pixel_round_trip(cc, example_fit):
    """BASELINE config 1: c(RowCol,1) <-> c(xyz,1) over every pixel of one 375x500 frame."""
    intr = example_fit["intr_tuple"]
    c = _calib(cc, intr, example_fit["view_list"], example_fit["files"])
    sz1, sz2 = example_fit["sz"]
    r, q = np.meshgrid(np.arange(1, sz1 + 1, dtype=np.float64), np.arange(1, sz2 + 1, dtype=np.float64),
                       indexing="ij")
    r, q = r.ravel(), q.ravel()
    for vi, (rv, tv) in enumerate(example_fit["view_list"]):
        ch = oc.chain(intr, rv, tv)
        ox, oy, oz = oc.img2world_soa(ch, r, q)
        x, y, z = c.img2world(_dev(r), _dev(q), vi)
        for got, ref in ((x, ox), (y, oy), (z, oz)):
            assert np.max(np.abs(got.cpu().numpy() - ref)) <= TOL64
        row, col = c.world2img(x, y, z, vi)
        assert np.max(np.abs(row.cpu().numpy() - r)) <= TOL64
        assert np.max(np.abs(col.cpu().numpy() - q)) <= TOL64
        # the AoS callable of the reference: (n,2) -> (n,3) -> (n,2)
        pts = torch.stack([_dev(r[:1000]), _dev(q[:1000])], dim=-1)
        back = c(c(pts, vi), vi)
        assert torch.max(torch.abs(back - pts)).item() <= TOL64


def test_reference_rectification_identity(cc, example_fit):
    """test/runtests.jl:79-85: rectification(c,1)(RowCol(1,2)) == c(RowCol(1,2),1)[[1,2]] (exact)."""
    c = _calib(cc, example_fit["intr_tuple"], example_fit["view_list"], example_fit["files"])
    i = torch.tensor([[1.0, 2.0]], dtype=torch.float64, device="cuda")
    f = cc.rectification(c, 0)
    assert torch.equal(f(i), c(i, 0)[:, :2])
    # host path, same identity and same numbers
    ih = np.array([[1.0, 2.0]])
    assert np.array_equal(cc.rectification(c, 0)(ih), c(ih, 0)[:, :2])
    assert np.array_equal(c(ih, 0), c(i, 0).cpu().numpy())
    # SURVEY Appendix A known answer
    assert abs(c(ih, 0)[0, 0] - (-0.709323329459491)) < 1e-12


@pytest.mark.parametrize("k", [-0.12, 0.0, 0.056417832172007555, 0.9])
def test_img2world_f64_random_points(cc, k):
    intr = C3_INTR[:4] + (k, 2.5)
    c = _calib(cc, intr, [SYN_VIEW])
    ch = oc.chain(intr, *SYN_VIEW)
    rng = np.random.default_rng(99)
    n = 1_000_003  # odd: exercises the scalar tail
    row, col = rng.uniform(0, 2160, n), rng.uniform(0, 3840, n)
    ox, oy, oz = oc.img2world_soa(ch, row, col)
    x, y, z = c.img2world(_dev(row), _dev(col), 0)
    scale = max(1.0, float(np.max(np.abs(ox))), float(np.max(np.abs(oy))))
    for got, ref in ((x, ox), (y, oy), (z, oz)):
        assert np.max(np.abs(got.cpu().numpy() - ref)) <= TOL64 * scale
    # rectification variant (z == NULL) gives the same x, y bit for bit
    x2, y2 = c.img2world(_dev(row), _dev(col), 0, want_z=False)
    assert torch.equal(x2, x) and torch.equal(y2, y)
    # unaligned views take the scalar path: same bits
    x3, y3, z3 = c.img2world(_dev(row)[1:], _dev(col)[1:], 0)
    assert torch.equal(x3, x[1:]) and torch.equal(z3, z[1:])
    # world -> pixel is the same operation order as the oracle: bit-exact
    orow, ocol = oc.world2img_soa(ch, ox, oy, oz)
    r2, c2 = c.world2img(_dev(ox), _dev(oy), _dev(oz), 0)
    assert np.array_equal(r2.cpu().numpy(), orow) and np.array_equal(c2.cpu().numpy(), ocol)
    assert np.max(np.abs(orow - row)) < 1e-8


def test_inverse_distortion_branches(cc):
    """c == 0, c > 0 large, -4/27 < c < 0 up to the double root, c < -4/27 (negative root)."""
    intr = (1.0, 1.0, 0.0, 0.0, 1.0, 1.0)   # u = row, v = col, k = 1  ->  c = row^2 + col^2
    view = ((0.0, 0.0, 0.0), (0.0, 0.0, 1.0))
    cs = np.concatenate([[0.0, 1e-300, 1e-12, 40.0, 1e3], np.linspace(1e-6, 8, 500)])
    row = np.sqrt(cs)
    col = np.zeros_like(row)
    c = _calib(cc, intr, [view])
    x, y, z = c.img2world(_dev(row), _dev(col), 0)
    ox, oy, oz = oc.img2world_soa(oc.chain(intr, *view), row, col)
    assert np.max(np.abs(x.cpu().numpy() - ox)) <= TOL64
    # negative k: c = -r^2
    intr = (1.0, 1.0, 0.0, 0.0, -1.0, 1.0)
    cneg = np.concatenate([np.linspace(1e-6, 0.148, 400), np.linspace(0.1485, 3.0, 200)])
    row = np.sqrt(cneg)
    col = np.zeros_like(row)
    c = _calib(cc, intr, [view])
    x, y, z = c.img2world(_dev(row), _dev(col), 0)
    ox, oy, oz = oc.img2world_soa(oc.chain(intr, *view), row, col)
    near = np.abs(cneg - 4 / 27) < 2e-3      # double root: conditioning ~ 1/sqrt(distance)
    assert np.max(np.abs(x.cpu().numpy() - ox)[~near]) <= TOL64
    assert np.max(np.abs(x.cpu().numpy() - ox)[near]) <= 1e-6
    assert np.all(x.cpu().numpy()[cneg > 0.1485] < 0)      # the reference divides by the negative root
    # c within a FLOAT ulp of -4/27 on either side: the branch (three real roots / one negative
    # root) is decided in the input precision, so the sign of the result follows the oracle's
    edge = 4.0 / 27.0 + np.array([-1e-8, -3e-9, -1e-10, 1e-10, 3e-9, 1e-8])
    row = np.sqrt(edge)
    x, y, z = c.img2world(_dev(row), _dev(np.zeros_like(row)), 0)
    ox, oy, oz = oc.img2world_soa(oc.chain(intr, *view), row, np.zeros_like(row))
    cedge = row * row                                      # what the chain actually sees
    assert np.array_equal(np.sign(x.cpu().numpy()), np.sign(ox))
    assert np.all(ox[cedge < 4.0 / 27.0 - 1e-12] > 0) and np.all(ox[cedge > 4.0 / 27.0 + 1e-12] < 0)
    assert np.max(np.abs(x.cpu().numpy() - ox)) <= 1e-3   # ill-conditioned at the double root: ~sqrt(distance)


def test_f32_fast_path_round_trip(cc):
    """FP32 kernels: world->pixel of the FP32 pixel->world result, evaluated in FP64 by the
    oracle, lands within 1e-3 px of the input pixel (4K camera)."""
    c = _calib(cc, C3_INTR, [SYN_VIEW])
    ch = oc.chain(C3_INTR, *SYN_VIEW)
    rng = np.random.default_rng(7)
    n = 400_001
    row = rng.uniform(0, 2160, n).astype(np.float32)
    col = rng.uniform(0, 3840, n).astype(np.float32)
    x, y, z = c.img2world(_dev(row), _dev(col), 0)
    assert x.dtype == torch.float32
    r64, c64 = oc.world2img_soa(ch, x.cpu().numpy().astype(np.float64), y.cpu().numpy().astype(np.float64),
                                z.cpu().numpy().astype(np.float64))
    err = np.maximum(np.abs(r64 - row), np.abs(c64 - col))
    assert np.max(err) <= TOL32_PX, np.max(err)
    # FP32 forward map against the FP64 oracle
    ox, oy, oz = oc.img2world_soa(ch, row.astype(np.float64), col.astype(np.float64))
    r32, c32 = c.world2img(_dev(ox, torch.float32), _dev(oy, torch.float32), None, 0)
    r64, c64 = oc.world2img_soa(ch, ox.astype(np.float32).astype(np.float64),
                                oy.astype(np.float32).astype(np.float64))
    assert np.max(np.abs(r32.cpu().numpy() - r64)) <= TOL32_PX
    assert np.max(np.abs(c32.cpu().numpy() - c64)) <= TOL32_PX


@pytest.mark.parametrize("k", [0.0, 0.056417832172007555, 0.9, 1.5, 3.0, -0.2])
def test_f32_inverse_distortion_fixed_and_generic_schedules(cc, k):
    """FP32 pixel->world over lenses whose c = k r^2 stays inside the fixed-schedule range
    [-0.12, 1] (k <= 1.5 on this frame), straddles its upper end (k = 3) or its lower end (k = -0.2:
    c down to -0.124): the FP64 oracle maps the FP32 world point back within 1e-3 px."""
    intr = C3_INTR[:4] + (k, 1.0)
    c = _calib(cc, intr, [SYN_VIEW])
    ch = oc.chain(intr, *SYN_VIEW)
    rng = np.random.default_rng(17)
    n = 200_003
    row = rng.uniform(0, 2160, n).astype(np.float32)
    col = rng.uniform(0, 3840, n).astype(np.float32)
    x, y, z = c.img2world(_dev(row), _dev(col), 0)
    r64, c64 = oc.world2img_soa(ch, x.cpu().numpy().astype(np.float64), y.cpu().numpy().astype(np.float64),
                                z.cpu().numpy().astype(np.float64))
    err = np.max(np.maximum(np.abs(r64 - row), np.abs(c64 - col)))
    if abs(k) <= 0.9:
        assert err <= TOL32_PX, err          # the stated tolerance, strictly
    else:
        # k = 1.5, 3: no real lens.  The FP32 RESULT FORMAT limits these: an FP32 world coordinate is
        # known to half an ulp, and the forward map multiplies that by its slope 1 + 3 k r^2 (up to 6.6)
        assert err <= TOL32_PX * (1.0 + 3.0 * abs(k) * 0.62), err
    # and the FP64 kernel (whose seed is the same FP32 schedule) stays at 1e-9
    x64, y64, z64 = c.img2world(_dev(row.astype(np.float64)), _dev(col.astype(np.float64)), 0)
    ox, oy, oz = oc.img2world_soa(ch, row.astype(np.float64), col.astype(np.float64))
    scale = max(1.0, float(np.max(np.abs(ox))), float(np.max(np.abs(oy))))
    assert np.max(np.abs(x64.cpu().numpy() - ox)) <= TOL64 * scale


def test_host_entry_points_match_device(cc):
    c = _calib(cc, C2_INTR, [SYN_VIEW])
    rng = np.random.default_rng(3)
    n = (1 << 22) * 2 + 12345     # three pipeline chunks
    row, col = rng.uniform(0, 1080, n), rng.uniform(0, 1920, n)
    hx, hy, hz = c.img2world(row, col, 0)
    dx, dy, dz = c.img2world(_dev(row), _dev(col), 0)
    assert np.array_equal(hx, dx.cpu().numpy()) and np.array_equal(hz, dz.cpu().numpy())
    hr, hc = c.world2img(hx, hy, hz, 0)
    dr, dc = c.world2img(dx, dy, dz, 0)
    assert np.array_equal(hr, dr.cpu().numpy()) and np.array_equal(hc, dc.cpu().numpy())
    # empty input
    e = np.empty(0)
    assert c.img2world(e, e, 0)[0].size == 0


def test_bad_arguments(cc):
    c = _calib(cc, C2_INTR, [SYN_VIEW])
    with pytest.raises(IndexError):
        c.img2world(np.zeros(4), np.zeros(4), 3)          # BoundsError in the reference
    with pytest.raises(IndexError):
        c(np.zeros((1, 2)))                               # no file named *extrinsic*
    c2 = _calib(cc, C2_INTR, [SYN_VIEW, SYN_VIEW], ["a.png", "my_extrinsic.png"])
    assert c2(np.array([[5.0, 6.0]])).shape == (1, 3)     # src/meta.jl:90-93
    with pytest.raises(cc.CamcalError):
        cc.warp(c, 0, np.zeros((1, 8, 8), np.float32), -1.0, (0, 0))
    f = torch.zeros((1, 8, 8), device="cuda")
    with pytest.raises(cc.CamcalError, match="in place"):
        cc.warp(c, 0, f, 1.0, (0, 0), out=f)              # rectification is out of place


# ------------------------------------------------------------------ rectification
def _rect_case(intr, sz, ratio_scale=1.0, view=SYN_VIEW):
    n1, n2 = 20, 14
    ch = oc.chain(intr, *view)
    a, b = np.meshgrid(np.arange(n1, dtype=np.float64), np.arange(n2, dtype=np.float64), indexing="ij")
    x, y = (a * intr[5]).ravel(), (b * intr[5]).ravel()
    row, col = oc.world2img_soa(ch, x, y)
    ip = np.stack([row, col], axis=-1).reshape(n1, n2, 2)
    ratio = oc.get_ratio(ip, intr[5]) * ratio_scale
    axs = oc.get_axes(ratio, intr[5], (n1, n2), sz)
    return ch, ip, ratio, axs


@pytest.mark.parametrize("sz", [(1080, 1920), (375, 500), (131, 77), (128, 8), (4, 3)])
def test_rectify_f32c1_bit_exact(cc, sz):
    intr = camera_for(sz)
    ch, ip, ratio, axs = _rect_case(intr, sz)
    c = _calib(cc, intr, [SYN_VIEW])
    assert abs(cc.get_ratio(ip, intr[5]) - ratio) == 0.0
    assert cc.get_axes(ratio, intr[5], (20, 14), sz) == axs
    rng = np.random.default_rng(1234)
    nf = 3 if sz[0] * sz[1] < 1_000_000 else 2
    frames = rng.random((nf, sz[1], sz[0]), dtype=np.float32)
    ref = oc.rectify_f32c1(ch, 1.0 / ratio, axs, frames, fill=np.nan)
    got = cc.warp(c, 0, _dev(frames), ratio, axs).cpu().numpy()
    assert np.array_equal(np.isnan(got), np.isnan(ref))
    ok = ~np.isnan(ref)
    assert np.array_equal(got[ok], ref[ok])               # bit-exact
    # the TMA-staged and the direct gather are the same function
    got_d = cc.warp(c, 0, _dev(frames), ratio, axs, gather="direct").cpu().numpy()
    assert np.array_equal(np.nan_to_num(got_d, nan=-7.0), np.nan_to_num(got, nan=-7.0))
    if sz[0] % 4 == 0:                                    # TMA needs a 16-byte multiple pitch
        got_t = cc.warp(c, 0, _dev(frames), ratio, axs, gather="tma").cpu().numpy()
        assert np.array_equal(np.nan_to_num(got_t, nan=-7.0), np.nan_to_num(got, nan=-7.0))
    else:
        with pytest.raises(cc.CamcalError):
            cc.warp(c, 0, _dev(frames), ratio, axs, gather="tma")
    if sz[1] >= 77:
        assert 0.3 < ok.mean()
    # the map itself: bit-exact source coordinates => bit-exact indices and weights
    mr, mc = cc.rectify_map(c, 0, ratio, axs, sz)
    omr, omc = oc.rectify_map(ch, 1.0 / ratio, axs, sz)
    assert np.array_equal(mr.cpu().numpy(), omr) and np.array_equal(mc.cpu().numpy(), omc)
    # host entry point, explicit fill value
    got_h = cc.warp(c, 0, frames, ratio, axs, fill=-5.0)
    ref_h = oc.rectify_f32c1(ch, 1.0 / ratio, axs, frames, fill=-5.0)
    assert np.array_equal(got_h, ref_h)


@pytest.mark.parametrize("kind", ["tiny", "zeros", "negative", "neg_zero", "inf", "nan", "mixed"])
def test_rectify_f32c1_exact_widening_special_values(cc, kind):
    """The exact kernel widens float taps with an integer multiply (bits * 2^29 read as a double is the
    value * 2^-896, rectify_f32c1.cuh) where every tap of a warp is finite and >= +0, and with F2F
    elsewhere.  Both must be the oracle's FP64 blend bit for bit: denormals, zeros, the smallest and
    largest normals on the integer path; negative values, -0, Inf and NaN on the other, per warp."""
    sz = (640, 360)
    intr = camera_for(sz)
    ch, ip, ratio, axs = _rect_case(intr, sz)
    c = _calib(cc, intr, [SYN_VIEW])
    rng = np.random.default_rng(77)
    frames = rng.random((3, sz[1], sz[0]), dtype=np.float32)
    bits = frames.view(np.uint32)
    pick = lambda p: rng.random(frames.shape) < p
    if kind == "tiny":            # denormals, the smallest normals, values far below 2^-100, FLT_MAX
        m = pick(0.5)
        bits[m] = rng.integers(0, 0x02000000, size=int(m.sum()), dtype=np.uint32)
        bits[pick(0.01)] = 0x7f7fffff
        bits[pick(0.01)] = 1
    elif kind == "zeros":
        frames[pick(0.7)] = 0.0
    elif kind == "negative":      # a negative tap anywhere in a warp's footprint sends that warp to F2F
        frames[0] -= 0.5
        frames[1][pick(1e-4)[1]] = -1.0
    elif kind == "neg_zero":
        bits[pick(0.3)] = 0x80000000
    elif kind == "inf":
        frames[pick(2e-4)] = np.inf
    elif kind == "nan":
        frames[pick(2e-4)] = np.nan
    else:
        bits[...] = rng.integers(0, 2 ** 32, size=frames.shape, dtype=np.uint32)
        bits[0] &= 0x7fffffff     # frame 0 non-negative, a few Inf/NaN by chance
    ref = oc.rectify_f32c1(ch, 1.0 / ratio, axs, frames, fill=-3.0)
    for gather in ("auto", "direct"):
        got = cc.warp(c, 0, _dev(frames), ratio, axs, fill=-3.0, gather=gather).cpu().numpy()
        assert np.array_equal(np.isnan(got), np.isnan(ref))
        ok = ~np.isnan(ref)
        assert np.array_equal(got[ok].view(np.uint32), ref[ok].view(np.uint32)), (kind, gather)   # bits: -0 vs +0 too


@pytest.mark.parametrize("sz", [(2160, 3840), (1080, 1920), (360, 640), (131, 77), (16, 5)])
def test_rectify_u8c3_bit_exact(cc, sz):
    intr = camera_for(sz)
    ch, ip, ratio, axs = _rect_case(intr, sz)
    c = _calib(cc, intr, [SYN_VIEW])
    rng = np.random.default_rng(4321)
    nf = 2 if sz[0] * sz[1] < 1_000_000 else 1
    frames = rng.integers(0, 256, (nf, sz[1], sz[0], 3), dtype=np.uint8)
    ref = oc.rectify_u8c3(ch, 1.0 / ratio, axs, frames, fill=(1, 2, 3))
    got = cc.warp(c, 0, _dev(frames), ratio, axs, fill=(1, 2, 3)).cpu().numpy()
    assert np.array_equal(got, ref)
    got_d = cc.warp(c, 0, _dev(frames), ratio, axs, fill=(1, 2, 3), gather="direct").cpu().numpy()
    assert np.array_equal(got_d, ref)
    if sz[0] % 16 == 0:
        got_t = cc.warp(c, 0, _dev(frames), ratio, axs, fill=(1, 2, 3), gather="tma").cpu().numpy()
        assert np.array_equal(got_t, ref)
    got_h = cc.warp(c, 0, frames, ratio, axs, fill=(1, 2, 3))
    assert np.array_equal(got_h, ref)


@pytest.mark.parametrize("rz", [0.3, -0.3, 0.04, -0.04, 0.9, -0.7])
@pytest.mark.parametrize("ratio_scale", [1.0, 0.8, 1.25])
def test_rectify_u8c3_staged_rotations_and_scales(cc, rz, ratio_scale):
    """The u8 box origin is a BYTE offset (multiple of 16) and the staged line pitch depends on which way the
    source line changes along a warp (RectPlan.tilt): both rotation directions, small and large angles,
    magnifying and shrinking ratios, through the forced TMA path; exact = bit-equal, fast = +-1 LSB."""
    sz = (368, 250)                                     # 368 * 3 bytes is a multiple of 16
    intr = camera_for(sz)
    view = ((0.15, -0.1, rz), (-8.0, -12.0, 30.0))
    ch, ip, ratio, axs = _rect_case(intr, sz, ratio_scale=ratio_scale, view=view)
    c = _calib(cc, intr, [view])
    rng = np.random.default_rng(77)
    frames = rng.integers(0, 256, (3, sz[1], sz[0], 3), dtype=np.uint8)
    ref = oc.rectify_u8c3(ch, 1.0 / ratio, axs, frames, fill=(9, 8, 7))
    try:
        got = cc.warp(c, 0, _dev(frames), ratio, axs, fill=(9, 8, 7), gather="tma").cpu().numpy()
    except cc.CamcalError:                              # footprint too large to stage at this angle: the direct path serves it
        got = cc.warp(c, 0, _dev(frames), ratio, axs, fill=(9, 8, 7)).cpu().numpy()
    assert np.array_equal(got, ref)
    fast = cc.warp(c, 0, _dev(frames), ratio, axs, fill=(9, 8, 7), coord="f32").cpu().numpy()
    inb = np.any(ref != np.array((9, 8, 7), dtype=np.uint8), axis=-1)
    # the FP32 map may move a sample across the frame edge: compare where both sampled
    both = inb & np.any(fast != np.array((9, 8, 7), dtype=np.uint8), axis=-1)
    assert both.mean() > 0.02
    d = np.abs(fast[both].astype(np.int16) - ref[both].astype(np.int16))
    assert d.max() <= 2 and (d > 1).mean() < 1e-3       # +-1 LSB; a 1e-3 px map error on white noise can add one more, rarely
    assert (inb != np.any(fast != np.array((9, 8, 7), dtype=np.uint8), axis=-1)).mean() < 2e-3


def test_rectify_tilted_views_staged_and_fallback(cc, example_fit):
    """The reference's own example views are tilted up to 0.8 rad: tile footprints reach 75 x 75
    texels, some exceed the staged box -> those pixels take the direct path inside the TMA
    kernel.  Every view, both pixel formats, both coordinate modes' fill decisions."""
    intr = example_fit["intr_tuple"]
    n1, n2 = example_fit["n_corners"]
    sz = (376, 500)                                    # 376: 16-byte multiple pitch for fp32
    c = _calib(cc, intr, example_fit["view_list"], example_fit["files"])
    rng = np.random.default_rng(11)
    frames = rng.random((2, sz[1], sz[0]), dtype=np.float32)
    for vi, (rv, tv) in enumerate(example_fit["view_list"]):
        ip = example_fit["corners_np"][vi].reshape(n2, n1, 2).transpose(1, 0, 2)
        ratio, axs = cc.image_transformations(c, vi, [example_fit["corners_np"][i].reshape(n2, n1, 2).transpose(1, 0, 2) for i in range(6)], 1.0, (n1, n2), sz)
        assert ratio == oc.get_ratio(ip, 1.0)
        ch = oc.chain(intr, rv, tv)
        ref = oc.rectify_f32c1(ch, 1.0 / ratio, axs, frames, fill=-2.0)
        for gather in ("auto", "direct"):
            got = cc.warp(c, vi, _dev(frames), ratio, axs, fill=-2.0, gather=gather).cpu().numpy()
            assert np.array_equal(got, ref), (vi, gather)
        assert (ref != -2.0).mean() > 0.2


def test_rectify_views_is_the_plot_loop(cc, example_fit):
    """cc_rectify_*_views: the six example images, each with ITS OWN extrinsic, ratio and axes
    (src/plot_calibration.jl:36-42), in one call; two frames per view; both pixel formats."""
    intr = example_fit["intr_tuple"]
    n1, n2 = example_fit["n_corners"]
    sz = (376, 500)
    c = _calib(cc, intr, example_fit["view_list"], example_fit["files"])
    rng = np.random.default_rng(12)
    nv, k = len(example_fit["view_list"]), 2
    frames = rng.random((nv * k, sz[1], sz[0]), dtype=np.float32)
    f8 = rng.integers(0, 256, (nv * k, sz[1], sz[0], 3), dtype=np.uint8)
    ratios, axss = [], []
    for vi in range(nv):
        r, a = cc.image_transformations(c, vi, example_fit["corners_np"], 1.0, (n1, n2), sz)   # detect_fit's flat layout
        ratios.append(r); axss.append(a)
    got = cc.warp_views(c, example_fit["files"], _dev(frames), ratios, axss, fill=-2.0).cpu().numpy()
    got8 = cc.warp_views(c, list(range(nv)), _dev(f8), ratios, axss, fill=(3, 2, 1)).cpu().numpy()
    for vi, (rv, tv) in enumerate(example_fit["view_list"]):
        ch = oc.chain(intr, rv, tv)
        sl = slice(vi * k, (vi + 1) * k)
        assert np.array_equal(got[sl], oc.rectify_f32c1(ch, 1.0 / ratios[vi], axss[vi], frames[sl], fill=-2.0)), vi
        assert np.array_equal(got8[sl], oc.rectify_u8c3(ch, 1.0 / ratios[vi], axss[vi], f8[sl], fill=(3, 2, 1))), vi
    with pytest.raises(ValueError):
        cc.warp_views(c, [0, 1, 2, 3], _dev(frames[:6]), ratios[:4], axss[:4])            # 6 frames, 4 views


def _perturbed_views(n):
    return [((BENCH_VIEW[0][0] + 0.004 * i, BENCH_VIEW[0][1] - 0.003 * i, BENCH_VIEW[0][2] + 0.002 * i),
             (BENCH_VIEW[1][0] + 0.03 * i, BENCH_VIEW[1][1] - 0.02 * i, BENCH_VIEW[1][2] + 0.1 * i)) for i in range(n)]


@pytest.mark.parametrize("nv,k,sz", [(5, 1, (384, 200)), (3, 5, (256, 131)), (70, 2, (128, 96))])
def test_rectify_views_one_launch_per_group(cc, nv, k, sz):
    """cc_rectify_*_views rectifies groups of up to 64 views in ONE launch (rectify_*_views_kernel: view
    table in the kernel's parameter space, common staged box, per-view tile headers).  Bit-equal to one
    launch per view (CAMCAL_VIEWS_SINGLE=0) in all four variants, and to the oracle for the exact ones;
    70 views = a group of 64 and a group of 6; k frames per view share the view's map."""
    import os
    intr = camera_for(sz)
    views = _perturbed_views(nv)
    if nv == 5:
        views[3] = views[1]                                # the same view twice in a group: planned once
    c = _calib(cc, intr, views)
    rng = np.random.default_rng(100 + nv)
    frames = rng.random((nv * k, sz[1], sz[0]), dtype=np.float32)
    f8 = rng.integers(0, 256, (nv * k, sz[1], sz[0], 3), dtype=np.uint8)
    ratios, axss = [], []
    for vi in range(nv):
        si = 1 if (nv == 5 and vi == 3) else vi % 5
        _, _, ratio, axs = _rect_case(intr, sz, ratio_scale=1.0 + 0.01 * si, view=views[vi])
        ratios.append(ratio); axss.append(axs)
    idx = list(range(nv))
    dfr, df8 = _dev(frames), _dev(f8)
    got = {}
    ctx = cc.context(0)
    for single in ("1", "0"):
        os.environ["CAMCAL_VIEWS_SINGLE"] = single
        try:
            for coord in ("f64", "f32"):
                n0 = ctx.launch_count()
                got[(single, coord, "f")] = cc.warp_views(c, idx, dfr, ratios, axss, fill=-2.0, coord=coord).cpu().numpy()
                got[(single, coord, "u")] = cc.warp_views(c, idx, df8, ratios, axss, fill=(3, 2, 1), coord=coord).cpu().numpy()
                # one launch per group of <= 64 views and pixel format, against one per view
                assert ctx.launch_count() - n0 == (2 * ((nv + 63) // 64) if single == "1" else 2 * nv), (single, coord)
        finally:
            os.environ.pop("CAMCAL_VIEWS_SINGLE", None)
    for coord in ("f64", "f32"):
        for px in ("f", "u"):
            assert np.array_equal(got[("1", coord, px)], got[("0", coord, px)]), (coord, px)
    for vi in sorted(set([0, nv // 2, nv - 1])):
        ch = oc.chain(intr, *views[vi])
        sl = slice(vi * k, (vi + 1) * k)
        ref = oc.rectify_f32c1(ch, 1.0 / ratios[vi], axss[vi], frames[sl], fill=-2.0)
        assert np.array_equal(got[("1", "f64", "f")][sl], ref), vi
        assert (ref != -2.0).mean() > 0.5
        assert np.array_equal(got[("1", "f64", "u")][sl], oc.rectify_u8c3(ch, 1.0 / ratios[vi], axss[vi], f8[sl], fill=(3, 2, 1))), vi


def test_rectify_bounds_checked_build(cc):
    """The rectification parity tests once more against libcamcal_b200_chk.so, the build of the same
    sources with -DCAMCAL_CHECK_BOUNDS: every shared-memory tap address of the staged kernels is
    range-checked on the device and a violation traps (the substitute for compute-sanitizer, which
    is closed on this pool).  Runs in a child process: the library is chosen at import time."""
    import os
    import subprocess
    import sys
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    lib = os.path.join(root, "cameracalibrations_b200", "libcamcal_b200_chk.so")
    if not os.path.exists(lib):
        pytest.skip("libcamcal_b200_chk.so not built (make -C cameracalibrations_b200/csrc chk)")
    if os.environ.get("CAMCAL_B200_LIB"):
        pytest.skip("already running against a variant library")
    env = dict(os.environ, CAMCAL_B200_LIB=lib)
    # "batching" selects all of test_gpu_batching.py: frame groups, pair kernels, views with several groups per view
    r = subprocess.run([sys.executable, "-m", "pytest", os.path.join(root, "tests", "test_gpu_parity.py"),
                        os.path.join(root, "tests", "test_gpu_batching.py"), "-x", "-q", "-m", "gpu",
                        "-k", "bit_exact or tilted or horizon or views_is or views_one_launch or alternating or strided or batching"],
                       env=env, capture_output=True, text=True, timeout=900)
    assert r.returncode == 0, r.stdout[-3000:] + r.stderr[-2000:]
    assert " passed" in r.stdout


def test_rectify_edge_rule(cc):
    """x == n in bounds with (i, delta) = (n-1, 1); just outside -> fill; exact grid hits."""
    intr = (1.0, 1.0, 0.0, 0.0, 0.0, 1.0)
    view = ((0.0, 0.0, 0.0), (0.0, 0.0, 1.0))
    c = _calib(cc, intr, [view])
    img = np.arange(12, dtype=np.float32).reshape(1, 3, 4)
    assert np.array_equal(cc.warp(c, 0, _dev(img), 1.0, (1, 1), fill=-1.0).cpu().numpy(), img)
    out = cc.warp(c, 0, _dev(img), 1.0, (0, 1), fill=-1.0).cpu().numpy()[0]
    assert np.all(out[:, 0] == -1.0) and np.array_equal(out[:, 1:], img[0][:, :3])
    out = cc.warp(c, 0, _dev(img), 2.0, (2, 2), fill=-1.0).cpu().numpy()[0]
    assert out[0, 0] == img[0, 0, 0] and out[0, 1] == 0.5 * (img[0, 0, 0] + img[0, 0, 1])


def test_rectify_u8c3_exact_ties_take_the_fp64_blend(cc):
    """The exact u8 kernel blends in FP32 and certifies the rounding; values within 6.5e-5 of a
    rounding boundary are re-blended in FP64.  Half-integer sample positions make every weight
    exactly 0.5, so a large share of the blended values are exact .5 / .25 / .75 ties or
    near-ties: the output must still be the oracle's (round-half-even of the FP64 blend)."""
    intr = (1.0, 1.0, 0.0, 0.0, 0.0, 1.0)
    view = ((0.0, 0.0, 0.0), (0.0, 0.0, 1.0))
    c = _calib(cc, intr, [view])
    ch = oc.chain(intr, *view)
    rng = np.random.default_rng(21)
    sz = (256, 192)                                    # 256 * 3 bytes: TMA-addressable pitch
    f8 = rng.integers(0, 256, (2, sz[1], sz[0], 3), dtype=np.uint8)
    for ratio, axs in ((2.0, (2, 2)), (2.0, (3, 2)), (4.0, (5, 7)), (1.0, (1, 1))):
        ref = oc.rectify_u8c3(ch, 1.0 / ratio, axs, f8, fill=(9, 8, 7))
        for gather in ("tma", "direct"):
            got = cc.warp(c, 0, _dev(f8), ratio, axs, fill=(9, 8, 7), gather=gather).cpu().numpy()
            assert np.array_equal(got, ref), (ratio, axs, gather)
        assert (ref != np.array([9, 8, 7], dtype=np.uint8)).any()


def _plan_cache_cases(cc):
    """67 parameter sets of one 128 x 96 camera, more than the context caches one-view plans for (64): the
    calibration, (view, chain, ratio, axes) per set, two frames on the device and the oracle's results"""
    sz = (128, 96)
    intr = camera_for(sz)
    rng = np.random.default_rng(3)
    frames = rng.random((2, sz[1], sz[0]), dtype=np.float32)
    cases = []
    for i in range(67):
        view = ((0.05 + 0.004 * i, -0.04, 0.02 * (i % 3)), (-9.3 + 0.05 * i, -6.4, 30.0 + 0.3 * i))
        ch, ip, ratio, axs = _rect_case(intr, sz, view=view)
        cases.append((view, ch, ratio, axs))
    c = _calib(cc, intr, [v for v, _, _, _ in cases])
    refs = [oc.rectify_f32c1(ch, 1.0 / ratio, axs, frames, fill=-3.0) for _, ch, ratio, axs in cases]
    return c, cases, _dev(frames), refs


def test_rectify_plan_cache_many_parameter_sets(cc):
    """More parameter sets than the context caches tile plans for (64), revisited in a different
    order and on two streams: every call must match the oracle (plans are keyed by calibration,
    ratio, axes and frame geometry; an evicted plan is rebuilt)."""
    c, cases, fd, refs = _plan_cache_cases(cc)
    N = len(cases)
    side = torch.cuda.Stream()
    side.wait_stream(torch.cuda.current_stream())
    for order in (range(N), reversed(range(N)), (0, 5, 0, N - 1, 5, 0)):
        for i in order:
            _, ch, ratio, axs = cases[i]
            got = cc.warp(c, i, fd, ratio, axs, fill=-3.0).cpu().numpy()
            assert np.array_equal(got, refs[i]), i
            with torch.cuda.stream(side):
                got2 = cc.warp(c, i, fd, ratio, axs, fill=-3.0, coord="f64")
            side.synchronize()
            assert np.array_equal(got2.cpu().numpy(), refs[i]), i


def test_rectify_plan_cache_unsynchronised_streams(cc):
    """The same 67 parameter sets in the same three orders, the calls alternating between two streams with no
    synchronisation until the end: plans are evicted and rebuilt while launches on the other stream may still
    read them.  Every output must match the oracle."""
    c, cases, fd, refs = _plan_cache_cases(cc)
    N = len(cases)
    streams = (torch.cuda.current_stream(), torch.cuda.Stream())
    streams[1].wait_stream(streams[0])
    outs = []
    for order in (range(N), reversed(range(N)), (0, 5, 0, N - 1, 5, 0)):
        for j, i in enumerate(order):
            _, ch, ratio, axs = cases[i]
            with torch.cuda.stream(streams[j % 2]):
                outs.append((i, cc.warp(c, i, fd, ratio, axs, fill=-3.0)))
    torch.cuda.synchronize()
    for i, out in outs:
        assert np.array_equal(out.cpu().numpy(), refs[i]), i


def test_rectify_alternating_large_and_small_boxes(cc):
    """A plan whose staged ring needs more than the 48 KB default of dynamic shared memory, then one
    that does not, then the first again from the plan cache: the kernel's shared-memory limit must
    only ever be raised (it belongs to the kernel, not to the plan).  Both pixel formats."""
    sz = (512, 384)
    intr = camera_for(sz)
    rng = np.random.default_rng(17)
    frames = rng.random((2, sz[1], sz[0]), dtype=np.float32)
    f8 = rng.integers(0, 256, (2, sz[1], sz[0], 3), dtype=np.uint8)
    c = _calib(cc, intr, [SYN_VIEW])
    cases = [_rect_case(intr, sz, ratio_scale=s) for s in (0.42, 1.0)]
    refs = [(oc.rectify_f32c1(ch, 1.0 / ratio, axs, frames, fill=-4.0), oc.rectify_u8c3(ch, 1.0 / ratio, axs, f8))
            for ch, _, ratio, axs in cases]
    for i in (0, 1, 0, 1, 0):
        _, _, ratio, axs = cases[i]
        for coord in ("f64", "f32"):
            got = cc.warp(c, 0, _dev(frames), ratio, axs, fill=-4.0, gather="tma", coord=coord).cpu().numpy()
            got8 = cc.warp(c, 0, _dev(f8), ratio, axs, coord=coord).cpu().numpy()   # (a u8 box is capped at 256 B per line)
            if coord == "f64":
                assert np.array_equal(got, refs[i][0]), i
                assert np.array_equal(got8, refs[i][1]), i


@pytest.mark.parametrize("pad1,padf", [(4, 64), (3, 7), (0, 16)])
def test_rectify_strided_layouts_through_the_abi(cc, pad1, padf):
    """pitch > sz1 and frame_stride > pitch * sz2 (the C ABI's layout parameters; the Python warp()
    always passes dense arrays): TMA-addressable strides (pad 4 px / 64 px) and odd ones (direct
    kernels).  The valid region equals the dense oracle result, the padding is never written."""
    from cameracalibrations_b200 import _lib
    sz = (128, 96)
    intr = camera_for(sz)
    ch, ip, ratio, axs = _rect_case(intr, sz)
    c = _calib(cc, intr, [SYN_VIEW])
    nf, pitch = 3, sz[0] + pad1
    stride = pitch * sz[1] + padf
    rng = np.random.default_rng(8)
    axs_c = (C.c_int64 * 2)(*axs)
    h = _lib.context(0).handle
    ci, cv = C.byref(c._intr), C.byref(c._views[0])
    # fp32 gray
    dense = rng.random((nf, sz[1], sz[0]), dtype=np.float32)
    ref = oc.rectify_f32c1(ch, 1.0 / ratio, axs, dense, fill=-4.0)
    buf = np.full(nf * stride, 777.0, np.float32)
    for f in range(nf):
        buf[f * stride: f * stride + pitch * sz[1]].reshape(sz[1], pitch)[:, :sz[0]] = dense[f]
    for coord in (_lib.COORD_F64,):
        src, dst = _dev(buf), _dev(np.full(nf * stride, 555.0, np.float32))
        _lib.check(_lib.lib.cc_rectify_f32c1(h, ci, cv, float(ratio), axs_c, C.c_void_p(src.data_ptr()),
                                             C.c_void_p(dst.data_ptr()), sz[0], sz[1], C.c_size_t(pitch),
                                             C.c_size_t(stride), nf, C.c_float(-4.0), coord, None))
        torch.cuda.synchronize()
        out = dst.cpu().numpy()
        seen = np.zeros(out.shape, bool)
        for f in range(nf):
            v = out[f * stride: f * stride + pitch * sz[1]].reshape(sz[1], pitch)
            assert np.array_equal(v[:, :sz[0]], ref[f])
            seen[f * stride: f * stride + pitch * sz[1]].reshape(sz[1], pitch)[:, :sz[0]] = True
        assert np.all(out[~seen] == 555.0)
    # u8 RGB
    d8 = rng.integers(0, 256, (nf, sz[1], sz[0], 3), dtype=np.uint8)
    ref8 = oc.rectify_u8c3(ch, 1.0 / ratio, axs, d8, fill=(1, 2, 3))
    b8 = np.full(nf * stride * 3, 77, np.uint8)
    for f in range(nf):
        b8[f * stride * 3: (f * stride + pitch * sz[1]) * 3].reshape(sz[1], pitch, 3)[:, :sz[0]] = d8[f]
    src, dst = _dev(b8), _dev(np.full(nf * stride * 3, 55, np.uint8))
    fill = (C.c_uint8 * 3)(1, 2, 3)
    _lib.check(_lib.lib.cc_rectify_u8c3(h, ci, cv, float(ratio), axs_c, C.c_void_p(src.data_ptr()),
                                        C.c_void_p(dst.data_ptr()), sz[0], sz[1], C.c_size_t(pitch),
                                        C.c_size_t(stride), nf, fill, _lib.COORD_F64, None))
    torch.cuda.synchronize()
    out = dst.cpu().numpy()
    seen = np.zeros(out.shape, bool)
    for f in range(nf):
        v = out[f * stride * 3: (f * stride + pitch * sz[1]) * 3].reshape(sz[1], pitch, 3)
        assert np.array_equal(v[:, :sz[0]], ref8[f])
        seen[f * stride * 3: (f * stride + pitch * sz[1]) * 3].reshape(sz[1], pitch, 3)[:, :sz[0]] = True
    assert np.all(out[~seen] == 55)


def test_rectify_view_with_a_horizon(cc):
    """A steeply tilted board: part of the output plane lies behind the camera, so P3 changes sign
    inside the frame (tiles the plan marks as unusable for the branch-free reciprocal), coordinates
    run through +-inf, and most pixels are fill.  Every kernel variant equals the oracle."""
    sz = (256, 192)
    intr = camera_for(sz)
    view = ((1.45, 0.1, 0.0), (-3.0, -2.0, 2.0))
    c = _calib(cc, intr, [view])
    ch = oc.chain(intr, *view)
    rng = np.random.default_rng(2)
    frames = rng.random((2, sz[1], sz[0]), dtype=np.float32)
    f8 = rng.integers(0, 256, (2, sz[1], sz[0], 3), dtype=np.uint8)
    for ratio, axs in ((6.0, (-40, -30)), (1.5, (-200, -400))):
        ref = oc.rectify_f32c1(ch, 1.0 / ratio, axs, frames, fill=-9.0)
        ref8 = oc.rectify_u8c3(ch, 1.0 / ratio, axs, f8, fill=(4, 5, 6))
        for gather in ("auto", "direct"):
            got = cc.warp(c, 0, _dev(frames), ratio, axs, fill=-9.0, gather=gather).cpu().numpy()
            assert np.array_equal(got, ref), (ratio, gather)
            got8 = cc.warp(c, 0, _dev(f8), ratio, axs, fill=(4, 5, 6), gather=gather).cpu().numpy()
            assert np.array_equal(got8, ref8), (ratio, gather)
        # the fast path may differ near the horizon only: where the FP64 map is inside the frame
        # by a margin it samples, elsewhere it fills
        gotf = cc.warp(c, 0, _dev(frames), ratio, axs, fill=-9.0, coord="f32").cpu().numpy()
        omr, omc = oc.rectify_map(ch, 1.0 / ratio, axs, sz)
        far_out = ~((omr > -50) & (omr < sz[0] + 50) & (omc > -50) & (omc < sz[1] + 50))
        assert np.all(gotf[0][far_out & np.isfinite(omr)] == -9.0)
    assert 0.01 < (ref != -9.0).mean() < 0.99


@pytest.mark.parametrize("intr,sz", [(C2_INTR, (1080, 1920)), (C3_INTR, (2160, 3840))])
def test_rectify_f32_coords_within_1e3_px(cc, intr, sz):
    """FP32 fast path: warp a row-ramp and a column-ramp; bilinear interpolation reproduces a
    ramp exactly, so the outputs ARE the FP32 map; compare with the FP64 oracle map."""
    ch, ip, ratio, axs = _rect_case(intr, sz)
    c = _calib(cc, intr, [SYN_VIEW])
    r = np.arange(1, sz[0] + 1, dtype=np.float32)
    q = np.arange(1, sz[1] + 1, dtype=np.float32)
    frames = np.stack([np.broadcast_to(r[None, :], (sz[1], sz[0])),
                       np.broadcast_to(q[:, None], (sz[1], sz[0]))]).astype(np.float32)
    got = cc.warp(c, 0, _dev(frames), ratio, axs, coord="f32").cpu().numpy().astype(np.float64)
    omr, omc = oc.rectify_map(ch, 1.0 / ratio, axs, sz)
    inb = (omr >= 1.001) & (omr <= sz[0] - 0.001) & (omc >= 1.001) & (omc <= sz[1] - 0.001)
    assert not np.any(np.isnan(got[0][inb]))
    # the FP32 map itself (cc_rectify_map_f32: the arithmetic of the fast kernels): strictly within 1e-3 px
    fr, fc = cc.rectify_map(c, 0, ratio, axs, sz, coord="f32")
    assert np.max(np.abs(fr.cpu().numpy().astype(np.float64)[inb] - omr[inb])) <= TOL32_PX
    assert np.max(np.abs(fc.cpu().numpy().astype(np.float64)[inb] - omc[inb])) <= TOL32_PX
    # and the warped ramps ARE that map up to the FP32 rounding of the blend (ulp(4096) = 4.9e-4)
    assert np.max(np.abs(got[0][inb] - fr.cpu().numpy().astype(np.float64)[inb])) <= 5e-4
    assert np.max(np.abs(got[1][inb] - fc.cpu().numpy().astype(np.float64)[inb])) <= 5e-4
    # fill decisions differ only within 1e-3 px of the frame border
    edge = ~inb & ~((omr < 0.999) | (omr > sz[0] + 0.001) | (omc < 0.999) | (omc > sz[1] + 0.001))
    outside = ~inb & ~edge
    assert np.all(np.isnan(got[0][outside]))
    # u8 fast path: at most 1 LSB away from the FP64 result, and rarely
    rng = np.random.default_rng(5)
    f8 = rng.integers(0, 256, (1, sz[1], sz[0], 3), dtype=np.uint8)
    # smooth image so that a 1e-3 px shift cannot move a value by more than 1 LSB
    f8 = (np.add.outer(np.arange(sz[1]) // 7, np.arange(sz[0]) // 5) % 256).astype(np.uint8)[None, :, :, None].repeat(3, -1)
    a = cc.warp(c, 0, _dev(f8), ratio, axs, coord="f32").cpu().numpy().astype(np.int16)
    b = oc.rectify_u8c3(ch, 1.0 / ratio, axs, f8).astype(np.int16)
    diff = np.abs(a - b)[0][inb]
    assert diff.max() <= 1 and (diff > 0).mean() < 5e-3


def test_rectify_batch_frames_independent(cc):
    """Size-independent property at BASELINE config 2 size: every frame of a batch is
    processed identically (equal inputs -> bitwise equal outputs), strided layouts work."""
    sz = (1080, 1920)
    ch, ip, ratio, axs = _rect_case(C2_INTR, sz, view=BENCH_VIEW)
    c = _calib(cc, C2_INTR, [BENCH_VIEW])
    g = torch.Generator(device="cuda").manual_seed(1234)
    one = torch.rand((1, sz[1], sz[0]), device="cuda", generator=g)
    batch = one.repeat(8, 1, 1).contiguous()
    out = cc.warp(c, 0, batch, ratio, axs)
    assert all(torch.equal(torch.nan_to_num(out[0], nan=-1.0), torch.nan_to_num(out[i], nan=-1.0))
               for i in range(1, 8))
    ref = oc.rectify_f32c1(ch, 1.0 / ratio, axs, one.cpu().numpy(), fill=-1.0)
    assert np.array_equal(torch.nan_to_num(out[3], nan=-1.0).cpu().numpy(), ref[0])
    assert (ref[0] != -1.0).mean() > 0.99      # SURVEY 8(d): >= 99 % of output pixels sample in-bounds


# ------------------------------------------------------------------ residual / Jacobian
def _c5_case(nviews, seed=7):
    rng = np.random.default_rng(seed)
    n1, n2 = 20, 14
    intr = C3_INTR
    obj = np.array([[a, b, 0.0] for b in range(n2) for a in range(n1)], dtype=np.float64)
    rv = rng.normal(0, 0.3, (nviews, 3))
    tv = np.array([-10.0, -7.0, 40.0]) + rng.normal(0, 2.0, (nviews, 3))
    views = [(rv[i], tv[i]) for i in range(nviews)]
    img = np.empty((nviews, n1 * n2, 2))
    for i in range(nviews):
        r, q = oc.world2img(oc.chain(intr, rv[i], tv[i]), obj)
        img[i, :, 0], img[i, :, 1] = r, q
    img += rng.normal(0, 0.25, img.shape)
    return intr, views, np.concatenate([rv, tv], axis=1), obj, img, (n1, n2)


def _relerr(a, b):
    return np.max(np.abs(a - b) / (1.0 + np.abs(b)))


def test_reproj_jtj_vs_oracle(cc):
    intr, views, vt, obj, img, _ = _c5_case(257)
    pv_o, sh_o, _ = oc.reproj_jtj(intr, 1.0, views, obj, img)
    pv, sh = cc.reproj_jtj(intr, 1.0, _dev(vt), _dev(obj), _dev(img))
    assert _relerr(pv.cpu().numpy(), pv_o) <= TOL64
    assert _relerr(sh.cpu().numpy(), sh_o) <= TOL64
    # bit-reproducible (fixed reduction order)
    pv2, sh2 = cc.reproj_jtj(intr, 1.0, _dev(vt), _dev(obj), _dev(img))
    assert torch.equal(pv, pv2) and torch.equal(sh, sh2)
    # host entry point
    pv_h, sh_h = cc.reproj_jtj(intr, 1.0, vt, obj, img)
    assert np.array_equal(pv_h, pv.cpu().numpy()) and np.array_equal(sh_h, sh.cpu().numpy())
    # aspect != 1 and checker_size != 1
    intr2 = (intr[0] * 1.1,) + intr[1:5] + (2.5,)
    pv_o, sh_o, _ = oc.reproj_jtj(intr2, 1.1, views[:5], obj * 2.5, img[:5])
    pv, sh = cc.reproj_jtj(intr2, 1.1, vt[:5], obj * 2.5, img[:5])
    assert _relerr(pv, pv_o) <= TOL64 and _relerr(sh, sh_o) <= TOL64


def test_reproj_jtj_vs_cv2_golden(cc, example_fit):
    """J'J assembled from cv2.projectPoints' own Jacobian (tests/golden/project_points.json)."""
    g = load_golden("project_points.json")
    obj, img = example_fit["obj_np"], example_fit["corners_np"]
    vt = np.array([list(r) + list(t) for r, t in example_fit["view_list"]])
    pv, sh = cc.reproj_jtj(example_fit["intr_tuple"], 1.0, vt, obj, img)
    tot = 0.0
    for vi, gg in enumerate(g["example"]):
        J = np.asarray(gg["jac"]).reshape(-1, 10)
        r = (np.asarray(gg["pix"]) - img[vi]).reshape(-1)
        JtJ = J.T @ J
        assert _relerr(pv[vi, :36].reshape(6, 6), JtJ[:6, :6]) < 1e-8
        assert _relerr(pv[vi, 36:60].reshape(6, 4), JtJ[:6, 6:]) < 1e-8
        assert _relerr(pv[vi, 60:66], J[:, :6].T @ r) < 1e-8
        tot += r @ r
    assert abs(sh[20] - tot) < 1e-8
    n = img.shape[0] * img.shape[1]
    assert abs(np.sqrt(sh[20] / n) - example_fit["cv2_rms"]) < 1e-6


def test_reproj_zero_theta_and_empty(cc):
    intr, views, vt, obj, img, _ = _c5_case(3)
    vt[0, :3] = 0.0
    views[0] = (np.zeros(3), views[0][1])
    pv_o, sh_o, _ = oc.reproj_jtj(intr, 1.0, views, obj, img)
    pv, sh = cc.reproj_jtj(intr, 1.0, vt, obj, img)
    assert _relerr(pv, pv_o) <= TOL64 and _relerr(sh, sh_o) <= TOL64
    pv, sh = cc.reproj_jtj(intr, 1.0, vt[:0], obj, img[:0])
    assert pv.shape == (0, 66) and np.all(sh == 0.0)


def test_calculate_errors_matches_reference_bounds(cc, example_fit):
    """test/runtests.jl:73-77 through the CUDA path, and equality with the oracle."""
    c = _calib(cc, example_fit["intr_tuple"], example_fit["view_list"], example_fit["files"])
    rng = np.random.default_rng(1)
    eps = cc.calculate_errors(c, example_fit["corners_np"], example_fit["obj_np"], 1.0, example_fit["sz"],
                              example_fit["files"], example_fit["n_corners"], 100, rng=rng)
    assert eps["n"] == 6
    assert all(eps[k] < 1 for k in ("reprojection", "projection", "distance", "inverse"))
    rng = np.random.default_rng(1)
    sz = np.asarray(example_fit["sz"], dtype=np.float64)
    samples = rng.random((6, 100, 2)) * (sz - 1) + 1
    ref = oc.calculate_errors(example_fit["intr_tuple"], example_fit["view_list"], example_fit["obj_np"],
                              example_fit["corners_np"], example_fit["n_corners"], samples)
    for k, r in zip(("reprojection", "projection", "distance"), ref[:3]):
        assert abs(eps[k] - r) <= 1e-9
    assert eps["inverse"] < 1e-10 and ref[3] < 1e-10
    # the host form of the ABI (numpy in, four raw sums out) is the same kernel behind copies
    import ctypes as C
    from cameracalibrations_b200 import _lib
    n1, n2 = example_fit["n_corners"]
    views = np.ascontiguousarray([list(r) + list(t) for r, t in example_fit["view_list"]], dtype=np.float64)
    obj = np.ascontiguousarray(example_fit["obj_np"], dtype=np.float64).reshape(-1, 3)
    img = np.ascontiguousarray(example_fit["corners_np"], dtype=np.float64).reshape(6, -1, 2)
    ir, ic = np.ascontiguousarray(samples[:, :, 0]), np.ascontiguousarray(samples[:, :, 1])
    sums = np.zeros(4)
    p = lambda a: C.c_void_p(a.ctypes.data)
    _lib.check(_lib.lib.cc_calculate_errors_f64_host(_lib.context(0).handle, C.byref(c._intr), p(views), 6, p(obj), p(img),
                                                     n1, n2, p(ir), p(ic), 100, p(sums)))
    n = n1 * n2 * 6
    assert abs(np.sqrt(sums[0] / n) - eps["reprojection"]) < 1e-12 and abs(np.sqrt(sums[1] / n) - eps["projection"]) < 1e-12
    assert abs(np.sqrt(sums[2] / ((n1 - 1) * (n2 - 1)) / 6) - eps["distance"]) < 1e-12


def test_save_load_round_trip(cc, tmp_path, example_fit):
    """test/runtests.jl:88-98 (files preserved) -- plus the numbers, which the reference leaves unpinned."""
    c = _calib(cc, example_fit["intr_tuple"], example_fit["view_list"], example_fit["files"])
    f = tmp_path / "calibration.json"
    cc.save(f, c)
    c2 = cc.load(f)
    assert c2.files == c.files and c2.intrinsic == c.intrinsic and c2.k == c.k
    assert c2.extrinsics == c.extrinsics and c2.scale == c.scale
    p = np.array([[10.0, 20.0], [300.0, 400.0]])
    assert np.array_equal(c(p, 2), c2(p, 2))


# ------------------------------------------------------------------ ingest (SURVEY 8f rank 4)
def test_jpeg_ingest_feeds_the_plot_loop(cc, example_fit):
    """src/plot_calibration.jl:36-42 on the device: compressed JPEG bytes -> cc_jpeg_decode_u8c3 (nvJPEG +
    the raster->frame transposition kernel) -> cc_rectify_u8c3_views, nothing returns to the host in
    between.  The decoder is checked against cv2.imdecode (libjpeg: IDCT / upsampling differ by a few
    LSB), the rectification of the DECODED frames is bit-equal to the oracle on the same bytes."""
    cv2 = pytest.importorskip("cv2")
    rng = np.random.default_rng(21)
    h, w = 250, 368                                     # rows, columns
    yy, xx = np.mgrid[0:h, 0:w]
    imgs = []
    for i in range(3):                                  # smooth content: JPEG keeps it within a few LSB
        im = np.stack([127 + 100 * np.sin(xx / (17.0 + i) + i) * np.cos(yy / 23.0),
                       127 + 90 * np.cos(xx / 31.0) * np.sin(yy / (13.0 + 2 * i)),
                       (xx * 255.0 / w + yy * 0.2 * i) % 256 * 0 + 60 + 0.5 * xx], axis=-1)
        imgs.append(np.clip(im + rng.normal(0, 2, im.shape), 0, 255).astype(np.uint8))
    enc = [cv2.imencode(".jpg", im[:, :, ::-1], [cv2.IMWRITE_JPEG_QUALITY, 95])[1].tobytes() for im in imgs]   # cv2 is BGR
    assert cc.jpeg_info(enc[0]) == (h, w, 3)
    try:
        frames = cc.load_jpegs(enc)
    except cc.CamcalError as e:
        if "libnvjpeg" in str(e):
            pytest.skip("libnvjpeg.so.12 not on this box")
        raise
    assert tuple(frames.shape) == (3, w, h, 3) and frames.is_cuda
    got = frames.cpu().numpy()
    for i in range(3):
        ref = cv2.imdecode(np.frombuffer(enc[i], np.uint8), cv2.IMREAD_COLOR)[:, :, ::-1]      # (h, w, RGB)
        d = np.abs(got[i].transpose(1, 0, 2).astype(np.int16) - ref.astype(np.int16))           # frame memory is [c][r]
        assert d.max() <= 12 and d.mean() < 2.0, (i, d.max(), d.mean())   # 4:2:0 chroma upsampling differs between the decoders
        assert np.abs(got[i].transpose(1, 0, 2).astype(np.int16) - imgs[i].astype(np.int16)).mean() < 4.0
    # grey stream: R = G = B, like RGB.(load(file))
    g = cv2.imencode(".jpg", imgs[0][:, :, 1], [cv2.IMWRITE_JPEG_QUALITY, 95])[1].tobytes()
    assert cc.jpeg_info(g) == (h, w, 1)
    gf = cc.load_jpegs([g]).cpu().numpy()[0]
    assert np.array_equal(gf[..., 0], gf[..., 1]) and np.array_equal(gf[..., 1], gf[..., 2])
    assert np.abs(gf[..., 0].T.astype(np.int16) - imgs[0][:, :, 1].astype(np.int16)).mean() < 3.0
    # decoded frames straight into the views call (three different extrinsics), against the oracle
    sz = (h, w)
    intr = camera_for(sz)
    views = [((0.15, -0.1, rz), (-8.0, -12.0, 30.0)) for rz in (0.02, 0.3, -0.2)]
    c = _calib(cc, intr, views)
    ras = [_rect_case(intr, sz, view=v) for v in views]
    out = cc.warp_views(c, [0, 1, 2], frames, [r[2] for r in ras], [r[3] for r in ras], fill=(0, 0, 0)).cpu().numpy()
    for i, (ch, _, ratio, axs) in enumerate(ras):
        ref = oc.rectify_u8c3(ch, 1.0 / ratio, axs, got[i:i + 1], fill=(0, 0, 0))[0]
        assert np.array_equal(out[i], ref), i
    # wrong size and garbage are errors, not crashes
    with pytest.raises(cc.CamcalError):
        cc.load_jpegs([enc[0], cv2.imencode(".jpg", imgs[0][:100])[1].tobytes()])
    with pytest.raises(cc.CamcalError):
        cc.jpeg_info(b"not a jpeg at all, just bytes")


def test_reproj_on_two_streams_of_one_context(cc):
    """The per-context scratch of reproj_jtj / calc_errors / LM is ordered across streams (ADVICE r1):
    the same call issued alternately on two streams gives the same block every time."""
    rng = np.random.default_rng(8)
    nv, nc = 3000, 280
    views = np.concatenate([rng.normal(0, 0.3, (nv, 3)), np.array([-10.0, -7.0, 40.0]) + rng.normal(0, 2.0, (nv, 3))], 1)
    obj = np.array([[a, b, 0.0] for b in range(14) for a in range(20)], dtype=np.float64)
    img = rng.normal(1000.0, 300.0, (nv, nc, 2))
    tv, to, ti = _dev(views), _dev(obj), _dev(img)
    tv2, ti2 = _dev(views[::-1].copy()), _dev(img[::-1].copy())
    ref = cc.reproj_jtj(C3_INTR, 1.0, tv, to, ti)[1].cpu().numpy()
    ref2 = cc.reproj_jtj(C3_INTR, 1.0, tv2, to, ti2)[1].cpu().numpy()
    s1, s2 = torch.cuda.Stream(), torch.cuda.Stream()
    torch.cuda.synchronize()
    outs = []
    for i in range(12):
        with torch.cuda.stream(s1 if i % 2 == 0 else s2):
            outs.append(cc.reproj_jtj(C3_INTR, 1.0, tv if i % 2 == 0 else tv2, to, ti if i % 2 == 0 else ti2)[1])
    torch.cuda.synchronize()
    for i, o in enumerate(outs):
        assert np.array_equal(o.cpu().numpy(), ref if i % 2 == 0 else ref2), i


def test_plot_writes_the_rectified_images(cc, example_fit, tmp_path):
    """plot(c, imgpointss, n_corners, checker_size, sz), src/plot_calibration.jl:36-44: every image rectified with
    its own extrinsic in one views call; the files on disk are the oracle's rectification of the red-cross images
    except where the blue crosses were drawn."""
    cv2 = pytest.importorskip("cv2")
    from cameracalibrations_b200.plotting import _draw_crosses, RED
    n1, n2 = example_fit["n_corners"]
    sz = (376, 500)                                     # rows, cols (376: word-aligned u8 lines)
    rng = np.random.default_rng(31)
    files, imgs = [], []
    for i in range(6):
        img = rng.integers(0, 256, (sz[0], sz[1], 3), dtype=np.uint8)      # (rows, cols, RGB)
        f = str(tmp_path / f"{i + 1}.png")
        cv2.imwrite(f, img[:, :, ::-1])
        files.append(f); imgs.append(img)
    c = _calib(cc, example_fit["intr_tuple"], example_fit["view_list"], files)
    ips = np.asarray(example_fit["corners_np"], dtype=np.float64).reshape(6, -1, 2)
    out = cc.plot(c, ips, (n1, n2), 1.0, sz, dir=str(tmp_path / "debug"))
    assert [os.path.basename(p) for p in out] == [f"{i + 1}.png" for i in range(6)]
    for i, p in enumerate(out):
        got = cv2.imread(p, cv2.IMREAD_COLOR)[:, :, ::-1]                   # (rows, cols, RGB)
        assert got.shape == (sz[0], sz[1], 3)
        frame = np.ascontiguousarray(imgs[i].transpose(1, 0, 2))            # frame layout [c][r]
        _draw_crosses(frame, ips[i], n1, RED)
        ratio, axs = cc.image_transformations(c, i, ips, 1.0, (n1, n2), sz)
        ch = oc.chain(example_fit["intr_tuple"], *example_fit["view_list"][i])
        ref = oc.rectify_u8c3(ch, 1.0 / ratio, axs, frame[None], fill=(0, 0, 0))[0].transpose(1, 0, 2)
        diff = np.any(got != ref, axis=-1)
        assert diff.mean() < 0.03                                           # only the blue crosses differ
        assert np.all(got[diff] == np.array([0, 0, 255], dtype=np.uint8))
        assert diff.sum() > 0                                               # and they were drawn


@pytest.mark.parametrize("seed", list(range(24)))
def test_rectify_random_geometries_bit_exact(cc, seed):
    """Randomised plan geometry: small and odd frame sizes, rotations up to +-1 rad about every axis, ratios 0.4-2.5,
    boards partly or wholly outside the frame -- u8 RGB and fp32, staged when the layout allows, against the oracle."""
    rng = np.random.default_rng(1000 + seed)
    sz1 = int(rng.choice([16, 32, 48, 64, 80, 112, 160, 208, 368]))
    sz2 = int(rng.integers(3, 120))
    sz = (sz1, sz2)
    intr = camera_for(sz, k=float(rng.choice([-0.12, 0.0, 0.05, 0.3])))
    rv = tuple(rng.uniform(-1.0, 1.0, 3) * np.array([0.5, 0.5, 1.0]))
    tv = (float(rng.uniform(-14, 2)), float(rng.uniform(-14, 2)), float(rng.uniform(18, 45)))
    view = (rv, tv)
    try:
        ch, ip, ratio, axs = _rect_case(intr, sz, ratio_scale=float(rng.uniform(0.4, 2.5)), view=view)
    except Exception:
        pytest.skip("degenerate view")
    if not np.isfinite(ratio) or ratio <= 0:
        pytest.skip("degenerate view")
    c = _calib(cc, intr, [view])
    nf = int(rng.integers(1, 5))
    f8 = rng.integers(0, 256, (nf, sz2, sz1, 3), dtype=np.uint8)
    ref8 = oc.rectify_u8c3(ch, 1.0 / ratio, axs, f8, fill=(3, 2, 1))
    got8 = cc.warp(c, 0, _dev(f8), ratio, axs, fill=(3, 2, 1)).cpu().numpy()
    assert np.array_equal(got8, ref8)
    f32 = rng.random((nf, sz2, sz1), dtype=np.float32)
    ref32 = oc.rectify_f32c1(ch, 1.0 / ratio, axs, f32, fill=-1.0)
    got32 = cc.warp(c, 0, _dev(f32), ratio, axs, fill=-1.0).cpu().numpy()
    assert np.array_equal(got32, ref32)
    # the FP32 fast path agrees wherever both sample: +-1 LSB on u8 (white noise amplifies a 1e-3 px map error)
    fast8 = cc.warp(c, 0, _dev(f8), ratio, axs, fill=(3, 2, 1), coord="f32").cpu().numpy()
    both = np.any(ref8 != np.array((3, 2, 1), np.uint8), -1) & np.any(fast8 != np.array((3, 2, 1), np.uint8), -1)
    if both.any():
        assert np.abs(fast8[both].astype(np.int16) - ref8[both].astype(np.int16)).max() <= 2


def test_plain_c_consumer_computes_on_the_gpu(cc, tmp_path):
    """tests/c/abi_consumer.c: world->pixel->world, a rectification and the error codes through the C ABI from C."""
    from test_abi import _build_c_consumer
    r = _build_c_consumer(tmp_path)
    assert r.returncode == 0 and r.stdout.strip() == "ok", r.stdout + r.stderr
