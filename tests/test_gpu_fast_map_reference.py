"""The FP32 fast path on the device against the independent reference of oracle/map_ref.py.

cc_rectify_map_f32 is within the per-pixel FP32 bound of the reference at every in-frame pixel and within
1e-3 px wherever the lens is monotone and the point is in front of the camera; cc_rectify_map_f64 is within
the FP64 bound.  Every fast kernel family (staged, direct, views with a full and a tail group, host, views
from host) warps row and column ramps: bilinear blending reproduces a ramp, so the outputs are the map.
The u8c3 fast kernels on white noise are held to a per-pixel bound from the map bound and the local tap
differences.  A pixel may switch between fill and sample only where the reference coordinate is within
the bound of the frame's edges."""
import numpy as np
import pytest

torch = pytest.importorskip("torch")

from oracle import map_ref as mr
from test_gpu_batching import _env, _staged_lines

pytestmark = pytest.mark.gpu

GEOMS = mr.geometries()
TOL32_PX = 1e-3
BLEND_U8 = 0.02          # IDP weights: 6 * 2^-17 of 255 (0.012 LSB); FP32 blend: a few u of 255


@pytest.fixture(scope="module")
def cc():
    import cameracalibrations_b200 as m
    assert torch.cuda.is_available(), "GPU tests need a CUDA device"
    m.context(0)
    return m


def _calib(cc, gs):
    g = gs[0]
    return cc.Calibration(g.intr[:4], [gg.view for gg in gs], 1.0 / g.intr[5], g.intr[4],
                          [f"{i}.png" for i in range(len(gs))])


def _ramps(sz, n=1):
    """n copies of (row ramp, column ramp): value = 1-based index along the first / second axis"""
    r = np.broadcast_to(np.arange(1, sz[0] + 1, dtype=np.float32)[None, :], (sz[1], sz[0]))
    q = np.broadcast_to(np.arange(1, sz[1] + 1, dtype=np.float32)[:, None], (sz[1], sz[0]))
    return np.ascontiguousarray(np.stack([r, q] * n))


def _edge(x, b, n):
    """the reference coordinate is within its bound of 1 or n"""
    return (np.abs(x - 1) <= b) | (np.abs(x - n) <= b)


def _check_sampled(name, g, ch, got_r, got_c, extra=0.0):
    """got (row, col) per pixel of chunk ch, NaN = fill: the fast path's map within its bound (+ extra * |x|)"""
    ref_r, ref_c = ch.row.astype(np.float64), ch.col.astype(np.float64)
    inf = ch.inframe(g.sz)
    assert np.all(np.isfinite(ch.b32_row[inf]) & np.isfinite(ch.b32_col[inf])), name
    filled = np.isnan(got_r) | np.isnan(got_c)
    assert np.array_equal(np.isnan(got_r), np.isnan(got_c)), name
    near = _edge(ref_r, ch.b32_row, g.sz[0]) | _edge(ref_c, ch.b32_col, g.sz[1])
    assert np.all(~(filled ^ ~inf) | near), name          # fill decisions change only at the edges
    s = ~filled
    er = np.abs(got_r[s] - ch.row[s]).astype(np.float64)
    ec = np.abs(got_c[s] - ch.col[s]).astype(np.float64)
    assert np.all(er <= ch.b32_row[s] + extra * np.abs(ref_r[s])), (name, er.max())
    assert np.all(ec <= ch.b32_col[s] + extra * np.abs(ref_c[s])), (name, ec.max())


@pytest.mark.parametrize("name", list(GEOMS))
def test_device_maps_within_bounds(cc, name):
    g = GEOMS[name]
    c = _calib(cc, [g])
    fr, fc = (t.cpu().numpy() for t in cc.rectify_map(c, 0, g.ratio, g.axs, g.sz, coord="f32"))
    dr, dc = (t.cpu().numpy() for t in cc.rectify_map(c, 0, g.ratio, g.axs, g.sz, coord="f64"))
    # per region: [largest device error, largest error of the numpy emulation, pixels]
    worst = {"monotone": [0.0, 0.0, 0], "past the fold": [0.0, 0.0, 0], "behind": [0.0, 0.0, 0]}
    for ch in mr.sweep(g):
        inf = ch.inframe(g.sz)
        assert np.all(np.isfinite(ch.b32_row[inf]) & np.isfinite(ch.b32_col[inf])), name
        er = np.abs(fr[ch.b, ch.a] - ch.row).astype(np.float64)
        ec = np.abs(fc[ch.b, ch.a] - ch.col).astype(np.float64)
        emr, emc = mr.emulate_fast(g, ch.a, ch.b)
        em = np.maximum(np.abs(emr - ch.row), np.abs(emc - ch.col)).astype(np.float64)
        assert np.all(er[inf] <= ch.b32_row[inf]) and np.all(ec[inf] <= ch.b32_col[inf]), \
            (name, np.max(er[inf] / ch.b32_row[inf]), np.max(ec[inf] / ch.b32_col[inf]))
        good = inf & ch.monotone & ch.front
        assert np.all(np.maximum(er, ec)[good] <= TOL32_PX), name
        for key, m in (("monotone", good), ("past the fold", inf & ch.front & ~ch.monotone),
                       ("behind", inf & ~ch.front)):
            if m.any():
                w = worst[key]
                worst[key] = [max(w[0], float(np.maximum(er, ec)[m].max())), max(w[1], float(em[m].max())),
                              w[2] + int(m.sum())]
        fin = np.isfinite(ch.row.astype(np.float64)) & np.isfinite(ch.col.astype(np.float64))
        e64r = np.abs(dr[ch.b, ch.a] - ch.row).astype(np.float64)
        e64c = np.abs(dc[ch.b, ch.a] - ch.col).astype(np.float64)
        assert np.all(e64r[fin] <= ch.b64_row[fin]) and np.all(e64c[fin] <= ch.b64_col[fin]), name
    print(f"\n{name}: cc_rectify_map_f32 max error (emulated) " +
          ", ".join(f"{k} {v[0]:.2e} ({v[1]:.2e}) px over {v[2]} px" for k, v in worst.items() if v[2]))


# name -> the whole frame stages (a TMA box holds every tile's footprint); the others reach past the fold or
# the horizon, where "auto" serves the tiles whose footprint is too large through the per-pixel path
FAMILY_GEOMS = {"c2_rx0.9_r1": True, "c2_far_axes": True, "c3_rx1.3_r0.4": False, "horizon_r6": False}


@pytest.mark.parametrize("name", list(FAMILY_GEOMS))
def test_fast_kernels_reproduce_the_map(cc, name):
    """Row and column ramps through the staged (TMA) and direct f32c1 kernels and the host pipeline"""
    g = GEOMS[name]
    c = _calib(cc, [g])
    frames = _ramps(g.sz)
    outs = {"host": cc.warp(c, 0, frames, g.ratio, g.axs, coord="f32"),
            "direct": cc.warp(c, 0, torch.from_numpy(frames).cuda(), g.ratio, g.axs, coord="f32",
                              gather="direct").cpu().numpy(),
            "auto": cc.warp(c, 0, torch.from_numpy(frames).cuda(), g.ratio, g.axs, coord="f32").cpu().numpy()}
    try:
        outs["tma"] = cc.warp(c, 0, torch.from_numpy(frames).cuda(), g.ratio, g.axs, coord="f32",
                              gather="tma").cpu().numpy()
    except cc.CamcalError:
        assert not FAMILY_GEOMS[name], name
    for kind, out in outs.items():
        for ch in mr.sweep(g):
            _check_sampled((name, kind), g, ch, out[0][ch.b, ch.a], out[1][ch.b, ch.a], extra=mr.U32)


def _view_geoms(nv, sz):
    """nv views of one camera whose common tile footprint stages: board tilts from frontal to rx = 0.6, both
    turn directions, ratios 1 to 2.5 times the board's"""
    rng = np.random.default_rng(nv)
    intr = mr.camera_for(sz)
    gs = []
    for v in range(nv):
        rx = 0.6 * v / (nv - 1)
        view = ((rx, float(rng.uniform(-0.2, 0.2)), float(rng.uniform(-0.6, 0.6))),
                (-8.0 + float(rng.uniform(-1, 1)), -12.0 + float(rng.uniform(-1, 1)), 30.0))
        gs.append(mr.geom(intr, view, sz, float(rng.choice([1.0, 1.6, 2.5]))))
    return gs


def test_fast_views_kernels_reproduce_the_map(cc, capfd):
    """cc_rectify_f32c1_views: 65 views in two staged launches, a 64-view group and a tail of one, each view
    with its own RectFast from the view table; cc_rectify_views_f32c1_host: every launch staged"""
    sz = (368, 250)
    gs = _view_geoms(65, sz)
    c = _calib(cc, gs)
    frames = _ramps(sz, len(gs))
    ratios, axs = [g.ratio for g in gs], [g.axs for g in gs]
    ctx = cc.context(0)
    fd = torch.from_numpy(frames).cuda()
    outs = {}
    for kind, src in (("views", fd), ("views_host", frames)):
        n0 = ctx.launch_count()
        capfd.readouterr()
        with _env(CAMCAL_DEBUG="1"):
            out = cc.warp_views(c, list(range(len(gs))), src, ratios, axs, coord="f32")
        outs[kind] = out if kind == "views_host" else out.cpu().numpy()
        launches, err = ctx.launch_count() - n0, capfd.readouterr().err
        if kind == "views":
            assert launches == 2 and len(_staged_lines(err)) == 2, err[-2000:]
        else:                                   # host chunks: one staged launch per group a chunk touches
            assert launches >= 2 and len(_staged_lines(err)) == launches, err[-2000:]
    for v, g in enumerate(gs):
        for ch in mr.sweep(g):
            for kind, out in outs.items():
                _check_sampled((v, kind), g, ch, out[2 * v][ch.b, ch.a], out[2 * v + 1][ch.b, ch.a], extra=mr.U32)


def _blend_ref(img, x1, x2):
    """bilinear blend of img (sz2, sz1, 3) at 1-based (x1, x2) by the reference's rule (in-frame points),
    and the largest tap difference of each channel over the 4 x 4 taps around the cell"""
    sz2, sz1 = img.shape[:2]
    i1 = np.minimum(np.floor(x1), sz1 - 1).astype(np.int64)
    i2 = np.minimum(np.floor(x2), sz2 - 1).astype(np.int64)
    d1, d2 = (x1 - i1)[:, None], (x2 - i2)[:, None]
    f = img.astype(np.float64)
    a00, a10 = f[i2 - 1, i1 - 1], f[i2 - 1, i1]
    a01, a11 = f[i2, i1 - 1], f[i2, i1]
    v = (1 - d1) * ((1 - d2) * a00 + d2 * a01) + d1 * ((1 - d2) * a10 + d2 * a11)
    lo, hi = np.full(v.shape, 255.0), np.zeros(v.shape)
    for o2 in (-2, -1, 0, 1):
        for o1 in (-2, -1, 0, 1):
            t = f[np.clip(i2 + o2, 0, sz2 - 1), np.clip(i1 + o1, 0, sz1 - 1)]
            lo, hi = np.minimum(lo, t), np.maximum(hi, t)
    return v, hi - lo


@pytest.mark.parametrize("name", ["c3_rx1.3_r0.4", "c2_rx0.6_r2.5", "c2_far_axes"])
@pytest.mark.parametrize("gather", ["auto", "direct"])
def test_u8c3_fast_on_white_noise(cc, name, gather):
    """Per pixel: |out - round(blend at the reference map)| <= ceil(0.5 + D (b_row + b_col) + blend error),
    D the largest tap difference around the cell; a pixel is fill (it follows the fill value) exactly where the
    reference is outside the frame, except within the bound of the edges."""
    g = GEOMS[name]
    c = _calib(cc, [g])
    rng = np.random.default_rng(17)
    img = rng.integers(0, 256, (1, g.sz[1], g.sz[0], 3), dtype=np.uint8)
    d = torch.from_numpy(img).cuda()
    o1 = cc.warp(c, 0, d, g.ratio, g.axs, fill=(0, 0, 0), coord="f32", gather=gather).cpu().numpy()[0]
    o2 = cc.warp(c, 0, d, g.ratio, g.axs, fill=(255, 255, 255), coord="f32", gather=gather).cpu().numpy()[0]
    for ch in mr.sweep(g):
        a1, a2 = o1[ch.b, ch.a], o2[ch.b, ch.a]
        filled = np.any(a1 != a2, axis=-1)
        assert np.all(filled == np.all(a1 != a2, axis=-1))
        x1, x2 = ch.row.astype(np.float64), ch.col.astype(np.float64)
        inf = ch.inframe(g.sz)
        near = _edge(x1, ch.b32_row, g.sz[0]) | _edge(x2, ch.b32_col, g.sz[1])
        assert np.all(~(filled ^ ~inf) | near), name
        s = inf & ~filled
        v, D = _blend_ref(img[0], x1[s], x2[s])
        lim = np.ceil(0.5 + D * (ch.b32_row[s] + ch.b32_col[s])[:, None] + BLEND_U8)
        diff = np.abs(a1[s].astype(np.float64) - np.rint(v))
        assert np.all(diff <= lim), (name, gather, float((diff - lim).max()))
