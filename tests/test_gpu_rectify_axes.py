"""Rectification into output axes of any size on the device: cc_rectify_axes_f32c1 / _u8c3 and their _host forms,
one view and many (3, and 70: a 64-view group and a tail), one frame per view and several frame groups per view.

  exact coordinates:  bit-equal to the reference of tests/rectify_axes_ref.py for a 2x downscale, a 2x upscale,
                      an interior crop at a shifted axs_min, odd extents with partial tiles on both axes, a window without an
                      in-frame pixel, and a padded out_pitch / out_frame_stride whose padding keeps its sentinel
  same size:          byte-identical to cc_rectify_* / _views / _host with the same launch count
  crop identity:      a window of a larger output equals a call with that window's axes, bit for bit
  fast coordinates:   the kernels sample cc_rectify_map_f32's map for the same extent (f32 ramps within 5e-4,
                      u8 within 1 LSB, rarely 2)
  paths:              a 2x downscale is staged; a 4x downscale and CC_GATHER_DIRECT are direct
  plan cache:         calls alternating two output extents of one view stay correct
  argument rules:     CC_ERR_INVALID_ARG and dst untouched
"""
import ctypes as C

import numpy as np
import pytest

torch = pytest.importorskip("torch")

from conftest import camera_for
from oracle import oracle_c as oc
import rectify_axes_ref as axref
from test_gpu_batching import _env, _staged_lines
from test_gpu_parity import _perturbed_views, _rect_case

pytestmark = pytest.mark.gpu

F_FILL, F_SENT = -3.0, -777.0
U_FILL, U_SENT = (9, 8, 7), 211
COORD_F32, GATHER_DIRECT = 1, 16


@pytest.fixture(scope="module")
def cc():
    import cameracalibrations_b200 as m
    assert torch.cuda.is_available(), "GPU tests need a CUDA device"
    m.context(0)
    return m


class Case:
    """A call: views (rvec, tvec), the camera, per-view ratio and axs_min, the output extent."""

    def __init__(self, intr, views, ratios, axs, out_sz):
        self.intr, self.views, self.ratios, self.axs, self.out_sz = intr, views, list(ratios), list(axs), out_sz


def _base(sz, nv):
    """nv views of a camera sized for frames sz, each with the ratio / axes get_ratio / get_axes give it"""
    intr = camera_for(sz)
    views = _perturbed_views(nv)
    ratios, axs = [], []
    for v in views:
        _, _, r, a = _rect_case(intr, sz, view=v)
        ratios.append(r)
        axs.append(a)
    return intr, views, ratios, axs


def _outputs(sz, nv):
    """name -> Case of the output kinds every form is checked on"""
    intr, views, ratios, axs = _base(sz, nv)
    sh = lambda d1, d2: [(a[0] + d1, a[1] + d2) for a in axs]
    return {
        "down2": Case(intr, views, [r / 2 for r in ratios], [(a[0] // 2, a[1] // 2) for a in axs], (sz[0] // 2, sz[1] // 2)),
        "up2": Case(intr, views, [r * 2 for r in ratios], [(2 * a[0], 2 * a[1]) for a in axs], (2 * sz[0], 2 * sz[1])),
        "crop": Case(intr, views, ratios, sh(sz[0] // 5, sz[1] // 4), (sz[0] // 2 + 3, sz[1] // 2 + 1)),
        "odd": Case(intr, views, ratios, sh(-17, 5), (1000, 77)),
        "all_fill": Case(intr, views, ratios, sh(50 * sz[0], 0), (97, 45)),
        "padded": Case(intr, views, [r * 0.75 for r in ratios], [(a[0] * 3 // 4, a[1] * 3 // 4) for a in axs],
                       (sz[0] * 3 // 4, sz[1] * 3 // 4)),
    }


def _src(fmt, n, sz, seed):
    rng = np.random.default_rng(seed)
    if fmt == "f32":
        return np.stack([rng.random((sz[1], sz[0]), dtype=np.float32) + np.float32(i) for i in range(n)])
    return rng.integers(0, 256, (n, sz[1], sz[0], 3), dtype=np.uint8)


def _oracle(fmt, case, src, fpv, fill=None):
    outs = []
    for v, view in enumerate(case.views):
        ch = oc.chain(case.intr, *view)
        fr = src[v * fpv:(v + 1) * fpv]
        if fmt == "f32":
            outs.append(axref.rectify_f32c1(ch, 1.0 / case.ratios[v], case.axs[v], fr, case.out_sz,
                                          fill=F_FILL if fill is None else fill))
        else:
            outs.append(axref.rectify_u8c3(ch, 1.0 / case.ratios[v], case.axs[v], fr, case.out_sz,
                                         fill=U_FILL if fill is None else fill))
    return np.concatenate(outs)


def _call(cc, fmt, host, case, src, fpv, out_pitch=None, out_fs=None, flags=0, sym=None):
    """One cc_rectify_axes_* call (or `sym` with the same-size arguments of the older entry points).  Returns
    (status, flat output buffer as numpy, launches).  The buffer starts filled with the sentinel."""
    L = cc._lib
    u8 = fmt == "u8"
    n, sz2, sz1 = src.shape[0], src.shape[1], src.shape[2]
    o1, o2 = case.out_sz
    op = o1 if out_pitch is None else out_pitch
    ofs = op * o2 if out_fs is None else out_fs
    ch = 3 if u8 else 1
    total = max(1, (n - 1) * ofs + (o2 - 1) * op + o1 if n else 1) * ch
    dt = np.uint8 if u8 else np.float32
    sent = U_SENT if u8 else F_SENT
    nv = len(case.views)
    views = (L.View * nv)(*[L.make_view(r, t) for r, t in case.views])
    ratios = (C.c_double * nv)(*case.ratios)
    axs = (C.c_int64 * (2 * nv))(*[int(x) for a in case.axs for x in a])
    intr = L.make_intr(*case.intr)
    fill = (C.c_uint8 * 3)(*U_FILL) if u8 else C.c_float(F_FILL)
    ctx = cc.context(0)
    if host:
        s = np.ascontiguousarray(src)
        d = np.full(total, sent, dt)
        sp, dp, tail = C.c_void_p(s.ctypes.data), C.c_void_p(d.ctypes.data), ()
    else:
        s = torch.from_numpy(np.ascontiguousarray(src)).cuda()
        d = torch.full((total,), sent, dtype=torch.uint8 if u8 else torch.float32, device="cuda")
        sp, dp, tail = C.c_void_p(s.data_ptr()), C.c_void_p(d.data_ptr()), (C.c_void_p(torch.cuda.current_stream().cuda_stream),)
        torch.cuda.synchronize()
    n0 = ctx.launch_count()
    kern = "u8c3" if u8 else "f32c1"
    if sym is None:
        fn = getattr(L.lib, f"cc_rectify_axes_{kern}{'_host' if host else ''}")
        st = fn(ctx.handle, C.byref(intr), views, nv, ratios, axs, o1, o2, sp, sz1, sz2, C.c_size_t(sz1),
                C.c_size_t(sz1 * sz2), dp, C.c_size_t(op), C.c_size_t(ofs), n // nv, fill, flags, *tail)
    elif nv == 1 and "views" not in sym:
        st = getattr(L.lib, sym)(ctx.handle, C.byref(intr), C.byref(views[0]), case.ratios[0], axs, sp, dp, sz1, sz2,
                                 C.c_size_t(sz1), C.c_size_t(sz1 * sz2), n, fill, flags, *tail)
    else:
        st = getattr(L.lib, sym)(ctx.handle, C.byref(intr), views, nv, ratios, axs, sp, dp, sz1, sz2, C.c_size_t(sz1),
                                 C.c_size_t(sz1 * sz2), n // nv, fill, flags, *tail)
    if not host:
        torch.cuda.synchronize()
        d = d.cpu().numpy()
    return st, d, ctx.launch_count() - n0


def _frames_of(flat, fmt, n, out_sz, out_pitch=None, out_fs=None):
    """the (n, out_sz2, out_sz1[, 3]) frames inside a flat output buffer, and the mask of bytes they own"""
    o1, o2 = out_sz
    op = o1 if out_pitch is None else out_pitch
    ofs = op * o2 if out_fs is None else out_fs
    chn = 3 if fmt == "u8" else 1
    idx = (np.arange(n)[:, None, None] * ofs + np.arange(o2)[None, :, None] * op + np.arange(o1)[None, None, :]) * chn
    idx = idx[..., None] + np.arange(chn)
    frames = flat[idx] if fmt == "u8" else flat[idx[..., 0]]
    owned = np.zeros(flat.shape, bool)
    owned[idx.ravel()] = True
    return frames, owned


def _same(a, b):
    return np.array_equal(a, b, equal_nan=a.dtype.kind == "f")


# ------------------------------------------------------------------ exact coordinates against the oracle
LAYOUTS = [(1, 1, (256, 192)), (1, 3, (256, 192)), (3, 1, (256, 192)), (3, 3, (192, 160)), (70, 1, (128, 96)),
           (70, 2, (96, 64))]


@pytest.mark.parametrize("nv, fpv, sz", LAYOUTS)
@pytest.mark.parametrize("host", [False, True])
@pytest.mark.parametrize("fmt", ["f32", "u8"])
def test_exact_outputs_match_the_oracle(cc, fmt, host, nv, fpv, sz):
    src = _src(fmt, nv * fpv, sz, seed=nv * 10 + fpv)
    for name, case in _outputs(sz, nv).items():
        o1, o2 = case.out_sz
        pad = name == "padded"
        op = o1 + (4 if fmt == "u8" else 13) if pad else None           # u8: lines stay 4-byte aligned (staged)
        ofs = op * o2 + 8 if pad else None
        st, flat, launches = _call(cc, fmt, host, case, src, fpv, op, ofs)
        assert st == 0, (name, cc._lib.last_error())
        got, owned = _frames_of(flat, fmt, nv * fpv, case.out_sz, op, ofs)
        ref = _oracle(fmt, case, src, fpv)
        assert _same(got, ref), (name, fmt, host, nv, fpv)
        assert np.all(flat[~owned] == (U_SENT if fmt == "u8" else F_SENT)), name     # padding never written
        if name == "all_fill":
            assert np.all(got == (np.array(U_FILL, np.uint8) if fmt == "u8" else np.float32(F_FILL)))
        else:
            fill = np.all(got == np.array(U_FILL, np.uint8), axis=-1) if fmt == "u8" else got == np.float32(F_FILL)
            assert not fill.all(), name
        assert launches >= 1


# ------------------------------------------------------------------ same-size identity
SYMS = {(False, False): "cc_rectify_{k}", (False, True): "cc_rectify_{k}_views", (True, False): "cc_rectify_{k}_host",
        (True, True): "cc_rectify_views_{k}_host"}


@pytest.mark.parametrize("nv, fpv, sz", [(1, 3, (256, 192)), (3, 2, (200, 120)), (70, 1, (128, 96))])
@pytest.mark.parametrize("host", [False, True])
@pytest.mark.parametrize("fmt", ["f32", "u8"])
@pytest.mark.parametrize("flags", [0, COORD_F32, GATHER_DIRECT])
def test_same_size_is_the_existing_entry_point(cc, fmt, host, nv, fpv, sz, flags):
    intr, views, ratios, axs = _base(sz, nv)
    case = Case(intr, views, ratios, axs, sz)
    src = _src(fmt, nv * fpv, sz, seed=5)
    st, new, n_new = _call(cc, fmt, host, case, src, fpv, flags=flags)
    assert st == 0, cc._lib.last_error()
    sym = SYMS[(host, nv > 1)].format(k="u8c3" if fmt == "u8" else "f32c1")
    st, old, n_old = _call(cc, fmt, host, case, src, fpv, flags=flags, sym=sym)
    assert st == 0, cc._lib.last_error()
    assert new.tobytes() == old.tobytes()
    assert n_new == n_old


# ------------------------------------------------------------------ crop identity
@pytest.mark.parametrize("host", [False, True])
@pytest.mark.parametrize("fmt", ["f32", "u8"])
def test_crop_identity(cc, fmt, host):
    sz = (320, 240)
    intr, views, ratios, axs = _base(sz, 3)
    big = Case(intr, views, ratios, axs, (2 * sz[0] // 3 * 2, sz[1]))
    src = _src(fmt, 6, sz, seed=9)
    st, flat, _ = _call(cc, fmt, host, big, src, 2)
    assert st == 0
    whole, _ = _frames_of(flat, fmt, 6, big.out_sz)
    for (d1, d2), (n1, n2) in [((0, 0), (32, 32)), ((5, 7), (200, 100)), ((33, 65), (1, 1)), ((96, 3), (300, 237))]:
        win = Case(intr, views, ratios, [(a[0] + d1, a[1] + d2) for a in axs], (n1, n2))
        st, flat, _ = _call(cc, fmt, host, win, src, 2)
        assert st == 0
        got, _ = _frames_of(flat, fmt, 6, (n1, n2))
        assert _same(got, whole[:, d2:d2 + n2, d1:d1 + n1]), ((d1, d2), (n1, n2))


# ------------------------------------------------------------------ fast coordinates: cc_rectify_map_f32's map
def _map_f32(cc, case, v):
    c = cc.Calibration(case.intr[:4], case.views, 1.0 / case.intr[5], case.intr[4], [f"{i}.png" for i in range(len(case.views))])
    mr, mc = cc.rectify_map(c, v, case.ratios[v], case.axs[v], case.out_sz, coord="f32")
    torch.cuda.synchronize()
    return mr.cpu().numpy().astype(np.float64), mc.cpu().numpy().astype(np.float64)


def _blend_u8(img, mr, mc):
    """the oracle's bilinear rule (FP64, rint) at the given coordinates; NaN outside [1, n]"""
    sz2, sz1 = img.shape[:2]
    inb = (mr >= 1) & (mr <= sz1) & (mc >= 1) & (mc <= sz2)
    r, c = np.where(inb, mr, 1.0), np.where(inb, mc, 1.0)
    i1 = np.minimum(np.floor(r), sz1 - 1).astype(int)
    i2 = np.minimum(np.floor(c), sz2 - 1).astype(int)
    d1, d2 = (r - i1)[..., None], (c - i2)[..., None]
    a = img.astype(np.float64)
    i1, i2 = i1 - 1, i2 - 1
    v = (1 - d1) * ((1 - d2) * a[i2, i1] + d2 * a[i2 + 1, i1]) + d1 * ((1 - d2) * a[i2, i1 + 1] + d2 * a[i2 + 1, i1 + 1])
    return np.rint(v), inb


def _edge_margin(mr, mc, sz, m=1e-2):
    """pixels whose FP32 map is farther than m from the frame's bounds: there the fill decision is certain"""
    return (np.abs(mr - 1) > m) & (np.abs(mr - sz[0]) > m) & (np.abs(mc - 1) > m) & (np.abs(mc - sz[1]) > m)


@pytest.mark.parametrize("host", [False, True])
@pytest.mark.parametrize("kind", ["down2", "up2", "odd"])
def test_fast_f32_samples_the_map_f32(cc, kind, host):
    sz = (256, 192)
    case = _outputs(sz, 3)[kind]
    ramps = np.stack([np.broadcast_to(np.arange(1, sz[0] + 1, dtype=np.float32)[None, :], (sz[1], sz[0])),
                      np.broadcast_to(np.arange(1, sz[1] + 1, dtype=np.float32)[:, None], (sz[1], sz[0]))] * 3)
    st, flat, _ = _call(cc, "f32", host, case, ramps, 2, flags=COORD_F32)
    assert st == 0
    got, _ = _frames_of(flat, "f32", 6, case.out_sz)
    for v in range(3):
        mr, mc = _map_f32(cc, case, v)
        sure = _edge_margin(mr, mc, sz)
        inb = (mr >= 1) & (mr <= sz[0]) & (mc >= 1) & (mc <= sz[1])
        assert (inb & sure).mean() > 0.1
        for j, m in enumerate((mr, mc)):
            g = got[2 * v + j].astype(np.float64)
            assert np.all(g[~inb & sure] == F_FILL)
            assert np.max(np.abs(g[inb & sure] - m[inb & sure])) <= 5e-4, (kind, v, j)


@pytest.mark.parametrize("host", [False, True])
@pytest.mark.parametrize("kind", ["down2", "up2", "crop"])
def test_fast_u8_samples_the_map_f32(cc, kind, host):
    sz = (256, 192)
    case = _outputs(sz, 3)[kind]
    src = _src("u8", 3, sz, seed=21)
    st, flat, _ = _call(cc, "u8", host, case, src, 1, flags=COORD_F32)
    assert st == 0
    got, _ = _frames_of(flat, "u8", 3, case.out_sz)
    over1 = total = 0
    for v in range(3):
        mr, mc = _map_f32(cc, case, v)
        ref, inb = _blend_u8(src[v], mr, mc)
        sure = _edge_margin(mr, mc, sz)
        g = got[v].astype(np.int64)
        assert np.all(g[~inb & sure] == np.array(U_FILL))
        d = np.abs(g[inb & sure] - ref[inb & sure])
        assert d.max() <= 2, (kind, v)
        over1 += int((d > 1).sum())
        total += d.size
    assert total > 0 and over1 <= 1e-3 * total


# ------------------------------------------------------------------ which path runs
@pytest.mark.parametrize("fmt", ["f32", "u8"])
@pytest.mark.parametrize("nv", [1, 3])
def test_paths(cc, capfd, fmt, nv):
    sz = (640, 480)
    intr, views, ratios, axs = _base(sz, nv)
    src = _src(fmt, 2 * nv, sz, seed=2)
    for scale, flags, staged in ((2, 0, True), (4, 0, False), (2, GATHER_DIRECT, False)):
        case = Case(intr, views, [r / scale for r in ratios], [(a[0] // scale, a[1] // scale) for a in axs],
                    (sz[0] // scale, sz[1] // scale))
        capfd.readouterr()
        with _env(CAMCAL_DEBUG="1"):
            st, flat, launches = _call(cc, fmt, False, case, src, 2, flags=flags)
        err = capfd.readouterr().err
        assert st == 0
        lines = _staged_lines(err)
        if staged:
            assert launches == 1 and len(lines) == 1, err[-2000:]
        else:
            assert launches == nv and lines == [], err[-2000:]
        got, _ = _frames_of(flat, fmt, 2 * nv, case.out_sz)
        assert _same(got, _oracle(fmt, case, src, 2)), (scale, flags)


# ------------------------------------------------------------------ the plan cache
@pytest.mark.parametrize("fmt", ["f32", "u8"])
def test_alternating_output_extents_share_no_plan(cc, fmt):
    sz = (256, 192)
    intr, views, ratios, axs = _base(sz, 1)
    src = _src(fmt, 2, sz, seed=4)
    cases = [Case(intr, views, ratios, axs, out) for out in ((256, 192), (128, 96), (300, 40))]
    refs = [_oracle(fmt, c, src, 2) for c in cases]
    for it in range(7):
        for host in (False, True):
            k = (it + host) % 3
            st, flat, _ = _call(cc, fmt, host, cases[k], src, 2)
            assert st == 0
            got, _ = _frames_of(flat, fmt, 2, cases[k].out_sz)
            assert _same(got, refs[k]), (it, host, k)


# ------------------------------------------------------------------ argument rules
@pytest.mark.parametrize("host", [False, True])
@pytest.mark.parametrize("fmt", ["f32", "u8"])
def test_argument_rules(cc, fmt, host):
    sz = (64, 48)
    intr, views, ratios, axs = _base(sz, 2)
    src = _src(fmt, 4, sz, seed=1)
    bad = [  # (out_sz, out_pitch, out_frame_stride, src == dst)
        ((0, 10), None, None, False), ((10, 0), None, None, False), ((-3, 10), 10, 100, False),
        ((1 << 22, 1), None, None, False), ((10, 1 << 22), None, None, False),
        ((32, 20), 31, 31 * 20, False),                        # out_pitch < out_sz1
        ((32, 20), 32, 32 * 19 + 31, False),                   # output frames overlap
        ((8, 2), 1 << 29, (1 << 30) + 8, False),               # out_pitch * out_sz2 >= 2^30
        ((32, 20), None, None, True),                          # src == dst
    ]
    for out_sz, op, ofs, same in bad:
        case = Case(intr, views, ratios, axs, out_sz)
        o1, o2 = max(out_sz[0], 1), max(out_sz[1], 1)
        probe = Case(intr, views, ratios, axs, (min(o1, 64), min(o2, 64)))
        st = _call_raw_invalid(cc, fmt, host, case, probe, src, op, ofs, same)
        assert st == cc._lib.CC_ERR_INVALID_ARG, (out_sz, op, ofs, same)


def _call_raw_invalid(cc, fmt, host, case, probe, src, op, ofs, same):
    """An invalid call with a small sentinel-filled dst (the probe's extent): the status, after checking that
    dst is unchanged."""
    L = cc._lib
    u8 = fmt == "u8"
    n, sz2, sz1 = src.shape[0], src.shape[1], src.shape[2]
    nv = len(case.views)
    chn = 3 if u8 else 1
    total = n * probe.out_sz[0] * probe.out_sz[1] * chn
    sent = U_SENT if u8 else F_SENT
    views = (L.View * nv)(*[L.make_view(r, t) for r, t in case.views])
    ratios = (C.c_double * nv)(*case.ratios)
    axs = (C.c_int64 * (2 * nv))(*[int(x) for a in case.axs for x in a])
    intr = L.make_intr(*case.intr)
    fill = (C.c_uint8 * 3)(*U_FILL) if u8 else C.c_float(F_FILL)
    o1, o2 = case.out_sz
    op = max(o1, 0) if op is None else op
    ofs = op * max(o2, 0) if ofs is None else ofs
    ctx = cc.context(0)
    if host:
        s = np.ascontiguousarray(src)
        d = np.full(total, sent, np.uint8 if u8 else np.float32)
        sp, dp, tail = C.c_void_p(s.ctypes.data), C.c_void_p(d.ctypes.data), ()
    else:
        s = torch.from_numpy(np.ascontiguousarray(src)).cuda()
        d = torch.full((total,), sent, dtype=torch.uint8 if u8 else torch.float32, device="cuda")
        sp, dp, tail = C.c_void_p(s.data_ptr()), C.c_void_p(d.data_ptr()), (C.c_void_p(torch.cuda.current_stream().cuda_stream),)
    if same:
        dp = sp
    n0 = ctx.launch_count()
    fn = getattr(L.lib, f"cc_rectify_axes_{'u8c3' if u8 else 'f32c1'}{'_host' if host else ''}")
    st = fn(ctx.handle, C.byref(intr), views, nv, ratios, axs, o1, o2, sp, sz1, sz2, C.c_size_t(sz1),
            C.c_size_t(sz1 * sz2), dp, C.c_size_t(op), C.c_size_t(ofs), n // nv, fill, 0, *tail)
    assert ctx.launch_count() == n0
    if not host:
        torch.cuda.synchronize()
        d = d.cpu().numpy()
        assert np.array_equal(s.cpu().numpy(), src)
    else:
        assert np.array_equal(s, src)
    assert np.all(d == sent)
    return st


@pytest.mark.parametrize("host", [False, True])
def test_source_rules_still_apply(cc, host):
    """pitch < sz1 on the source is rejected as by cc_rectify_*, whatever the output"""
    sz = (64, 48)
    intr, views, ratios, axs = _base(sz, 1)
    L = cc._lib
    src = _src("f32", 1, sz, seed=0)
    views_a = (L.View * 1)(L.make_view(*views[0]))
    ratios_a = (C.c_double * 1)(ratios[0])
    axs_a = (C.c_int64 * 2)(*axs[0])
    if host:
        s, d = src, np.full(32 * 32, F_SENT, np.float32)
        sp, dp, tail = C.c_void_p(s.ctypes.data), C.c_void_p(d.ctypes.data), ()
    else:
        s, d = torch.from_numpy(src).cuda(), torch.full((32 * 32,), F_SENT, device="cuda")
        sp, dp, tail = C.c_void_p(s.data_ptr()), C.c_void_p(d.data_ptr()), (C.c_void_p(0),)
    fn = L.lib.cc_rectify_axes_f32c1_host if host else L.lib.cc_rectify_axes_f32c1
    st = fn(cc.context(0).handle, C.byref(L.make_intr(*intr)), views_a, 1, ratios_a, axs_a, 32, 32, sp, sz[0], sz[1],
            C.c_size_t(sz[0] - 1), C.c_size_t(sz[0] * sz[1]), dp, C.c_size_t(32), C.c_size_t(32 * 32), 1,
            C.c_float(F_FILL), 0, *tail)
    assert st == L.CC_ERR_INVALID_ARG
    out = d if host else d.cpu().numpy()
    assert np.all(out == F_SENT)


def test_warp_out_size_end_to_end(cc):
    """warp / warp_views with out_size on CUDA tensors and numpy arrays: the oracle's output"""
    sz = (256, 192)
    case = _outputs(sz, 3)["down2"]
    c = cc.Calibration(case.intr[:4], case.views, 1.0 / case.intr[5], case.intr[4], ["a.png", "b.png", "c.png"])
    src = _src("f32", 3, sz, seed=8)
    ref = _oracle("f32", case, src, 1, fill=np.nan)
    for frames in (src, torch.from_numpy(src).cuda()):
        y = cc.warp(c, 1, frames[1:2], case.ratios[1], case.axs[1], out_size=case.out_sz)
        y = y.cpu().numpy() if isinstance(y, torch.Tensor) else y
        assert _same(y, ref[1:2])
        y = cc.warp_views(c, [0, 1, 2], frames, case.ratios, case.axs, out_size=case.out_sz)
        y = y.cpu().numpy() if isinstance(y, torch.Tensor) else y
        assert _same(y, ref)
