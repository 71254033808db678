"""Point maps on interleaved points, the reference's own layout: cc_img2world_* / cc_world2img_* `_aos` (device,
one launch) and `_aos_host` (chunked pipeline).  Every point's result must be bit-identical to the SoA entry
point with the same view, whatever the alignment; nothing may be written outside the output; against the
oracle at the SoA tolerances.

The CPU tests at the end need no device."""
import ctypes as C

import numpy as np
import pytest

from conftest import C2_INTR, SYN_VIEW
from test_abi import _header_params, _julia_ccalls

torch = pytest.importorskip("torch")

CHUNK = 1 << 22                 # kPointChunk of csrc/abi.cu: points per host pipeline stage
SENTINEL = -7.25
GUARD = 16                      # sentinel elements on each side of every output
SIZES = [0, 1, 2, 3, 5, 4095, 4096, 4097, (1 << 20) + 3]
SMALL_COUNTS = [0, 1, 2, 3, 0, 1, 1, 1, 4, 5, 6, 7, 0, 0, 9, 1, 130, 2, 3]   # ends at every residue mod 2 and 4
SMALL_VIEWS = [0, 1, 2, 0, 3, 1, 5, 2, 0, 7, 0, 9, 4, 4, 11, 0, 6, 3, 0]


@pytest.fixture(scope="module")
def cc():
    import cameracalibrations_b200 as m
    assert torch.cuda.is_available(), "GPU tests need a CUDA device"
    m.context(0)
    return m


def _poses(n, seed):
    rng = np.random.default_rng(seed)
    r0, t0 = np.asarray(SYN_VIEW[0]), np.asarray(SYN_VIEW[1])
    return [(tuple(r0 + rng.uniform(-0.15, 0.15, 3)), tuple(t0 + rng.uniform(-3, 3, 3))) for _ in range(n)]


@pytest.fixture(scope="module")
def cal(cc):
    """C2 camera with 40 views (k = -0.12)."""
    return cc.Calibration(C2_INTR[:4], _poses(40, 1), 1.0, C2_INTR[4], [f"{i}.png" for i in range(40)])


def _points(kind, dt, n, in_dim, seed):
    """(n, in_dim) interleaved numpy points."""
    rng = np.random.default_rng(seed)
    if kind == "img2world":
        cols = [rng.uniform(1, 1080, n), rng.uniform(1, 1920, n)]
    else:
        cols = [rng.uniform(-2, 20, n), rng.uniform(-2, 14, n), rng.uniform(-0.5, 0.5, n)][:in_dim]
    return np.stack(cols, -1).astype(dt)


def _sfx(dt):
    return "f64" if np.dtype(dt) == np.float64 else "f32"


def _buf(n_elems, dt, host, shift=0):
    """A sentinel-filled 1-D buffer with GUARD elements on each side (plus `shift` more in front)."""
    total = n_elems + 2 * GUARD + shift
    if host:
        return np.full(total, SENTINEL, dtype=dt)
    return torch.full((total,), SENTINEL, dtype=torch.float64 if np.dtype(dt) == np.float64 else torch.float32,
                      device="cuda")


def _np(a):
    return a.cpu().numpy() if torch.is_tensor(a) else a


def _ptr(a, elem=0):
    if a is None:
        return None
    if torch.is_tensor(a):
        return C.c_void_p(a.data_ptr() + elem * a.element_size())
    return C.c_void_p(a.ctypes.data + elem * a.itemsize)


def _raw(cal, kind, dt, host, views, offsets, src, src_at, dst, dst_at, dim, n, nviews=None):
    """One cc_{kind}_{sfx}_aos[_host] call; src / dst are buffers, the arrays start at element src_at / dst_at."""
    from cameracalibrations_b200 import _lib
    v = (_lib.View * max(1, len(views)))(*[cal._views[i] for i in views]) if views is not None else None
    o = (C.c_size_t * len(offsets))(*offsets) if offsets is not None else None
    nv = (len(views) if views is not None else 1) if nviews is None else nviews
    io = (_ptr(src, src_at), _ptr(dst, dst_at), dim) if kind == "img2world" else (_ptr(src, src_at), dim,
                                                                                  _ptr(dst, dst_at))
    fn = getattr(_lib.lib, f"cc_{kind}_{_sfx(dt)}_aos" + ("_host" if host else ""))
    args = [_lib.context(0).handle, C.byref(cal._intr), v, nv, o, *io, C.c_size_t(n)]
    if not host:
        args.append(C.c_void_p(torch.cuda.current_stream().cuda_stream))
    return fn(*args)


def _soa(cal, kind, pts, views, counts, dim):
    """The SoA entry points on the same points: single view when counts is None, else the _views form.
    Returns the result interleaved as (n, out_dim) numpy."""
    cols = [np.ascontiguousarray(pts[:, d]) for d in range(pts.shape[1])]
    if kind == "img2world":
        if counts is None:
            outs = cal.img2world(cols[0], cols[1], views[0], want_z=dim == 3)
        else:
            outs = cal.img2world_views(cols[0], cols[1], views, counts, want_z=dim == 3)
    else:
        z = cols[2] if dim == 3 else None
        if counts is None:
            outs = cal.world2img(cols[0], cols[1], z, views[0])
        else:
            outs = cal.world2img_views(cols[0], cols[1], z, views, counts)
    return np.stack(outs, -1)


def _check(cal, kind, dt, dim, host, pts, views, counts, shift_in=0, shift_out=0):
    """AoS call (offsets = None when counts is None) against the SoA entry point, bit for bit, with the guard
    elements around the output untouched."""
    n = pts.shape[0]
    in_dim, out_dim = (2, dim) if kind == "img2world" else (dim, 2)
    src = _buf(n * in_dim, dt, host, shift_in)
    _np_src = np.full(src.shape, SENTINEL, dtype=dt)
    _np_src[GUARD + shift_in:GUARD + shift_in + n * in_dim] = pts.ravel()
    if host:
        src[:] = _np_src
    else:
        src.copy_(torch.from_numpy(_np_src))
    dst = _buf(n * out_dim, dt, host, shift_out)
    offsets = None if counts is None else [0] + np.cumsum(counts).tolist()
    assert _raw(cal, kind, dt, host, views, offsets, src, GUARD + shift_in, dst, GUARD + shift_out, dim, n) == 0
    torch.cuda.synchronize()
    got = _np(dst)
    lo, hi = GUARD + shift_out, GUARD + shift_out + n * out_dim
    assert np.all(got[:lo] == SENTINEL) and np.all(got[hi:] == SENTINEL), "written outside the output"
    if n:
        ref = _soa(cal, kind, pts, views, counts, dim)
        assert np.array_equal(got[lo:hi].reshape(n, out_dim), ref), (kind, n)


CASES = [(k, dt, d) for k in ("img2world", "world2img") for dt in (np.float64, np.float32) for d in (3, 2)]


def _ids(c):
    return f"{c[0]}-{np.dtype(c[1]).name}-{c[2]}"


# ---------------------------------------------------------------- bit-identity with SoA
@pytest.mark.gpu
@pytest.mark.parametrize("case", CASES, ids=_ids)
@pytest.mark.parametrize("host", [False, True], ids=["device", "host"])
def test_single_view_bit_identical(cal, case, host):
    kind, dt, dim = case
    in_dim = 2 if kind == "img2world" else dim
    for n in SIZES:
        _check(cal, kind, dt, dim, host, _points(kind, dt, n, in_dim, n), [7], None)


@pytest.mark.gpu
@pytest.mark.parametrize("case", CASES, ids=_ids)
@pytest.mark.parametrize("host", [False, True], ids=["device", "host"])
def test_segments_bit_identical(cal, case, host):
    """Small segments (every boundary residue, empty segments, a view in non-adjacent segments), 10 000 x 280,
    and one segment holding every point between empty ones (the single-view kernel)."""
    kind, dt, dim = case
    in_dim = 2 if kind == "img2world" else dim
    rng = np.random.default_rng(5)
    layouts = [(SMALL_VIEWS, SMALL_COUNTS),
               (rng.integers(0, 40, 10_000).tolist(), [280] * 10_000),
               ([3, 9, 4], [0, 4097, 0])]
    for i, (views, counts) in enumerate(layouts):
        _check(cal, kind, dt, dim, host, _points(kind, dt, sum(counts), in_dim, 20 + i), views, counts)


@pytest.mark.gpu
@pytest.mark.parametrize("case", CASES, ids=_ids)
def test_unaligned_bases_bit_identical(cal, case):
    """Input and output one element (8 / 4 bytes) off 16-byte alignment: the scalar path, same bits."""
    kind, dt, dim = case
    in_dim = 2 if kind == "img2world" else dim
    for n in (5, 4097):
        pts = _points(kind, dt, n, in_dim, 40 + n)
        for si, so in ((1, 0), (0, 1), (1, 1)):
            _check(cal, kind, dt, dim, False, pts, [2], None, si, so)
            _check(cal, kind, dt, dim, False, pts, SMALL_VIEWS[:3], [1, n - 3, 2], si, so)


@pytest.mark.gpu
@pytest.mark.parametrize("case", [c for c in CASES if c[2] == 3], ids=_ids)
def test_host_chunk_boundaries(cal, case):
    """Host pipeline over more than one chunk with an odd remainder: one view, then chunk boundaries inside
    segments."""
    kind, dt, dim = case
    in_dim = 2 if kind == "img2world" else dim
    _check(cal, kind, dt, dim, True, _points(kind, dt, CHUNK + 12_345, in_dim, 50), [4], None)
    counts = [5, 3 * CHUNK - 2, 3, 0, 1, CHUNK + 7, 2, 1_001]
    views = [1, 2, 3, 4, 1, 5, 2, 6]
    _check(cal, kind, dt, dim, True, _points(kind, dt, sum(counts), in_dim, 51), views, counts)


# ---------------------------------------------------------------- against the oracle
@pytest.mark.gpu
@pytest.mark.parametrize("host", [False, True], ids=["device", "host"])
def test_example_fit_views_against_oracle(cc, example_fit, host):
    """The six example-fit views through c(list, views): FP64 world->pixel bit-exact to the oracle, pixel->world
    within 1e-9 (scaled)."""
    from oracle import oracle_c as oc
    intr = example_fit["intr_tuple"]
    c = cc.Calibration(intr[:4], example_fit["view_list"], 1.0 / intr[5], intr[4], example_fit["files"])
    nv = len(example_fit["view_list"])
    chains = [oc.chain(intr, *v) for v in example_fit["view_list"]]
    obj = example_fit["obj_np"]
    rng = np.random.default_rng(21)
    dev = (lambda a: torch.from_numpy(np.ascontiguousarray(a)).cuda()) if not host else np.ascontiguousarray
    xyz = [np.concatenate([obj, np.stack([rng.uniform(-2, 10, 1000 * v), rng.uniform(-2, 7, 1000 * v),
                                          rng.uniform(-0.2, 0.2, 1000 * v)], -1)]) for v in range(nv)]
    rcs = c([dev(p) for p in xyz], list(range(nv)))
    for v in range(nv):
        orow, ocol = oc.world2img_soa(chains[v], xyz[v][:, 0], xyz[v][:, 1], xyz[v][:, 2])
        assert np.array_equal(_np(rcs[v]), np.stack([orow, ocol], -1))
        one = _np(c(dev(xyz[v]), v))
        assert np.array_equal(one, np.stack([orow, ocol], -1))
    rc = [np.concatenate([example_fit["corners_np"][v], np.stack([rng.uniform(1, 375, 1000 * v),
                                                                  rng.uniform(1, 500, 1000 * v)], -1)])
          for v in range(nv)]
    ws = c([dev(p) for p in rc], list(range(nv)))
    for v in range(nv):
        o = np.stack(oc.img2world_soa(chains[v], rc[v][:, 0], rc[v][:, 1]), -1)
        scale = max(1.0, float(np.max(np.abs(o[:, :2]))))
        assert np.max(np.abs(_np(ws[v]) - o)) <= 1e-9 * scale


# ---------------------------------------------------------------- launches, errors
@pytest.mark.gpu
@pytest.mark.parametrize("nviews", [1, 64, 10_000])
def test_one_launch_per_device_call(cc, cal, nviews):
    ctx = cc.context(0)
    rng = np.random.default_rng(nviews)
    views = rng.integers(0, 40, nviews).tolist()
    counts = rng.integers(0, 300, nviews).tolist()
    n = sum(counts)
    offsets = [0] + np.cumsum(counts).tolist()
    src = torch.from_numpy(_points("world2img", np.float64, n, 3, 3)).cuda()
    dst = torch.empty(3 * n + 1, dtype=torch.float64, device="cuda")
    for kind, offs in (("img2world", offsets), ("world2img", offsets), ("img2world", None)):
        vs = views if offs is not None else views[:1]
        before = ctx.launch_count()
        assert _raw(cal, kind, np.float64, False, vs, offs, src, 0, dst, 0, 3, n) == 0
        assert ctx.launch_count() == before + 1
    before = ctx.launch_count()
    assert _raw(cal, "img2world", np.float64, False, views, [0] * (nviews + 1), None, 0, None, 0, 3, 0) == 0
    assert _raw(cal, "world2img", np.float64, False, [0], None, None, 0, None, 0, 2, 0) == 0
    e = torch.empty((0, 2), dtype=torch.float64, device="cuda")
    assert cal(e, 0).shape == (0, 3)
    assert ctx.launch_count() == before


@pytest.mark.gpu
@pytest.mark.parametrize("kind", ["img2world", "world2img"])
@pytest.mark.parametrize("dt", [np.float64, np.float32], ids=["f64", "f32"])
@pytest.mark.parametrize("host", [False, True], ids=["device", "host"])
def test_argument_errors_write_nothing(cc, cal, kind, dt, host):
    from cameracalibrations_b200 import _lib
    n = 8
    src = _buf(3 * n, dt, host)
    dst = _buf(3 * n, dt, host)
    ok = ([0, 1], [0, 3, 8])

    def call(views=ok[0], offsets=ok[1], dim=3, nn=n, s=src, d=dst, nviews=None):
        return _raw(cal, kind, dt, host, views, offsets, s, 0, d, 0, dim, nn, nviews)

    cases = [
        (dict(dim=4), "out_dim / in_dim"),
        (dict(dim=1), "out_dim / in_dim"),
        (dict(s=None), "NULL point array"),
        (dict(d=None), "NULL point array"),
        (dict(offsets=None), "nviews == 1"),
        (dict(nn=7), "offsets[nviews]"),
        (dict(nviews=0), "nviews"),
        (dict(views=None), "NULL"),
        (dict(offsets=[1, 3, 8]), "offsets[0]"),
        (dict(offsets=[0, 3, 2], nn=2), "decrease"),
        (dict(views=None, offsets=None, nviews=1), "view is NULL"),
    ]
    for kw, msg in cases:
        assert call(**kw) == -1, kw
        assert msg in _lib.last_error(), (kw, _lib.last_error())
    for field, msg in (("frow", "focal"), ("checker_size", "checker_size")):
        saved = getattr(cal._intr, field)
        setattr(cal._intr, field, 0.0)
        try:
            assert call() == -1 and msg in _lib.last_error()
            assert call(offsets=None, views=[0]) == -1 and msg in _lib.last_error()
        finally:
            setattr(cal._intr, field, saved)
    torch.cuda.synchronize()
    assert np.all(_np(dst) == SENTINEL)
    assert call() == 0
    assert call(offsets=None, views=[1]) == 0
    assert call(offsets=[0, 0, 0], nn=0, s=None, d=None) == 0          # n == 0: no point array needed


# ---------------------------------------------------------------- the Python layer
@pytest.mark.gpu
@pytest.mark.parametrize("dt", [np.float64, np.float32], ids=["f64", "f32"])
@pytest.mark.parametrize("on_dev", [False, True], ids=["numpy", "cuda"])
def test_python_layer_matches_soa_methods(cal, dt, on_dev):
    """c(pts, i), rectification(c, i) and c(list, views) against the SoA methods: same values, shapes, dtypes;
    C-contiguous, non-contiguous and odd-offset inputs."""
    import cameracalibrations_b200 as m
    rng = np.random.default_rng(3)
    rc = np.stack([rng.uniform(1, 1080, (7, 9)), rng.uniform(1, 1920, (7, 9))], -1).astype(dt)
    to = (lambda a: torch.from_numpy(np.ascontiguousarray(a)).cuda()) if on_dev else (lambda a: a)
    want_dt = torch.float64 if dt == np.float64 else torch.float32
    for inp in (to(rc), to(rc).transpose(0, 1) if on_dev else rc.transpose(1, 0, 2), to(rc)[1:]):
        flat = _np(inp).reshape(-1, 2)
        x, y, z = cal.img2world(flat[:, 0].copy(), flat[:, 1].copy(), 5)
        got = cal(inp, 5)
        assert got.shape == tuple(inp.shape[:-1]) + (3,)
        assert (got.dtype == want_dt) if on_dev else (got.dtype == dt)
        assert np.array_equal(_np(got).reshape(-1, 3), np.stack([x, y, z], -1))
        r = m.rectification(cal, 5)(inp)
        assert r.shape == tuple(inp.shape[:-1]) + (2,)
        assert np.array_equal(_np(r).reshape(-1, 2), np.stack([x, y], -1))
        back = cal(got, 5)
        fx = _np(got).reshape(-1, 3)
        rr, cc_ = cal.world2img(fx[:, 0].copy(), fx[:, 1].copy(), fx[:, 2].copy(), 5)
        assert back.shape == tuple(inp.shape[:-1]) + (2,)
        assert np.array_equal(_np(back).reshape(-1, 2), np.stack([rr, cc_], -1))
    # the list form: slices of one output
    pts = [to(rc[i]) for i in range(4)]
    outs = cal(pts, [3, 1, "5.png", 3])
    for p, v, o in zip(pts, [3, 1, "5.png", 3], outs):
        assert o.shape == (p.shape[0], 3)
        assert np.array_equal(_np(o), _np(cal(p, v)))
    # a single point
    assert cal(to(rc[0, 0]), 2).shape == (3,)


# ---------------------------------------------------------------- CPU
def test_aos_symbols_declared_and_bound():
    from cameracalibrations_b200 import _lib
    names = {f"cc_{k}_{p}_aos{h}" for k in ("img2world", "world2img") for p in ("f64", "f32") for h in ("", "_host")}
    hdr = _header_params()
    for n in names:
        assert n in hdr and n in _lib.EXPORTS and hasattr(_lib.lib, n), n
        assert hdr[n] == ["ptr", "ptr", "ptr", "scalar", "ptr"] + (
            ["ptr", "ptr", "scalar"] if "img2world" in n else ["ptr", "scalar", "ptr"]) + ["scalar"] + (
            [] if n.endswith("_host") else ["ptr"]), (n, hdr[n])


def test_aos_entry_points_need_a_device():
    """Bad arguments are rejected before the device is touched; good ones fail with CC_ERR_NO_DEVICE.  The
    context is a zeroed stand-in: without a device the library reads nothing from it but the device index."""
    if torch.cuda.is_available():
        pytest.skip("a device is present")
    import cameracalibrations_b200 as m
    from cameracalibrations_b200 import _lib
    c = m.Calibration((100.0, 100.0, 50.0, 50.0), [((0, 0, 0), (0, 0, 1.0))] * 2, 1.0, 0.0, ["a", "b"])
    fake = C.create_string_buffer(1 << 16)
    views = (_lib.View * 2)(*c._views)
    for kind in ("img2world", "world2img"):
        for p, dt in (("f64", np.float64), ("f32", np.float32)):
            for host in ("", "_host"):
                fn = getattr(_lib.lib, f"cc_{kind}_{p}_aos{host}")
                a, b = np.zeros(12, dt), np.zeros(12, dt)

                def call(dim=3, offs=None, nv=1, src=a, n=4):
                    o = (C.c_size_t * len(offs))(*offs) if offs is not None else None
                    io = (_ptr(src), _ptr(b), dim) if kind == "img2world" else (_ptr(src), dim, _ptr(b))
                    return fn(fake, C.byref(c._intr), views, nv, o, *io, C.c_size_t(n), *(() if host else (None,)))

                for kw in (dict(dim=4), dict(src=None), dict(nv=2), dict(offs=[0, 1, 3], nv=2),
                           dict(offs=[0, 3, 1], nv=2)):
                    assert call(**kw) == -1, (fn, kw)
                assert call() == -2 and call(offs=[0, 1, 4], nv=2) == -2 and call(dim=2) == -2, fn
    for call in (lambda: c(np.zeros((4, 2)), 0), lambda: c(np.zeros((2, 4, 3), np.float32), 1),
                 lambda: m.rectification(c, 0)(np.zeros((3, 2))), lambda: c([np.zeros((3, 2)), np.zeros((1, 2))], [0, 1])):
        with pytest.raises(m.CamcalError) as e:
            call()
        assert e.value.status == -2                      # CC_ERR_NO_DEVICE
    with pytest.raises(TypeError):
        c(np.zeros((4, 4)), 0)
    with pytest.raises(TypeError):
        c(torch.zeros((4, 2), dtype=torch.float64), 0)   # CPU tensors do not take the host path


def test_julia_aos_ccalls_match_the_header():
    hdr = _header_params()
    calls = [(n, k) for n, k in _julia_ccalls() if "_aos" in n]
    assert {n for n, _ in calls} == {"cc_img2world_f64_aos_host", "cc_world2img_f64_aos_host"}
    assert len(calls) == 4                               # one view, and many views, per direction
    for name, kinds in calls:
        assert kinds == hdr[name], (name, kinds, hdr[name])
