"""Point maps over many views in one call: cc_img2world_* / cc_world2img_* `_views` (device, one launch)
and `_views_host` (chunked pipeline).  Every segment's result must be bit-identical to the single-view
entry point called with that segment's view; against the oracle at the single-view tolerances.

The CPU tests at the end need no device."""
import ctypes as C

import numpy as np
import pytest

from conftest import C2_INTR, SYN_VIEW
from test_abi import _header_params, _julia_ccalls

torch = pytest.importorskip("torch")

CHUNK = 1 << 22                 # kPointChunk of csrc/abi.cu: points per host pipeline stage
SENTINEL = -7.25


@pytest.fixture(scope="module")
def cc():
    import cameracalibrations_b200 as m
    assert torch.cuda.is_available(), "GPU tests need a CUDA device"
    m.context(0)
    return m


def _poses(n, seed):
    """SYN_VIEW-like random poses: the board 25-35 units in front of the camera, tilted by < 0.3 rad."""
    rng = np.random.default_rng(seed)
    r0, t0 = np.asarray(SYN_VIEW[0]), np.asarray(SYN_VIEW[1])
    return [(tuple(r0 + rng.uniform(-0.15, 0.15, 3)), tuple(t0 + rng.uniform(-3, 3, 3))) for _ in range(n)]


@pytest.fixture(scope="module")
def cal(cc):
    """C2 camera with 40 views (k = -0.12)."""
    return cc.Calibration(C2_INTR[:4], _poses(40, 1), 1.0, C2_INTR[4], [f"{i}.png" for i in range(40)])


def _inputs(kind, dt, n, seed, torch_dev):
    rng = np.random.default_rng(seed)
    if kind == "img2world":
        a = [rng.uniform(1, 1080, n), rng.uniform(1, 1920, n)]
    else:
        a = [rng.uniform(-2, 20, n), rng.uniform(-2, 14, n), rng.uniform(-0.5, 0.5, n)]
    a = [x.astype(dt) for x in a]
    return [torch.from_numpy(x).cuda() for x in a] if torch_dev else a


def _run_views(cal, kind, ins, views, counts, with_z):
    if kind == "img2world":
        return cal.img2world_views(ins[0], ins[1], views, counts, want_z=with_z)
    return cal.world2img_views(ins[0], ins[1], ins[2] if with_z else None, views, counts)


def _run_single(cal, kind, ins, view, with_z):
    if kind == "img2world":
        return cal.img2world(ins[0], ins[1], view, want_z=with_z)
    return cal.world2img(ins[0], ins[1], ins[2] if with_z else None, view)


def _equal(a, b):
    return torch.equal(a, b) if torch.is_tensor(a) else np.array_equal(a, b)


def _check_segments(cal, kind, ins, views, counts, with_z, got=None):
    """The views call against one single-view call per segment, bit for bit."""
    got = _run_views(cal, kind, ins, views, counts, with_z) if got is None else got
    off = np.concatenate([[0], np.cumsum(counts)])
    for s, v in enumerate(views):
        a, b = int(off[s]), int(off[s + 1])
        if a == b:
            continue
        ref = _run_single(cal, kind, [t[a:b] for t in ins], v, with_z)
        for g, r in zip(got, ref):
            assert _equal(g[a:b], r), (kind, s, v, a, b)
    return got


SMALL_COUNTS = [0, 1, 2, 3, 0, 1, 1, 1, 4, 5, 6, 7, 0, 0, 9, 1, 130, 2, 3]   # ends at every residue mod 2 and 4
SMALL_VIEWS = [0, 1, 2, 0, 3, 1, 5, 2, 0, 7, 0, 9, 4, 4, 11, 0, 6, 3, 0]       # view 0 in non-adjacent segments

CASES = [(k, dt, z) for k in ("img2world", "world2img") for dt in (np.float64, np.float32) for z in (True, False)]


def _ids(c):
    return f"{c[0]}-{np.dtype(c[1]).name}-{'z' if c[2] else 'noz'}"


def test_small_layouts_residues():
    off = np.cumsum(SMALL_COUNTS)
    assert set(off % 4) == {0, 1, 2, 3} and set(off % 2) == {0, 1}


@pytest.mark.gpu
@pytest.mark.parametrize("case", CASES, ids=_ids)
@pytest.mark.parametrize("host", [False, True], ids=["device", "host"])
def test_small_segments_bit_identical(cal, case, host):
    kind, dt, with_z = case
    n = sum(SMALL_COUNTS)
    ins = _inputs(kind, dt, n, 11, not host)
    _check_segments(cal, kind, ins, SMALL_VIEWS, SMALL_COUNTS, with_z)
    # unaligned pointers: the scalar path, same bits
    if not host:
        ins1 = [t[1:] for t in ins]
        counts1 = list(SMALL_COUNTS)
        counts1[1] -= 1                                   # the segment of length 1 loses its point
        _check_segments(cal, kind, ins1, SMALL_VIEWS, counts1, with_z)


@pytest.mark.gpu
@pytest.mark.parametrize("case", CASES, ids=_ids)
@pytest.mark.parametrize("host", [False, True], ids=["device", "host"])
def test_c5_shape_bit_identical(cal, case, host):
    """10 000 segments x 280 points, views drawn at random from the calibration's 40 poses."""
    kind, dt, with_z = case
    rng = np.random.default_rng(5)
    views = rng.integers(0, 40, 10_000).tolist()
    counts = [280] * 10_000
    ins = _inputs(kind, dt, 280 * 10_000, 12, not host)
    _check_segments(cal, kind, ins, views, counts, with_z)


@pytest.mark.gpu
@pytest.mark.parametrize("case", CASES, ids=_ids)
def test_large_segments_bit_identical(cal, case):
    """64 segments of 1.5 M points (device)."""
    kind, dt, with_z = case
    views = [(7 * s) % 40 for s in range(64)]
    counts = [1_500_000] * 64
    ins = _inputs(kind, dt, sum(counts), 13, True)
    _check_segments(cal, kind, ins, views, counts, with_z)
    del ins
    torch.cuda.empty_cache()


@pytest.mark.gpu
@pytest.mark.parametrize("case", [c for c in CASES if c[2]], ids=_ids)
def test_host_chunk_boundaries_inside_segments(cal, case):
    """Host pipeline: one segment over three chunks, then chunk boundaries inside segments, with
    small segments around them."""
    kind, dt, with_z = case
    counts = [5, 3 * CHUNK - 2, 3, 0, 1, CHUNK + 7, 2, 1_000]
    views = [1, 2, 3, 4, 1, 5, 2, 6]
    ins = _inputs(kind, dt, sum(counts), 14, False)
    _check_segments(cal, kind, ins, views, counts, with_z)


# ---------------------------------------------------------------- against the oracle
@pytest.mark.gpu
@pytest.mark.parametrize("host", [False, True], ids=["device", "host"])
def test_example_fit_views_against_oracle(cc, example_fit, host):
    """The six example-fit views in one call: FP64 world->pixel bit-exact to the oracle, pixel->world within
    1e-9 (scaled), the FP32 round trip within 1e-3 px."""
    from oracle import oracle_c as oc
    intr = example_fit["intr_tuple"]
    c = cc.Calibration(intr[:4], example_fit["view_list"], 1.0 / intr[5], intr[4], example_fit["files"])
    nv = len(example_fit["view_list"])
    chains = [oc.chain(intr, *v) for v in example_fit["view_list"]]
    obj = example_fit["obj_np"]
    rng = np.random.default_rng(21)
    counts = [obj.shape[0] + 1000 * v for v in range(nv)]
    xs = [np.concatenate([obj[:, 0], rng.uniform(-2, 10, 1000 * v)]) for v in range(nv)]
    ys = [np.concatenate([obj[:, 1], rng.uniform(-2, 7, 1000 * v)]) for v in range(nv)]
    zs = [np.concatenate([obj[:, 2], rng.uniform(-0.2, 0.2, 1000 * v)]) for v in range(nv)]
    dev = (lambda a: torch.from_numpy(np.ascontiguousarray(a)).cuda()) if not host else np.ascontiguousarray
    back = (lambda t: t.cpu().numpy()) if not host else (lambda a: a)
    x, y, z = np.concatenate(xs), np.concatenate(ys), np.concatenate(zs)
    r, q = c.world2img_views(dev(x), dev(y), dev(z), list(range(nv)), counts)
    off = np.concatenate([[0], np.cumsum(counts)])
    for v in range(nv):
        orow, ocol = oc.world2img_soa(chains[v], xs[v], ys[v], zs[v])
        assert np.array_equal(back(r)[off[v]:off[v + 1]], orow) and np.array_equal(back(q)[off[v]:off[v + 1]], ocol)
    # pixel -> world on the detected corners plus random pixels
    pr = [np.concatenate([example_fit["corners_np"][v][:, 0], rng.uniform(1, 375, 1000 * v)]) for v in range(nv)]
    pc = [np.concatenate([example_fit["corners_np"][v][:, 1], rng.uniform(1, 500, 1000 * v)]) for v in range(nv)]
    gx, gy, gz = c.img2world_views(dev(np.concatenate(pr)), dev(np.concatenate(pc)), list(range(nv)), counts)
    for v in range(nv):
        ox, oy, oz = oc.img2world_soa(chains[v], pr[v], pc[v])
        scale = max(1.0, float(np.max(np.abs(ox))), float(np.max(np.abs(oy))))
        for g, o in ((gx, ox), (gy, oy), (gz, oz)):
            assert np.max(np.abs(back(g)[off[v]:off[v + 1]] - o)) <= 1e-9 * scale
    # FP32 round trip: pixel -> world (FP32 kernel) -> pixel (FP64 oracle)
    pr32, pc32 = [a.astype(np.float32) for a in pr], [a.astype(np.float32) for a in pc]
    fx, fy, fz = c.img2world_views(dev(np.concatenate(pr32)), dev(np.concatenate(pc32)), list(range(nv)), counts)
    for v in range(nv):
        sl = slice(off[v], off[v + 1])
        r64, c64 = oc.world2img_soa(chains[v], back(fx)[sl].astype(np.float64), back(fy)[sl].astype(np.float64),
                                    back(fz)[sl].astype(np.float64))
        assert np.max(np.maximum(np.abs(r64 - pr32[v]), np.abs(c64 - pc32[v]))) <= 1e-3


@pytest.mark.gpu
def test_list_call_returns_per_view_results(cc, cal):
    """c([pts_0, pts_1, ...], [v_0, v_1, ...]): one call, the list of per-view results."""
    rng = np.random.default_rng(8)
    pts = [np.stack([rng.uniform(1, 1080, n), rng.uniform(1, 1920, n)], -1) for n in (7, 0, 300, 1)]
    views = [3, 1, "5.png", 3]
    out = cal(pts, views)
    assert len(out) == 4
    for p, v, o in zip(pts, views, out):
        assert o.shape == (p.shape[0], 3)
        assert np.array_equal(o, cal(p, v))
    back = cal([torch.from_numpy(o).cuda() for o in out], views)
    for o, v, b in zip(out, views, back):
        assert torch.equal(b, cal(torch.from_numpy(o).cuda(), v)) and b.shape == (o.shape[0], 2)


# ---------------------------------------------------------------- the C ABI directly
def _raw(cc, cal, fn_name, views, offsets, arrays, stream=None):
    from cameracalibrations_b200 import _lib
    v = (_lib.View * max(1, len(views)))(*[cal._views[i] for i in views]) if views is not None else None
    o = (C.c_size_t * len(offsets))(*offsets) if offsets is not None else None
    ptrs = [None if a is None else C.c_void_p(a.data_ptr() if torch.is_tensor(a) else a.ctypes.data) for a in arrays]
    fn = getattr(_lib.lib, fn_name)
    args = [_lib.context(0).handle, C.byref(cal._intr), v, len(views) if views is not None else 1, o, *ptrs]
    if not fn_name.endswith("_host"):
        args.append(C.c_void_p(torch.cuda.current_stream().cuda_stream if stream is None else stream))
    return fn(*args)


@pytest.mark.gpu
@pytest.mark.parametrize("nviews", [1, 64, 10_000])
def test_one_launch_per_device_call(cc, cal, nviews):
    ctx = cc.context(0)
    rng = np.random.default_rng(nviews)
    views = rng.integers(0, 40, nviews).tolist()
    counts = rng.integers(0, 300, nviews).tolist()
    n = sum(counts)
    row, col = _inputs("img2world", np.float64, n, 3, True)
    for kind, ins in (("img2world", (row, col)), ("world2img", (row, col, None))):
        before = ctx.launch_count()
        _run_views(cal, kind, ins, views, counts, kind == "img2world")
        assert ctx.launch_count() == before + 1
    before = ctx.launch_count()
    e = torch.empty(0, dtype=torch.float64, device="cuda")
    x, y, z = cal.img2world_views(e, e, views, [0] * nviews)
    assert x.numel() == 0 and ctx.launch_count() == before


@pytest.mark.gpu
@pytest.mark.parametrize("dt", [torch.float64, torch.float32], ids=["f64", "f32"])
@pytest.mark.parametrize("host", [False, True], ids=["device", "host"])
def test_nothing_written_outside_the_output(cc, cal, dt, host):
    sfx = ("f64" if dt == torch.float64 else "f32") + "_views" + ("_host" if host else "")
    counts = [3, 0, 17, 1, 2]
    views = [0, 1, 2, 3, 0]
    n = sum(counts)
    offs = [0] + np.cumsum(counts).tolist()
    mk = (lambda: torch.full((n + 16,), SENTINEL, dtype=dt, device="cuda")) if not host else \
         (lambda: np.full(n + 16, SENTINEL, dtype=np.float64 if dt == torch.float64 else np.float32))
    ins = _inputs("world2img", np.float64 if dt == torch.float64 else np.float32, n, 4, not host)
    outs = [mk() for _ in range(3)]
    assert _raw(cc, cal, f"cc_img2world_{sfx}", views, offs, [ins[0], ins[1], *outs]) == 0
    outs2 = [mk() for _ in range(2)]
    assert _raw(cc, cal, f"cc_world2img_{sfx}", views, offs, [*ins, *outs2]) == 0
    torch.cuda.synchronize()
    for o in outs + outs2:
        tail = o[n:].cpu().numpy() if torch.is_tensor(o) else o[n:]
        assert np.all(tail == SENTINEL)
        head = o[:n].cpu().numpy() if torch.is_tensor(o) else o[:n]
        assert not np.any(head == SENTINEL)
    # a rejected call writes nothing
    outs3 = [mk() for _ in range(3)]
    bad = [0, 3, 2] + offs[3:]                             # offsets decrease
    assert _raw(cc, cal, f"cc_img2world_{sfx}", views, bad, [ins[0], ins[1], *outs3]) == -1
    torch.cuda.synchronize()
    for o in outs3:
        assert np.all((o.cpu().numpy() if torch.is_tensor(o) else o) == SENTINEL)


@pytest.mark.gpu
def test_table_reuse_across_streams(cc, cal):
    """Back-to-back calls on two streams with no synchronisation, then a larger table on the first stream
    (the context's table grows): all three equal the single-view results."""
    rng = np.random.default_rng(9)
    s1, s2 = torch.cuda.Stream(), torch.cuda.Stream()
    layouts = [(rng.integers(0, 40, 37).tolist(), rng.integers(0, 20_000, 37).tolist()),
               (rng.integers(0, 40, 5).tolist(), rng.integers(100_000, 400_000, 5).tolist()),
               (rng.integers(0, 40, 30_000).tolist(), rng.integers(0, 60, 30_000).tolist())]
    ins = [_inputs("img2world", np.float64, sum(c), 30 + i, True) for i, (_, c) in enumerate(layouts)]
    torch.cuda.synchronize()
    got = []
    for (views, counts), x, st in zip(layouts, ins, (s1, s2, s1)):
        with torch.cuda.stream(st):
            got.append(cal.img2world_views(x[0], x[1], views, counts))
    torch.cuda.synchronize()
    for (views, counts), x, g in zip(layouts, ins, got):
        _check_segments(cal, "img2world", x, views, counts, True, got=g)


@pytest.mark.gpu
@pytest.mark.parametrize("fn", ["cc_img2world_f64_views", "cc_img2world_f64_views_host",
                                "cc_world2img_f32_views", "cc_world2img_f32_views_host"])
def test_argument_errors(cc, cal, fn):
    from cameracalibrations_b200 import _lib
    dt = torch.float64 if "f64" in fn else torch.float32
    host = fn.endswith("_host")
    mk = (lambda: torch.zeros(8, dtype=dt, device="cuda")) if not host else \
         (lambda: np.zeros(8, dtype=np.float64 if dt == torch.float64 else np.float32))
    arrs = [mk() for _ in range(5)]
    ok = ([0, 1], [0, 3, 8])

    def call(views, offsets, arrays=arrs, nviews=None):
        v = (_lib.View * 2)(*[cal._views[i] for i in ok[0]]) if views else None
        o = (C.c_size_t * len(offsets))(*offsets) if offsets is not None else None
        ptrs = [None if a is None else C.c_void_p(a.data_ptr() if torch.is_tensor(a) else a.ctypes.data) for a in arrays]
        args = [_lib.context(0).handle, C.byref(cal._intr), v, 2 if nviews is None else nviews, o, *ptrs]
        if not host:
            args.append(None)
        return getattr(_lib.lib, fn)(*args)

    cases = [
        (dict(views=True, offsets=ok[1], nviews=0), "nviews"),
        (dict(views=False, offsets=ok[1]), "NULL"),
        (dict(views=True, offsets=None), "NULL"),
        (dict(views=True, offsets=[1, 3, 8]), "offsets[0]"),
        (dict(views=True, offsets=[0, 3, 2]), "decrease"),
        (dict(views=True, offsets=ok[1], arrays=[None] + arrs[1:]), "NULL point array"),
    ]
    for kw, msg in cases:
        assert call(**kw) == -1, kw
        assert msg in _lib.last_error(), (kw, _lib.last_error())
    for field, msg in (("frow", "focal"), ("checker_size", "checker_size")):
        saved = getattr(cal._intr, field)
        setattr(cal._intr, field, 0.0)
        try:
            assert call(True, ok[1]) == -1 and msg in _lib.last_error()
        finally:
            setattr(cal._intr, field, saved)
    assert call(True, ok[1]) == 0
    # n == 0: no point array needed
    assert call(True, [0, 0, 0], arrays=[None] * 5) == 0


# ---------------------------------------------------------------- CPU
def test_python_layer_rejects_bad_views_and_counts(cc_cpu):
    c = cc_cpu.Calibration((1.0, 1.0, 0.0, 0.0), [((0, 0, 0), (0, 0, 1.0))] * 3, 1.0, 0.0, ["a", "b", "c"])
    with pytest.raises(IndexError):
        c.img2world_views(np.zeros(4), np.zeros(4), [0, 3], [2, 2])
    with pytest.raises(IndexError):
        c.world2img_views(np.zeros(4), np.zeros(4), None, [-1], [4])
    with pytest.raises(ValueError):
        c.img2world_views(np.zeros(4), np.zeros(4), [0, 1], [4])
    with pytest.raises(ValueError):
        c([np.zeros((2, 2))], [0, 1])


@pytest.fixture(scope="module")
def cc_cpu():
    import cameracalibrations_b200 as m
    return m


def test_views_entry_points_need_a_device(cc_cpu):
    if torch.cuda.is_available():
        pytest.skip("a device is present")
    c = cc_cpu.Calibration((100.0, 100.0, 50.0, 50.0), [((0, 0, 0), (0, 0, 1.0))] * 2, 1.0, 0.0, ["a", "b"])
    for call in (lambda: c.img2world_views(np.zeros(4), np.zeros(4), [0, 1], [1, 3]),
                 lambda: c.world2img_views(np.zeros(4, np.float32), np.zeros(4, np.float32), None, [1, 0], [4, 0]),
                 lambda: c([np.zeros((3, 2)), np.zeros((1, 2))], [0, 1])):
        with pytest.raises(cc_cpu.CamcalError) as e:
            call()
        assert e.value.status == -2                      # CC_ERR_NO_DEVICE


def test_julia_views_ccalls_match_the_header():
    hdr = _header_params()
    calls = [(n, k) for n, k in _julia_ccalls() if n.endswith("_views_host")]
    assert {n for n, _ in calls} == {"cc_img2world_f64_views_host", "cc_world2img_f64_views_host"}
    for name, kinds in calls:
        assert name in hdr, name
        assert kinds == hdr[name], (name, kinds, hdr[name])
