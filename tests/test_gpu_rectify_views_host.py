"""Frames of many views from host memory in one call: cc_rectify_views_f32c1_host / cc_rectify_views_u8c3_host.

The host form runs the chunk pipeline of cc_rectify_*_host over the frame axis of the whole call.  A chunk may start
or end inside a view and span two 64-view groups; it makes one staged launch per group it touches, over the window
of that group's frames it holds (rectify_ring.cuh: the VIEWS producer's frame window).  Every frame differs, every
output is prefilled with a sentinel; exact coordinates are compared with the oracle bit for bit, fast coordinates
with the device call cc_rectify_*_views on the same frames, bit for bit.  The path each case takes is asserted from
the `[camcal] staged:` lines of CAMCAL_DEBUG and the context's launch counter.
"""
import ctypes as C
import re

import numpy as np
import pytest

torch = pytest.importorskip("torch")

from conftest import camera_for
from oracle import oracle_c as oc
from test_gpu_batching import (F_FILL, F_SENT, U_FILL, U_SENT, _env, _frames_f32, _frames_u8, _staged_lines)
from test_gpu_parity import _calib, _dev, _perturbed_views, _rect_case
from test_abi import _header_params, _julia_ccalls

GROUP = 64                    # views per staged launch (rectify.cu: kMaxViews)
_FOOTPRINT = re.compile(r"\[camcal\] views: common footprint")


@pytest.fixture(scope="module")
def cc():
    import cameracalibrations_b200 as m
    assert torch.cuda.is_available(), "GPU tests need a CUDA device"
    m.context(0)
    return m


class _Views:
    """nv perturbed views of one frame size with their ratios and axes (scale: a distinct ratio family, so that
    the plans of one test are not those of another)"""

    def __init__(self, cc, nv, sz, scale=0.01, views=None):
        self.cc, self.nv, self.sz = cc, nv, sz
        self.intr = camera_for(sz)
        self.views = views if views is not None else _perturbed_views(nv)
        self.c = _calib(cc, self.intr, self.views)
        self.ratios, self.axss = [], []
        for vi in range(nv):
            _, _, ratio, axs = _rect_case(self.intr, sz, ratio_scale=1.0 + scale * (vi % 5), view=self.views[vi])
            self.ratios.append(ratio)
            self.axss.append(axs)

    def frames(self, fmt, n, seed):
        return _frames_f32(n, self.sz, seed) if fmt == "f32" else _frames_u8(n, self.sz, seed)

    def oracle(self, fmt, frames, fpv):
        rect = oc.rectify_f32c1 if fmt == "f32" else oc.rectify_u8c3
        return np.concatenate([rect(oc.chain(self.intr, *self.views[v]), 1.0 / self.ratios[v], self.axss[v],
                                    frames[v * fpv:(v + 1) * fpv], fill=_fill(fmt)) for v in range(self.nv)])

    def device(self, fmt, frames, coord):
        """cc_rectify_*_views on the same frames (device memory, the caller's stream)"""
        fd = _dev(frames)
        out = torch.empty_like(fd)
        out[...] = torch.tensor(_sent(fmt), dtype=out.dtype, device=out.device)
        self.cc.warp_views(self.c, list(range(self.nv)), fd, self.ratios, self.axss, fill=_fill(fmt), coord=coord,
                           out=out)
        return out.cpu().numpy()

    def host(self, fmt, frames, out, coord="f64", pitch=None, stride=None, fpv=None, flags=0, **over):
        """the raw ABI call on host buffers (dense unless pitch / stride are given); `over` replaces arguments"""
        from cameracalibrations_b200 import _lib
        nv = self.nv
        fpv = (frames.shape[0] // nv if frames.ndim > 1 else 1) if fpv is None else fpv
        pitch = self.sz[0] if pitch is None else pitch
        stride = pitch * self.sz[1] if stride is None else stride
        a = dict(ctx=self.cc.context(0).handle, intr=C.byref(self.c._intr),
                 views=(_lib.View * nv)(*[self.c._views[i] for i in range(nv)]), nviews=nv,
                 ratios=(C.c_double * nv)(*self.ratios), axs=(C.c_int64 * (2 * nv))(*[x for am in self.axss for x in am]),
                 src=C.c_void_p(frames.ctypes.data), dst=C.c_void_p(out.ctypes.data), sz1=self.sz[0], sz2=self.sz[1],
                 pitch=C.c_size_t(pitch), stride=C.c_size_t(stride), fpv=fpv,
                 fill=C.c_float(F_FILL) if fmt == "f32" else (C.c_uint8 * 3)(*U_FILL),
                 flags=(_lib.COORD_F32 if coord == "f32" else _lib.COORD_F64) | flags)
        a.update(over)
        fn = _lib.lib.cc_rectify_views_f32c1_host if fmt == "f32" else _lib.lib.cc_rectify_views_u8c3_host
        return fn(*a.values())


def _fill(fmt):
    return F_FILL if fmt == "f32" else U_FILL


def _sent(fmt):
    return F_SENT if fmt == "f32" else U_SENT


def _out_like(frames, fmt):
    out = np.empty_like(frames)
    out[...] = np.array(_sent(fmt), dtype=frames.dtype)
    return out


def _assert_equal(got, ref, what):
    assert got.shape == ref.shape, what
    for f in range(got.shape[0]):
        if got.dtype == np.float32:
            assert np.array_equal(got[f].view(np.uint32), ref[f].view(np.uint32)), (what, f)
        else:
            assert np.array_equal(got[f], ref[f]), (what, f)


def _chunks(nframes, frame_bytes, fpv, mb=32, ramp=True):
    """abi.cu, chunk_schedule: ~mb MB per chunk, at most 64 views' frames, the 1, 2, 4 ... / ... 4, 2, 1 ramp"""
    per = min(max(1, (mb << 20) // frame_bytes), GROUP * fpv, nframes)
    rf = rs = 0
    c = 1
    while ramp and c < per:
        rf, rs, c = rf + c, rs + 1, c * 2
    if 2 * rf + per > nframes:
        rf = rs = 0
    out, f0, it = [], 0, 0
    while f0 < nframes:
        left = nframes - f0
        if it < rs:
            m = 1 << it
        elif left > rf:
            m = min(per, left - rf)
        else:
            m = 1
            while 2 * m - 1 < left:
                m *= 2
        out.append(m)
        f0, it = f0 + m, it + 1
    return out


def _groups_per_chunk(chunks, fpv):
    """groups each chunk touches"""
    out, f0 = [], 0
    for m in chunks:
        out.append((f0 + m - 1) // (GROUP * fpv) - f0 // (GROUP * fpv) + 1)
        f0 += m
    return out


def _run(cc, capfd, vs, fmt, frames, coord, **kw):
    ctx = cc.context(0)
    out = _out_like(frames, fmt)
    n0 = ctx.launch_count()
    capfd.readouterr()
    with _env(CAMCAL_DEBUG="1"):
        rc = vs.host(fmt, frames, out, coord=coord, **kw)
    err = capfd.readouterr().err
    assert rc == 0, cc._lib.lib.cc_last_error_string()
    return out, ctx.launch_count() - n0, err


def _check(vs, fmt, coord, frames, out, fpv, what):
    if coord == "f64":
        _assert_equal(out, vs.oracle(fmt, frames, fpv), what)
    else:
        _assert_equal(out, vs.device(fmt, frames, coord), what)


# ------------------------------------------------------------------ the plot loop
@pytest.mark.gpu
@pytest.mark.parametrize("coord", ["f64", "f32"])
@pytest.mark.parametrize("fmt", ["f32", "u8"])
def test_plot_loop_example_fit(cc, capfd, example_fit, fmt, coord):
    """The six example_fit views, one frame each (src/plot_calibration.jl:36-42): one call, one staged launch."""
    intr = example_fit["intr_tuple"]
    sz = tuple(example_fit["sz"])
    vs = _Views(cc, len(example_fit["view_list"]), sz, views=example_fit["view_list"])
    vs.intr = intr
    vs.c = _calib(cc, intr, vs.views, example_fit["files"])
    vs.ratios, vs.axss = [], []
    for v in vs.views:
        _, _, ratio, axs = _rect_case(intr, sz, view=v)
        vs.ratios.append(ratio)
        vs.axss.append(axs)
    frames = vs.frames(fmt, vs.nv, 40)
    out, launches, err = _run(cc, capfd, vs, fmt, frames, coord)
    pxb = 4 if fmt == "f32" else 3
    chunks = _chunks(vs.nv, sz[0] * sz[1] * pxb, 1)
    if (sz[0] * pxb) % 16 == 0:                          # device lines TMA can address: one launch per chunk
        assert len(_staged_lines(err)) == launches == len(chunks), err[-2000:]
    else:                                                # 375-px lines: one launch per view, on the slot streams
        assert not _staged_lines(err) and launches == vs.nv, err[-2000:]
    _check(vs, fmt, coord, frames, out, 1, "example_fit")


# ------------------------------------------------------------------ groups and chunks
@pytest.mark.gpu
@pytest.mark.parametrize("coord", ["f64", "f32"])
@pytest.mark.parametrize("fmt", ["f32", "u8"])
def test_more_than_one_group(cc, capfd, fmt, coord):
    """130 views x 1 frame, 1 MB chunks: chunks cross the group boundaries at 64 and 128 views."""
    sz = (256, 192)
    vs = _Views(cc, 130, sz, scale=0.013)
    frames = vs.frames(fmt, 130, 300)
    with _env(CAMCAL_CHUNK_MB="1"):
        out, launches, err = _run(cc, capfd, vs, fmt, frames, coord)
    chunks = _chunks(130, sz[0] * sz[1] * (4 if fmt == "f32" else 3), 1, mb=1)
    per_chunk = _groups_per_chunk(chunks, 1)
    assert max(per_chunk) == 2, chunks                   # the case covers what it is written for
    assert len(_staged_lines(err)) == launches == sum(per_chunk), err[-2000:]
    _check(vs, fmt, coord, frames, out, 1, "130 views")


@pytest.mark.gpu
@pytest.mark.parametrize("coord", ["f64", "f32"])
@pytest.mark.parametrize("fmt", ["f32", "u8"])
@pytest.mark.parametrize("nv,fpv,ramp", [(3, 17, "1"), (3, 17, "0"), (5, 7, "1"), (5, 7, "0"), (2, 2, "1")])
def test_chunk_boundaries_inside_views(cc, capfd, nv, fpv, ramp, fmt, coord):
    """Chunks of a few frames start and end inside views; frame groups stay inside a view.  Every chunk makes
    exactly one staged launch (one group); 2 x 2 frames are too few for the ramp."""
    sz = (256, 192)
    vs = _Views(cc, nv, sz, scale=0.011)
    frames = vs.frames(fmt, nv * fpv, 500 + nv)
    with _env(CAMCAL_CHUNK_MB="1", CAMCAL_CHUNK_RAMP=ramp):
        out, launches, err = _run(cc, capfd, vs, fmt, frames, coord)
    chunks = _chunks(nv * fpv, sz[0] * sz[1] * (4 if fmt == "f32" else 3), fpv, mb=1, ramp=ramp == "1")
    assert len(chunks) > 1 or nv * fpv == 4, chunks
    assert len(_staged_lines(err)) == launches == len(chunks), err[-2000:]
    _check(vs, fmt, coord, frames, out, fpv, f"{nv}x{fpv}")


# ------------------------------------------------------------------ plans
@pytest.mark.gpu
@pytest.mark.parametrize("fmt", ["f32", "u8"])
def test_group_plans_once_per_call_and_warm(cc, capfd, fmt):
    """A cold call builds each group's plan once (one `common footprint` line per group, however many chunks
    read it); a warm second call with the same views builds none.  Both give the same frames."""
    sz = (256, 192)
    vs = _Views(cc, 100, sz, scale=0.017 if fmt == "f32" else 0.019)
    frames = vs.frames(fmt, 200, 700)
    with _env(CAMCAL_CHUNK_MB="1"):
        cold, _, err = _run(cc, capfd, vs, fmt, frames, "f64")
        assert len(_FOOTPRINT.findall(err)) == 2, err[-2000:]
        warm, _, err = _run(cc, capfd, vs, fmt, frames, "f64")
        assert not _FOOTPRINT.findall(err), err[-2000:]
    _assert_equal(warm, cold, "warm")
    _check(vs, fmt, "f64", frames, cold, 2, "cold")


# ------------------------------------------------------------------ layouts
@pytest.mark.gpu
@pytest.mark.parametrize("fmt", ["f32", "u8"])
@pytest.mark.parametrize("pad1,padf", [(4, 64), (3, 7)])
def test_strided_host_layouts(cc, capfd, fmt, pad1, padf):
    """pitch > sz1 and frame_stride > pitch * sz2 on the host: the frames are the dense results, the padding
    between lines and frames is never written.  Pad 4 stages (16-byte device lines); pad 3 runs per-view launches."""
    sz, nv, fpv = (252, 160), 4, 3
    vs = _Views(cc, nv, sz, scale=0.012)
    ch = 1 if fmt == "f32" else 3
    dt = np.float32 if fmt == "f32" else np.uint8
    nfr, pitch = nv * fpv, sz[0] + pad1
    stride = pitch * sz[1] + padf
    dense = vs.frames(fmt, nfr, 900)
    pad_in, pad_out = (777.0, 555.0) if fmt == "f32" else (77, 55)

    def frame_view(buf, f):
        v = buf[f * stride * ch: (f * stride + pitch * sz[1]) * ch].reshape((sz[1], pitch) + ((3,) if ch == 3 else ()))
        return v[:, :sz[0]]

    src = np.full(nfr * stride * ch, pad_in, dt)
    for f in range(nfr):
        frame_view(src, f)[...] = dense[f]
    dst = np.full(nfr * stride * ch, pad_out, dt)
    ctx = cc.context(0)
    n0 = ctx.launch_count()
    capfd.readouterr()
    with _env(CAMCAL_DEBUG="1"):
        assert vs.host(fmt, src, dst, pitch=pitch, stride=stride, fpv=fpv) == 0
    err = capfd.readouterr().err
    staged = ((pitch * ch * (4 if fmt == "f32" else 1)) % 16) == 0
    chunks = _chunks(nfr, pitch * sz[1] * ch * (4 if fmt == "f32" else 1), fpv)
    if staged:
        assert len(_staged_lines(err)) == ctx.launch_count() - n0 == len(chunks), err[-2000:]
    else:
        assert not _staged_lines(err) and ctx.launch_count() - n0 >= nv, err[-2000:]
    ref = vs.oracle(fmt, dense, fpv)
    seen = np.zeros(dst.shape, bool)
    for f in range(nfr):
        assert np.array_equal(frame_view(dst, f), ref[f]), f
        frame_view(seen, f)[...] = True
    assert np.all(dst[~seen] == pad_out)


@pytest.mark.gpu
@pytest.mark.parametrize("coord", ["f64", "f32"])
def test_1080p_u8c3_falls_back_on_the_slot_streams(cc, capfd, coord):
    """1080p u8c3 lines are 3240 bytes, which TMA cannot address: every chunk runs one launch per view it
    touches (on its own slot stream), no staged launch; still bit-exact."""
    sz, nv, fpv = (1080, 1920), 3, 2
    vs = _Views(cc, nv, sz, scale=0.014)
    frames = vs.frames("u8", nv * fpv, 1100)
    out, launches, err = _run(cc, capfd, vs, "u8", frames, coord)
    assert not _staged_lines(err), err[-2000:]
    chunks = _chunks(nv * fpv, sz[0] * sz[1] * 3, fpv)
    views_touched, f0 = 0, 0
    for m in chunks:
        views_touched += (f0 + m - 1) // fpv - f0 // fpv + 1
        f0 += m
    assert launches == views_touched, (launches, chunks)
    _check(vs, "u8", coord, frames, out, fpv, "1080p u8c3")


@pytest.mark.gpu
@pytest.mark.parametrize("fmt", ["f32", "u8"])
def test_gather_direct_and_repeated_views(cc, capfd, fmt):
    """CC_GATHER_DIRECT takes the per-view kernels; views that repeat (the same view at 0, 2, 3) are rectified
    with their own entry each time.  Both bit-exact."""
    from cameracalibrations_b200 import _lib
    sz = (256, 192)
    base = _perturbed_views(2)
    views = [base[0], base[1], base[0], base[0]]
    vs = _Views(cc, 4, sz, scale=0.0, views=views)
    frames = vs.frames(fmt, 8, 1300)
    out, launches, err = _run(cc, capfd, vs, fmt, frames, "f64")
    assert len(_staged_lines(err)) == launches, err[-2000:]
    _check(vs, fmt, "f64", frames, out, 2, "repeated")
    out, launches, err = _run(cc, capfd, vs, fmt, frames, "f64", flags=_lib.GATHER_DIRECT)
    assert not _staged_lines(err) and launches >= 4, err[-2000:]
    _check(vs, fmt, "f64", frames, out, 2, "direct")


# ------------------------------------------------------------------ interleaving
@pytest.mark.gpu
@pytest.mark.parametrize("coord", ["f64", "f32"])
@pytest.mark.parametrize("fmt", ["f32", "u8"])
def test_host_call_between_device_calls(cc, fmt, coord):
    """device _views (caller's stream, not synchronised) -> host form with the same groups -> device _views
    again: all three agree bit for bit.  65 views: a group of 64 and a group of one, whose plan is a one-view
    plan.  Before and after the host call, single-view warp calls of views 0..63 run on a side stream that is
    never synchronised until the end: their one-view plans push the last group's plan out of the cache, so the
    host call installs it again over a plan that a side-stream launch may still read.  Each single-view result
    equals its view's frames of the device call."""
    sz, nv = (256, 192), 65
    vs = _Views(cc, nv, sz, scale=0.015)
    frames = vs.frames(fmt, 2 * nv, 1500)
    fd = _dev(frames)
    outs = []
    for _ in range(2):
        o = torch.empty_like(fd)
        o[...] = torch.tensor(_sent(fmt), dtype=o.dtype, device=o.device)
        outs.append(o)
    side = torch.cuda.Stream()
    side.wait_stream(torch.cuda.current_stream())

    def singles():
        with torch.cuda.stream(side):
            return [cc.warp(vs.c, v, fd[2 * v:2 * v + 2], vs.ratios[v], vs.axss[v], fill=_fill(fmt), coord=coord)
                    for v in range(GROUP)]

    cc.warp_views(vs.c, list(range(nv)), fd, vs.ratios, vs.axss, fill=_fill(fmt), coord=coord, out=outs[0])
    before = singles()
    host = _out_like(frames, fmt)
    with _env(CAMCAL_CHUNK_MB="1"):
        assert vs.host(fmt, frames, host, coord=coord) == 0
    after = singles()
    cc.warp_views(vs.c, list(range(nv)), fd, vs.ratios, vs.axss, fill=_fill(fmt), coord=coord, out=outs[1])
    torch.cuda.synchronize()
    a, b = outs[0].cpu().numpy(), outs[1].cpu().numpy()
    _assert_equal(host, a, "host vs device before")
    _assert_equal(b, a, "device after vs before")
    for v in range(GROUP):
        _assert_equal(before[v].cpu().numpy(), a[2 * v:2 * v + 2], ("single before", v))
        _assert_equal(after[v].cpu().numpy(), a[2 * v:2 * v + 2], ("single after", v))
    if coord == "f64":
        _assert_equal(host, vs.oracle(fmt, frames, 2), "oracle")


# ------------------------------------------------------------------ Python
@pytest.mark.gpu
@pytest.mark.parametrize("coord", ["f64", "f32"])
@pytest.mark.parametrize("fmt", ["f32", "u8"])
def test_python_numpy_equals_cuda(cc, fmt, coord):
    sz = (256, 192)
    vs = _Views(cc, 5, sz, scale=0.018)
    frames = vs.frames(fmt, 10, 1900)
    got = cc.warp_views(vs.c, list(range(5)), frames, vs.ratios, vs.axss, fill=_fill(fmt), coord=coord)
    assert isinstance(got, np.ndarray)
    _assert_equal(got, vs.device(fmt, frames, coord), "numpy vs cuda")
    with pytest.raises(TypeError):
        cc.warp_views(vs.c, list(range(5)), torch.from_numpy(frames), vs.ratios, vs.axss)


# ------------------------------------------------------------------ CPU
def test_host_views_entry_points_need_a_device():
    import cameracalibrations_b200 as m
    from cameracalibrations_b200 import _lib
    for name in ("cc_rectify_views_f32c1_host", "cc_rectify_views_u8c3_host"):
        assert hasattr(_lib.lib, name), name
    if torch.cuda.is_available():
        pytest.skip("a device is present")
    c = m.Calibration((100.0, 100.0, 50.0, 50.0), [((0, 0, 0), (0, 0, 1.0))] * 2, 1.0, 0.0, ["a", "b"])
    for frames in (np.zeros((2, 8, 8), np.float32), np.zeros((4, 8, 8, 3), np.uint8)):
        with pytest.raises(m.CamcalError) as e:
            m.warp_views(c, [0, 1], frames, [1.0, 1.0], [(0, 0), (0, 0)])
        assert e.value.status == -2                      # CC_ERR_NO_DEVICE
    with pytest.raises(TypeError):
        m.warp_views(c, [0, 1], torch.zeros((2, 8, 8)), [1.0, 1.0], [(0, 0), (0, 0)])


def test_julia_host_views_ccalls_match_the_header():
    hdr = _header_params()
    calls = [(n, k) for n, k in _julia_ccalls() if n.startswith("cc_rectify_views_")]
    assert {n for n, _ in calls} == {"cc_rectify_views_f32c1_host", "cc_rectify_views_u8c3_host"}
    for name, kinds in calls:
        assert name in hdr, name
        assert kinds == hdr[name], (name, kinds, hdr[name])
