"""Rectification along the frame axis: frame groups (one tile map reused by the consecutive frames of a unit),
the two-frames-per-stage f32 kernels, several frame groups per view in the views kernels, strided layouts of
cc_rectify_*_views and the chunk pipeline of cc_rectify_*_host -- against the oracle, with a different frame in
every slot and the output prefilled with a sentinel, so that a frame taken from the wrong slot, a swapped pair,
a skipped odd end of a unit or a chunk written at the wrong place fails.

Every case asserts which path ran, from the `[camcal] staged:` line CAMCAL_DEBUG prints per launch (frames per
group, ring stages, shared memory) or from the context's launch counter, so that a change of the launcher's
rules fails here instead of quietly moving a case off the path it was written for.

  exact coordinates: bit-equal to oracle.rectify_f32c1 / rectify_u8c3, frame by frame
  fast coordinates:  bit-equal to the same frame rectified alone, and within the fast path's tolerance of
                     the oracle (f32: ramp frames reproduce the FP32 map within 5e-4; u8: +-1 LSB, rarely 2)
"""
import contextlib
import ctypes as C
import os
import re

import numpy as np
import pytest

torch = pytest.importorskip("torch")

from conftest import BENCH_VIEW, C2_INTR, C3_INTR, SYN_VIEW, camera_for
from oracle import oracle_c as oc
from test_gpu_parity import _calib, _dev, _perturbed_views, _rect_case

pytestmark = pytest.mark.gpu

F_FILL, F_SENT, F_SENT_ALONE = -3.0, -777.0, -555.0
U_FILL, U_SENT, U_SENT_ALONE = (9, 8, 7), (201, 202, 203), (101, 102, 103)
# most frames per group, rectify.cu (kFGf32Exact, kFGf32Fast, kFGu8Exact, kFGu8Fast): (pixel format, coordinates) -> fg_max
FG_MAX = {("f32", "f64"): 12, ("f32", "f32"): 4, ("u8", "f64"): 16, ("u8", "f32"): 16}
TILE = 32                     # output tile: 32 x 32 pixels, both pixel formats


@pytest.fixture(scope="module")
def cc():
    import cameracalibrations_b200 as m
    assert torch.cuda.is_available(), "GPU tests need a CUDA device"
    m.context(0)
    return m


@contextlib.contextmanager
def _env(**kv):
    """Set environment knobs the library reads at every call; restore the previous values."""
    old = {k: os.environ.get(k) for k in kv}
    os.environ.update(kv)
    try:
        yield
    finally:
        for k, v in old.items():
            if v is None:
                os.environ.pop(k, None)
            else:
                os.environ[k] = v


_STAGED = re.compile(r"\[camcal\] staged: box \d+x\d+ pitch \d+ \((\d+) B\) stages (\d+) units (\d+) "
                     r"\(fg (\d+)\) grid \d+ \(\d+/SM\) smem (\d+)")


def _staged_lines(err):
    return [dict(zip(("box_bytes", "stages", "units", "fg", "smem"), map(int, m))) for m in _STAGED.findall(err)]


def _one_staged(err):
    lines = _staged_lines(err)
    assert len(lines) == 1, err[-2000:]
    return lines[0]


def _tiles(sz):
    return -(-sz[0] // TILE) * -(-sz[1] // TILE)


def _mirror_fg(units_per_group, fg_max, n):
    """unit_cfg / views_window (rectify.cu): halve the group until there are ~8 units per resident CTA slot
    (sm_count * 48 units); units_per_group = tiles (x views) of one frame group."""
    want = torch.cuda.get_device_properties(0).multi_processor_count * 48
    fg = min(fg_max, n)
    while fg > 1 and units_per_group * -(-n // fg) < want:
        fg = (fg + 1) // 2
    return fg


def _check_ring(d, fmt, fg):
    """Stages and shared memory of the launch the debug line reports (rectify.cu, plan_tma and the launchers):
    a 48 KB ring of 2..8 boxes, at most 56 KB; f32 puts two frames in a stage when the ring holds >= 4 boxes and
    the units have >= 2 frames (rectify_f32c1_kernel, NF == 2).  Returns True when the pair kernel ran."""
    bb = d["box_bytes"]
    stages = min(8, max(2, 48 * 1024 // bb))
    while stages > 2 and stages * bb > 56 * 1024:
        stages -= 1
    if fmt == "u8":
        assert (d["stages"], d["smem"]) == (stages, stages * bb + 16), d
        return False
    nf = 2 if stages >= 4 and fg >= 2 else 1
    assert (d["stages"], d["smem"]) == (stages // nf, stages // nf * nf * bb), d
    return nf == 2


# ------------------------------------------------------------------ frames and checks
def _frames_f32(n, sz, seed, ramps=()):
    """frame i = uniform noise + i (a frame from the wrong slot is off by whole units); at the indices in
    `ramps` a row ramp and a column ramp, whose bilinear blend reproduces the sampled coordinate"""
    f = np.empty((n, sz[1], sz[0]), np.float32)
    for i in range(n):
        f[i] = np.random.default_rng(seed + i).random((sz[1], sz[0]), dtype=np.float32) + np.float32(i)
    for j, i in enumerate(ramps):
        if i < n:
            f[i] = (np.arange(1, sz[0] + 1, dtype=np.float32)[None, :] if j % 2 == 0
                    else np.arange(1, sz[1] + 1, dtype=np.float32)[:, None])
    return f


def _frames_u8(n, sz, seed):
    return np.stack([np.random.default_rng(seed + i).integers(0, 256, (sz[1], sz[0], 3), dtype=np.uint8)
                     for i in range(n)])


def _prefilled(like, fmt, sentinel):
    out = torch.empty_like(like)
    out[...] = torch.tensor(sentinel, dtype=out.dtype, device=out.device)
    return out


def _assert_exact(got, ref, fmt, what):
    for f in range(got.shape[0]):
        if fmt == "f32":
            assert np.array_equal(got[f].view(np.uint32), ref[f].view(np.uint32)), (what, f)
        else:
            assert np.array_equal(got[f], ref[f]), (what, f)
    if fmt == "f32":
        assert not np.any(got == F_SENT), what


def _assert_u8_fast_near(fast, ref, what):
    """+-1 LSB, rarely 2, where both sampled; fill decisions agree almost everywhere
    (test_gpu_parity.py::test_rectify_u8c3_staged_rotations_and_scales)"""
    fv = np.array(U_FILL, dtype=np.uint8)
    for f in range(fast.shape[0]):
        inb = np.any(ref[f] != fv, axis=-1)
        sampled = np.any(fast[f] != fv, axis=-1)
        both = inb & sampled
        assert both.mean() > 0.02, (what, f)
        d = np.abs(fast[f][both].astype(np.int16) - ref[f][both].astype(np.int16))
        assert d.max() <= 2 and (d > 1).mean() < 1e-3, (what, f, int(d.max()))
        assert (inb != sampled).mean() < 2e-3, (what, f)


class _Case:
    """One view and frame size with n distinct frames in both pixel formats, the oracle's results and, lazily,
    every frame rectified alone with fast coordinates."""

    def __init__(self, cc, sz, n, seed, intr=None, view=SYN_VIEW, ratio_scale=1.0, ramps=(1, 2)):
        self.cc, self.sz, self.n, self.ramps = cc, sz, n, ramps
        self.intr = intr or camera_for(sz)
        self.ch, _, self.ratio, self.axs = _rect_case(self.intr, sz, ratio_scale=ratio_scale, view=view)
        self.c = _calib(cc, self.intr, [view])
        self.seed = seed
        self._host, self._dev, self._ref, self._alone, self._map = {}, {}, {}, {}, None

    def host(self, fmt):
        if fmt not in self._host:
            self._host[fmt] = (_frames_f32(self.n, self.sz, self.seed, self.ramps) if fmt == "f32"
                               else _frames_u8(self.n, self.sz, self.seed + 1000))
        return self._host[fmt]

    def dev(self, fmt):
        if fmt not in self._dev:
            self._dev[fmt] = _dev(self.host(fmt))
        return self._dev[fmt]

    def fill(self, fmt):
        return F_FILL if fmt == "f32" else U_FILL

    def ref(self, fmt):
        if fmt not in self._ref:
            rect = oc.rectify_f32c1 if fmt == "f32" else oc.rectify_u8c3
            self._ref[fmt] = rect(self.ch, 1.0 / self.ratio, self.axs, self.host(fmt), fill=self.fill(fmt))
        return self._ref[fmt]

    def warp(self, fmt, coord, n, sentinel):
        fd = self.dev(fmt)[:n]
        out = _prefilled(fd, fmt, sentinel)
        self.cc.warp(self.c, 0, fd, self.ratio, self.axs, fill=self.fill(fmt), coord=coord, out=out)
        return out

    def alone(self, fmt):
        """fast coordinates, every frame in a call of its own (default configuration, one-frame units)"""
        if fmt not in self._alone:
            fd = self.dev(fmt)
            out = _prefilled(fd, fmt, F_SENT_ALONE if fmt == "f32" else U_SENT_ALONE)
            for i in range(self.n):
                self.cc.warp(self.c, 0, fd[i:i + 1], self.ratio, self.axs, fill=self.fill(fmt), coord="f32",
                             out=out[i:i + 1])
            self._alone[fmt] = out
        return self._alone[fmt]

    def fp32_map(self):
        """(FP32 map row, FP32 map col, pixels the FP64 map puts inside the frame by 1e-3 px)"""
        if self._map is None:
            sz = self.sz
            omr, omc = oc.rectify_map(self.ch, 1.0 / self.ratio, self.axs, sz)
            inb = (omr >= 1.001) & (omr <= sz[0] - 0.001) & (omc >= 1.001) & (omc <= sz[1] - 0.001)
            fr, fc = self.cc.rectify_map(self.c, 0, self.ratio, self.axs, sz, coord="f32")
            self._map = (fr.cpu().numpy().astype(np.float64), fc.cpu().numpy().astype(np.float64), inb)
        return self._map

    def check(self, fmt, coord, out, what):
        """out: the CUDA result for the first out.shape[0] frames"""
        n = out.shape[0]
        if coord == "f64":
            _assert_exact(out.cpu().numpy(), self.ref(fmt)[:n], fmt, what)
            return
        alone = self.alone(fmt)[:n]
        for f in range(n):
            a, b = (out[f].view(torch.int32), alone[f].view(torch.int32)) if fmt == "f32" else (out[f], alone[f])
            assert torch.equal(a, b), (what, f)
        got = out.cpu().numpy()
        if fmt == "u8":
            _assert_u8_fast_near(got, self.ref(fmt)[:n], what)
            return
        assert not np.any(got == F_SENT), what
        fr, fc, inb = self.fp32_map()
        for j, i in enumerate(self.ramps):
            if i < n:
                m = fr if j % 2 == 0 else fc
                assert np.max(np.abs(got[i][inb].astype(np.float64) - m[inb])) <= 5e-4, (what, i)


# ------------------------------------------------------------------ A. single-view staged kernels
SWEEP_FG = (1, 2, 3, 4, 5, 12, 16)
SWEEP_N = (1, 2, 3, 7, 12, 13, 17, 25)


@pytest.fixture(scope="module")
def small(cc):
    # 256 px lines: 1 KB (f32) and 768 B (u8) pitches, TMA-addressable; small boxes, so the f32 ring holds >= 4
    return _Case(cc, (256, 192), max(SWEEP_N), seed=500)


@pytest.fixture(scope="module")
def large_box(cc):
    # magnified 2.4x (test_gpu_parity.py::test_rectify_alternating_large_and_small_boxes): a ~30 KB f32 box, a
    # ring of 2 stages -> the single-frame kernel at any group size (the u8 box does not fit a 256-byte TMA line)
    return _Case(cc, (512, 384), max(SWEEP_N), seed=600, ratio_scale=0.42)


def _sweep(cc, capfd, case, fmt, coord, fg, expect_pair):
    tiles = _tiles(case.sz)
    for n in SWEEP_N:
        capfd.readouterr()
        with _env(CAMCAL_FG=str(fg), CAMCAL_DEBUG="1"):
            out = case.warp(fmt, coord, n, F_SENT if fmt == "f32" else U_SENT)
        d = _one_staged(capfd.readouterr().err)
        what = (fmt, coord, fg, n)
        fg_eff = min(fg, n)
        assert d["fg"] == fg_eff and d["units"] == tiles * -(-n // fg_eff), (what, d)
        pair = _check_ring(d, fmt, fg_eff)
        if fmt == "f32":
            assert pair == expect_pair(fg_eff), (what, d)
        case.check(fmt, coord, out, what)


@pytest.mark.parametrize("fg", SWEEP_FG)
@pytest.mark.parametrize("coord", ["f64", "f32"])
@pytest.mark.parametrize("fmt", ["f32", "u8"])
def test_staged_frame_groups_small_frame(cc, capfd, small, fmt, coord, fg):
    """CAMCAL_FG x frame counts: units of 1..16 frames, the last unit short (13 frames at fg 12: a unit of one
    frame; 25 at fg 2: an odd end of a pair unit; 7 at fg 5: a pair and an odd end), both coordinate modes,
    both pixel formats.  Small boxes: every f32 unit of >= 2 frames takes the pair kernel."""
    _sweep(cc, capfd, small, fmt, coord, fg, lambda fg_eff: fg_eff >= 2)


@pytest.mark.parametrize("fg", SWEEP_FG)
@pytest.mark.parametrize("coord", ["f64", "f32"])
def test_staged_frame_groups_large_box(cc, capfd, large_box, coord, fg):
    """A ring of fewer than 4 boxes keeps one frame per stage whatever the group size."""
    _sweep(cc, capfd, large_box, "f32", coord, fg, lambda fg_eff: False)


def _u8_stageable(sz):
    """TMA addresses lines of 16-byte multiples: 3 * sz1 bytes for RGB (a 1080-px line is 3240 B: direct kernels)"""
    return sz[0] * 3 % 16 == 0


@pytest.mark.parametrize("coord", ["f64", "f32"])
@pytest.mark.parametrize("fmt,sz,n", [pytest.param("f32", (1080, 1920), 63, id="f32-1080p-63"),
                                      pytest.param("u8", (2160, 3840), 17, id="u8-4k-17"),
                                      pytest.param("u8", (1080, 1920), 33, id="u8-1080p-33")])
def test_default_groups_full_size(cc, capfd, fmt, sz, n, coord):
    """The benchmark's configurations (the bench view, no knob) with batches that do not divide into whole groups:
    on 148 SMs, 1080p f32 exact runs pair units of 12 frames and f32 fast of 4, each batch ending in a unit of 3
    (a pair and an odd end); 4K u8 runs units of 16 ending in a unit of 1.  1080p u8 lines cannot be staged: the
    direct kernel, one launch for the batch."""
    intr = C2_INTR if sz[0] == 1080 else C3_INTR
    case = _Case(cc, sz, n, seed=700, intr=intr, view=BENCH_VIEW, ramps=(n - 2, n - 1))   # ramps in the last unit
    ctx = cc.context(0)
    n0 = ctx.launch_count()
    capfd.readouterr()
    with _env(CAMCAL_DEBUG="1"):
        out = case.warp(fmt, coord, n, F_SENT if fmt == "f32" else U_SENT)
    err = capfd.readouterr().err
    assert ctx.launch_count() - n0 == 1
    if fmt == "u8" and not _u8_stageable(sz):
        assert not _staged_lines(err), err[-2000:]
    else:
        d = _one_staged(err)
        fg = _mirror_fg(_tiles(sz), FG_MAX[(fmt, coord)], n)
        assert fg >= 2 and n % fg and d["fg"] == fg and d["units"] == _tiles(sz) * -(-n // fg), d
        assert _check_ring(d, fmt, fg) == (fmt == "f32"), d
    case.check(fmt, coord, out, (fmt, coord, n))


# ------------------------------------------------------------------ B. views kernels, several groups per view
# (size, views, frames per view); on 148 SMs frames per group f32 exact / f32 fast / u8:
#   (1024, 512)  7 x 5   3 / 4 / 3  (units of 3 + 2, 4 + 1)
#   (1024, 512)  7 x 8   4 / 4 / 4  (two whole groups per view)
#   (1024, 512)  3 x 17  3 / 4 / 4  (5 x 3 + 2, 4 x 4 + 1)
#   (1080, 1920) 3 x 9   5 / 4 / -  (5 + 4, 4 + 4 + 1; u8: 1080-px lines cannot be staged, one direct launch per view)
#   (512, 384)  40 x 3   3 / 3 / 3  (one whole group per view)
VIEWS_CASES = [((1024, 512), 7, 5), ((1024, 512), 7, 8), ((1024, 512), 3, 17), ((1080, 1920), 3, 9),
               ((512, 384), 40, 3)]


@pytest.mark.parametrize("fmt", ["f32", "u8"])
@pytest.mark.parametrize("sz,nv,fpv", VIEWS_CASES)
def test_views_frame_groups_per_view(cc, capfd, sz, nv, fpv, fmt):
    """cc_rectify_*_views with frame groups inside a view (rectify_ring.cuh: producer_loop, VIEWS): every view its
    own extrinsic, ratio and axes; one launch for the group (1080p u8: one direct launch per view), bit-equal to
    one launch per view (CAMCAL_VIEWS_SINGLE=0), and the exact results equal the oracle view by view."""
    intr = camera_for(sz)
    views = _perturbed_views(nv)
    c = _calib(cc, intr, views)
    ratios, axss = [], []
    for vi in range(nv):
        _, _, ratio, axs = _rect_case(intr, sz, ratio_scale=1.0 + 0.01 * (vi % 5), view=views[vi])
        ratios.append(ratio)
        axss.append(axs)
    host = _frames_f32(nv * fpv, sz, 800) if fmt == "f32" else _frames_u8(nv * fpv, sz, 900)
    fd = _dev(host)
    fill = F_FILL if fmt == "f32" else U_FILL
    ctx = cc.context(0)
    tiles = _tiles(sz)
    group = fmt == "f32" or _u8_stageable(sz)
    for coord in ("f64", "f32"):
        what = (sz, nv, fpv, fmt, coord)
        got = {}
        for single, sentinel in (("1", F_SENT if fmt == "f32" else U_SENT), ("0", F_SENT_ALONE if fmt == "f32" else U_SENT_ALONE)):
            out = _prefilled(fd, fmt, sentinel)
            capfd.readouterr()
            n0 = ctx.launch_count()
            with _env(CAMCAL_VIEWS_SINGLE=single, CAMCAL_DEBUG="1"):
                cc.warp_views(c, list(range(nv)), fd, ratios, axss, fill=fill, coord=coord, out=out)
            assert ctx.launch_count() - n0 == (1 if single == "1" and group else nv), what
            err = capfd.readouterr().err
            if not group:
                assert not _staged_lines(err), what
            elif single == "1":
                d = _one_staged(err)
                fg = _mirror_fg(tiles * nv, FG_MAX[(fmt, coord)], fpv)
                assert fg >= 2 and d["fg"] == fg and d["units"] == tiles * nv * -(-fpv // fg), (what, d)
                _check_ring(d, fmt, 1)                   # the views kernels keep one frame per stage
            got[single] = out
        a, b = got["1"], got["0"]
        if fmt == "f32":
            a, b = a.view(torch.int32), b.view(torch.int32)
        for f in range(nv * fpv):
            assert torch.equal(a[f], b[f]), (what, f)
        res = got["1"].cpu().numpy()
        if fmt == "f32":
            assert not np.any(res == F_SENT), what
        if coord == "f64":
            rect = oc.rectify_f32c1 if fmt == "f32" else oc.rectify_u8c3
            for vi in range(nv):
                sl = slice(vi * fpv, (vi + 1) * fpv)
                ref = rect(oc.chain(intr, *views[vi]), 1.0 / ratios[vi], axss[vi], host[sl], fill=fill)
                _assert_exact(res[sl], ref, fmt, what + (vi,))


# ------------------------------------------------------------------ C. views through the ABI, strided layouts
@pytest.mark.parametrize("fpv,nv", [(1, 5), (3, 4)])
@pytest.mark.parametrize("pad1,padf,group", [(4, 64, True), (3, 7, False)])
@pytest.mark.parametrize("fmt", ["f32", "u8"])
def test_views_strided_layouts_through_the_abi(cc, fmt, pad1, padf, group, fpv, nv):
    """cc_rectify_*_views with pitch > sz1 and frame_stride > pitch * sz2.  Pad 4 / 64 px keeps lines and frames
    16-byte aligned for both pixel formats (256-px lines): one launch for the group.  Pad 3 / 7 px cannot be
    staged: one launch per view, round-robin over the side streams.  The valid region equals the dense oracle
    result, the padding is never written."""
    from cameracalibrations_b200 import _lib
    sz = (252, 160)
    intr = camera_for(sz)
    views = _perturbed_views(nv)
    c = _calib(cc, intr, views)
    ratios, axss = [], []
    for vi in range(nv):
        _, _, ratio, axs = _rect_case(intr, sz, ratio_scale=1.0 + 0.01 * vi, view=views[vi])
        ratios.append(ratio)
        axss.append(axs)
    nfr, pitch = nv * fpv, sz[0] + pad1
    stride = pitch * sz[1] + padf
    ch = 1 if fmt == "f32" else 3
    dense = _frames_f32(nfr, sz, 1100) if fmt == "f32" else _frames_u8(nfr, sz, 1200)
    dt = np.float32 if fmt == "f32" else np.uint8
    pad_in, pad_out = (777.0, 555.0) if fmt == "f32" else (77, 55)

    def frame_view(buf, f):
        v = buf[f * stride * ch: (f * stride + pitch * sz[1]) * ch].reshape((sz[1], pitch) + ((3,) if ch == 3 else ()))
        return v[:, :sz[0]]

    buf = np.full(nfr * stride * ch, pad_in, dt)
    for f in range(nfr):
        frame_view(buf, f)[...] = dense[f]
    src, dst = _dev(buf), _dev(np.full(nfr * stride * ch, pad_out, dt))
    vw = (_lib.View * nv)(*[c._views[i] for i in range(nv)])
    rat = (C.c_double * nv)(*ratios)
    axs = (C.c_int64 * (2 * nv))(*[a for am in axss for a in am])
    ctx = cc.context(0)
    n0 = ctx.launch_count()
    if fmt == "f32":
        fn, fv = _lib.lib.cc_rectify_f32c1_views, C.c_float(F_FILL)
    else:
        fn, fv = _lib.lib.cc_rectify_u8c3_views, (C.c_uint8 * 3)(*U_FILL)
    _lib.check(fn(ctx.handle, C.byref(c._intr), vw, nv, rat, axs, C.c_void_p(src.data_ptr()), C.c_void_p(dst.data_ptr()),
                  sz[0], sz[1], C.c_size_t(pitch), C.c_size_t(stride), fpv, fv, _lib.COORD_F64, None))
    torch.cuda.synchronize()
    assert ctx.launch_count() - n0 == (1 if group else nv)
    out = dst.cpu().numpy()
    seen = np.zeros(out.shape, bool)
    rect = oc.rectify_f32c1 if fmt == "f32" else oc.rectify_u8c3
    for vi in range(nv):
        ref = rect(oc.chain(intr, *views[vi]), 1.0 / ratios[vi], axss[vi], dense[vi * fpv:(vi + 1) * fpv],
                   fill=F_FILL if fmt == "f32" else U_FILL)
        for j in range(fpv):
            f = vi * fpv + j
            assert np.array_equal(frame_view(out, f), ref[j]), (vi, j)
            frame_view(seen, f)[...] = True
    assert np.all(out[~seen] == pad_out)


# ------------------------------------------------------------------ D. host chunk pipeline
# cc_rectify_*_host (abi.cu, rectify_host) with CAMCAL_CHUNK_MB=1: `per` whole frames per chunk; a head ramp of
# 1, 2, 4 ... frames (< per), body chunks of `per` (the last one cut to what the tail leaves), a tail whose
# chunks halve down to 1; no ramp when 2 * ramp + per > nframes.  One launch per chunk.
#   256 x 256 f32 dense, 1 MB: per 4, ramp 1 + 2      23 frames: 1, 2, 4, 4, 4, 4, 1, 2, 1
#   256 x 256 u8 dense:        per 5, ramp 1 + 2 + 4  23 frames: 1, 2, 4, 5, 4, 4, 2, 1
#   pitch 272 f32:             per 3, ramp 1 + 2      23 frames: 1, 2, 3, 3, 3, 3, 3, 2, 2, 1
#   pitch 272 u8:              per 5                  23 frames: 1, 2, 4, 5, 4, 4, 2, 1
#   CAMCAL_CHUNK_RAMP=0, dense 23 frames:             f32 4, 4, 4, 4, 4, 3; u8 5, 5, 5, 5, 3
#   9 frames, dense (2 * ramp + per > 9: no ramp):    f32 4, 4, 1; u8 5, 4
HOST_CASES = {
    ("dense", 23, "1"): {"f32": [1, 2, 4, 4, 4, 4, 1, 2, 1], "u8": [1, 2, 4, 5, 4, 4, 2, 1]},
    ("strided", 23, "1"): {"f32": [1, 2, 3, 3, 3, 3, 3, 2, 2, 1], "u8": [1, 2, 4, 5, 4, 4, 2, 1]},
    ("dense", 23, "0"): {"f32": [4, 4, 4, 4, 4, 3], "u8": [5, 5, 5, 5, 3]},
    ("dense", 9, "1"): {"f32": [4, 4, 1], "u8": [5, 4]},
}


@pytest.mark.parametrize("coord", ["f64", "f32"])
@pytest.mark.parametrize("fmt", ["f32", "u8"])
@pytest.mark.parametrize("layout,n,ramp", list(HOST_CASES))
def test_host_chunk_pipeline(cc, layout, n, ramp, fmt, coord):
    """Host frames through the chunked upload / rectify / download pipeline (consecutive chunks on different
    streams; strided host layouts copied frame by frame with 2-D copies): exact results equal the oracle frame by
    frame, fast results the device call on the same layout, host padding is never written."""
    from cameracalibrations_b200 import _lib
    sz = (256, 256)
    case = _Case(cc, sz, n, seed=1300)
    chunks = HOST_CASES[(layout, n, ramp)][fmt]
    assert sum(chunks) == n
    ctx = cc.context(0)
    fill = case.fill(fmt)
    dense = case.host(fmt)
    dt = np.float32 if fmt == "f32" else np.uint8
    flags = _lib.COORD_F64 if coord == "f64" else _lib.COORD_F32
    if layout == "dense":
        out = np.empty_like(dense)
        out[...] = np.array(F_SENT if fmt == "f32" else U_SENT, dtype=dt)
        n0 = ctx.launch_count()
        with _env(CAMCAL_CHUNK_MB="1", CAMCAL_CHUNK_RAMP=ramp):
            cc.warp(case.c, 0, dense, case.ratio, case.axs, fill=fill, coord=coord, out=out)
        assert ctx.launch_count() - n0 == len(chunks)
        if coord == "f64":
            _assert_exact(out, case.ref(fmt), fmt, (layout, n, ramp))
        else:
            dev = case.warp(fmt, "f32", n, F_SENT_ALONE if fmt == "f32" else U_SENT_ALONE).cpu().numpy()
            assert np.array_equal(out.view(np.uint8), dev.view(np.uint8))
        return
    ch = 1 if fmt == "f32" else 3
    pitch = sz[0] + 16                                   # 16-byte aligned lines: the device chunks stay staged
    stride = pitch * sz[1] + 64
    pad_in, pad_out = (F_SENT_ALONE, F_SENT) if fmt == "f32" else (U_SENT_ALONE[0], U_SENT[0])

    def frame_view(buf, f):
        v = buf[f * stride * ch: (f * stride + pitch * sz[1]) * ch].reshape((sz[1], pitch) + ((3,) if ch == 3 else ()))
        return v[:, :sz[0]]

    src = np.full(n * stride * ch, pad_in, dt)
    for f in range(n):
        frame_view(src, f)[...] = dense[f]
    dst = np.full(n * stride * ch, pad_out, dt)
    axs = (C.c_int64 * 2)(*case.axs)
    ci, cv = C.byref(case.c._intr), C.byref(case.c._views[0])
    if fmt == "f32":
        fn_h, fn_d, fv = _lib.lib.cc_rectify_f32c1_host, _lib.lib.cc_rectify_f32c1, C.c_float(fill)
    else:
        fn_h, fn_d, fv = _lib.lib.cc_rectify_u8c3_host, _lib.lib.cc_rectify_u8c3, (C.c_uint8 * 3)(*fill)
    geom = (sz[0], sz[1], C.c_size_t(pitch), C.c_size_t(stride), n)
    n0 = ctx.launch_count()
    with _env(CAMCAL_CHUNK_MB="1", CAMCAL_CHUNK_RAMP=ramp):
        _lib.check(fn_h(ctx.handle, ci, cv, float(case.ratio), axs, C.c_void_p(src.ctypes.data),
                        C.c_void_p(dst.ctypes.data), *geom, fv, flags))
    assert ctx.launch_count() - n0 == len(chunks)
    seen = np.zeros(dst.shape, bool)
    for f in range(n):
        frame_view(seen, f)[...] = True
    assert np.all(dst[~seen] == pad_out)
    got = np.stack([frame_view(dst, f) for f in range(n)])
    if coord == "f64":
        _assert_exact(got, case.ref(fmt), fmt, (layout, n, ramp))
    else:                                                # the device call on the same strided layout
        dsrc, ddst = _dev(src), _dev(np.full(n * stride * ch, pad_out, dt))
        _lib.check(fn_d(ctx.handle, ci, cv, float(case.ratio), axs, C.c_void_p(dsrc.data_ptr()),
                        C.c_void_p(ddst.data_ptr()), *geom, fv, flags, None))
        torch.cuda.synchronize()
        assert np.array_equal(ddst.cpu().numpy().view(np.uint8), dst.view(np.uint8))
