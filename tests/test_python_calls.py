"""The C calls of the Python layer, pinned.

The library handle of `calibration` and `lm` is replaced by a recorder that logs every call and returns CC_OK,
and `_lib.context` by a stand-in whose handle encodes the device it was asked for.  So no device is touched and
the cases run on a CPU-only box; with a CUDA device the same cases run again on CUDA tensors.  For every public
function that makes one C call and returns, each case asserts the entry point, every scalar and flag, the
contents of the structs and ctypes arrays, and for each array argument its dtype, shape, C-contiguity and
whether it is the caller's buffer or a copy; then the type, shape and dtype of what comes back.
"""
import ctypes as C
import math
import sys

import numpy as np
import pytest
import torch

from cameracalibrations_b200 import _lib, calibration as cal, lm

_H = 0xC7000                           # handle of the stand-in context of device d: _H + d
FILES = ["a.png", "b_extrinsic.png", "c.png"]
EXT = [((0.1, -0.2, 0.3), (1.0, 2.0, 30.0)), ((0.2, 0.1, -0.1), (-1.0, 0.5, 25.0)),
       ((-0.3, 0.05, 0.2), (0.0, -2.0, 40.0))]
INTR = (100.0, 110.0, 50.0, 60.0, -0.125, 2.0)
VIEW = [r + t for r, t in EXT]
NAN = float("nan")


def _cal(files=FILES):
    return cal.Calibration(INTR[:4], EXT, 1.0 / INTR[5], INTR[4], files)


# ---------------------------------------------------------------- the recorder
class _Call:
    def __init__(self, name, args, keep):
        self.name, self.args, self.keep = name, [_norm(a) for a in args], keep


class _Recorder:
    """Stands in for the ctypes library: logs (name, args) and returns CC_OK.  It also keeps every array and
    tensor the layer's frames hold at the call, so that the buffers behind the pointers stay alive to be
    inspected."""

    def __init__(self):
        self.calls = []

    def __getattr__(self, name):
        if not name.startswith("cc_"):
            raise AttributeError(name)

        def fn(*args):
            self.calls.append(_Call(name, args, _held(sys._getframe(1))))
            return 0
        return fn


class _Ctx:
    def __init__(self, device=0):
        self.device = int(device)
        self.handle = C.c_void_p(_H + self.device)


def _held(frame):
    keep = []

    def walk(v, depth):
        if isinstance(v, (np.ndarray, torch.Tensor)):
            keep.append(v)
        elif isinstance(v, (list, tuple)) and depth < 3:
            for e in v:
                walk(e, depth + 1)
    while frame is not None and frame.f_code.co_filename != __file__:
        for v in frame.f_locals.values():
            walk(v, 0)
        frame = frame.f_back
    return keep


def _norm(a):
    """What the C side receives, as plain Python values: pointers as addresses (NULL = 0), structs as tuples of
    their fields, ctypes arrays as lists."""
    if a is None:
        return 0
    if type(a).__name__ == "CArgObject":           # C.byref(x)
        return _norm(a._obj)
    if isinstance(a, C.Structure):
        return tuple(x for f, _ in a._fields_ for x in np.ravel(_norm(getattr(a, f))))
    if isinstance(a, C.Array):
        return [_norm(e) for e in a]
    if isinstance(a, C._SimpleCData):
        return 0 if a.value is None else a.value
    if isinstance(a, (int, float)):
        return a
    raise AssertionError(f"unexpected argument {a!r}")


def _addr(a):
    return a.data_ptr() if isinstance(a, torch.Tensor) else a.ctypes.data


def _dt(a):
    return str(a.dtype).replace("torch.", "")


def _contig(a):
    return a.is_contiguous() if isinstance(a, torch.Tensor) else a.flags.c_contiguous


def _host(a):
    return a.cpu().numpy() if isinstance(a, torch.Tensor) else np.asarray(a)


class Buf:
    """An array argument: its dtype and shape, C-contiguous; `own` = the caller's object it must be (an input
    passed as is, or the output returned); `copy_of` = the caller's input it must be a copy of; `values` = the
    contents it must hold."""

    def __init__(self, dtype, shape, own=None, copy_of=None, values=None):
        self.dtype, self.shape = np.dtype(dtype).name, tuple(shape)
        self.own, self.copy_of, self.values = own, copy_of, values

    def check(self, call, addr, where):
        found = list(call.keep) + ([self.own] if self.own is not None else [])
        cands = [a for a in found if _addr(a) == addr]
        ok = [a for a in cands if _dt(a) == self.dtype and tuple(a.shape) == self.shape and _contig(a)]
        assert ok, (where, self.dtype, self.shape, [(_dt(a), tuple(a.shape), _contig(a)) for a in cands])
        if self.own is not None:
            assert addr == _addr(self.own), (where, "not the caller's buffer")
        if self.copy_of is not None:
            assert addr != _addr(self.copy_of), (where, "the caller's buffer, not a copy")
            want = _host(self.copy_of).astype(self.dtype).reshape(self.shape)
            assert np.array_equal(_host(ok[0]), want, equal_nan=True), (where, "copy of other contents")
        if self.values is not None:
            want = np.asarray(self.values, dtype=self.dtype).reshape(self.shape)
            assert np.array_equal(_host(ok[0]), want, equal_nan=True), (where, "contents")


def _same(a, b):
    if isinstance(a, float) and isinstance(b, float) and math.isnan(a) and math.isnan(b):
        return True
    if isinstance(a, (list, tuple)) and isinstance(b, (list, tuple)):
        return len(a) == len(b) and all(_same(x, y) for x, y in zip(a, b))
    return type(a) is not bool and a == b


def _expect(rec, name, want):
    """The one C call of the case: its entry point and every argument."""
    assert [c.name for c in rec.calls] == [name]
    call = rec.calls.pop()
    assert len(call.args) == len(want), (name, call.args)
    for i, (got, w) in enumerate(zip(call.args, want)):
        if isinstance(w, Buf):
            w.check(call, got, (name, i))
        else:
            assert _same(got, w), (name, i, got, w)
    return call


def _ret(y, mode, shape, dtype):
    if mode.cuda:
        assert isinstance(y, torch.Tensor) and y.is_cuda and y.device == mode.device
    else:
        assert isinstance(y, np.ndarray)
    assert tuple(y.shape) == tuple(shape) and _dt(y) == np.dtype(dtype).name


def _rejects(rec, exc, fn):
    with pytest.raises(exc):
        fn()
    assert rec.calls == []


# ---------------------------------------------------------------- fixtures
class _Mode:
    def __init__(self, cuda):
        self.cuda = cuda
        if cuda:
            self.device = torch.device("cuda", torch.cuda.current_device())
            self.stream = torch.cuda.Stream(self.device)
            self.h = _H + self.device.index
        else:
            self.h = _H + (torch.cuda.current_device() if torch.cuda.is_available() else 0)

    def to(self, x):
        return torch.as_tensor(np.asarray(x)).to(self.device) if self.cuda else x

    def name(self, base):
        return base if self.cuda else base + "_host"

    @property
    def tail(self):
        return [self.stream.cuda_stream] if self.cuda else []


def _cuda_mode():
    if not torch.cuda.is_available():
        pytest.skip("no CUDA device")
    return _Mode(True)


@pytest.fixture(params=["numpy", pytest.param("cuda", marks=pytest.mark.gpu)])
def mode(request):
    if request.param == "numpy":
        yield _Mode(False)
        return
    m = _cuda_mode()
    with torch.cuda.stream(m.stream):
        yield m


@pytest.fixture
def cuda():
    m = _cuda_mode()
    with torch.cuda.stream(m.stream):
        yield m


@pytest.fixture
def rec(monkeypatch):
    r = _Recorder()
    monkeypatch.setattr(cal, "lib", r)
    monkeypatch.setattr(lm, "lib", r)
    monkeypatch.setattr(_lib, "context", _Ctx)
    return r


def _pts(shape, dtype=np.float64, seed=0):
    return (np.random.default_rng(seed).random(shape) * 100).astype(dtype)


# ---------------------------------------------------------------- c(pts, extrinsic): the interleaved layout
@pytest.mark.parametrize("ext, vi", [("c.png", 2), (None, 1), (0, 0), (np.int64(2), 2)])
def test_call_picks_the_view(rec, mode, ext, vi):
    x = mode.to(_pts((5, 2)))
    y = _cal()(x, ext)
    _ret(y, mode, (5, 3), np.float64)
    _expect(rec, mode.name("cc_img2world_f64_aos"), [mode.h, INTR, VIEW[vi], 1, 0, Buf(np.float64, (5, 2), own=x),
                                                     Buf(np.float64, (5, 3), own=y), 3, 5] + mode.tail)


@pytest.mark.parametrize("dtype", [np.float32, np.float64])
def test_call_world2img_keeps_the_leading_axes(rec, mode, dtype):
    x = mode.to(_pts((2, 3, 3), dtype))
    y = _cal()(x, 1)
    _ret(y, mode, (2, 3, 2), dtype)
    sfx = "f32" if dtype == np.float32 else "f64"
    _expect(rec, mode.name(f"cc_world2img_{sfx}_aos"), [mode.h, INTR, VIEW[1], 1, 0, Buf(dtype, (2, 3, 3), own=x), 3,
                                                        Buf(dtype, (2, 3, 2), own=y), 6] + mode.tail)


def test_call_single_point(rec, mode):
    x = mode.to(_pts((2,)))
    y = _cal()(x, 2)
    _ret(y, mode, (3,), np.float64)
    _expect(rec, mode.name("cc_img2world_f64_aos"), [mode.h, INTR, VIEW[2], 1, 0, Buf(np.float64, (2,), own=x),
                                                     Buf(np.float64, (3,), own=y), 3, 1] + mode.tail)


@pytest.mark.parametrize("dtype, passed", [(np.float32, np.float32), (np.float64, np.float64), (np.float16, np.float64),
                                           (np.int32, np.float64), (np.uint8, np.float64)])
def test_call_dtype_rule_numpy(rec, dtype, passed):
    x = _pts((4, 2), dtype)
    y = _cal()(x, 0)
    _ret(y, _Mode(False), (4, 3), passed)
    sfx = "f32" if passed == np.float32 else "f64"
    arg = Buf(passed, (4, 2), own=x) if dtype == passed else Buf(passed, (4, 2), copy_of=x)
    _expect(rec, f"cc_img2world_{sfx}_aos_host", [_Mode(False).h, INTR, VIEW[0], 1, 0, arg,
                                                  Buf(passed, (4, 3), own=y), 3, 4])


@pytest.mark.parametrize("layout", ["strided", "transposed", "list"])
def test_call_copies_other_layouts(rec, mode, layout):
    base = _pts((8, 3))
    if layout == "list" and mode.cuda:
        pytest.skip("host arrays only")
    x = {"strided": lambda: mode.to(base)[::2], "transposed": lambda: mode.to(_pts((3, 4))).T,
         "list": lambda: base[::2].tolist()}[layout]()
    y = _cal()(x, 2)
    _ret(y, mode, (4, 2), np.float64)
    arg = Buf(np.float64, (4, 3), values=_host(x) if layout != "list" else base[::2])
    if layout != "list":
        arg.copy_of = x
    _expect(rec, mode.name("cc_world2img_f64_aos"), [mode.h, INTR, VIEW[2], 1, 0, arg, 3,
                                                     Buf(np.float64, (4, 2), own=y), 4] + mode.tail)


def test_call_list_form(rec, mode):
    a, b = _pts((2, 2), np.float32, 1), _pts((3, 2), np.float32, 2)
    ys = _cal()([mode.to(a), mode.to(b)], [2, "a.png"])
    assert isinstance(ys, list) and len(ys) == 2
    _ret(ys[0], mode, (2, 3), np.float32)
    _ret(ys[1], mode, (3, 3), np.float32)
    _expect(rec, mode.name("cc_img2world_f32_aos"), [
        mode.h, INTR, Buf(np.float64, (2, 6), values=[VIEW[2], VIEW[0]]), 2, Buf(np.uint64, (3,), values=[0, 2, 5]),
        Buf(np.float32, (5, 2), values=np.concatenate([a, b])), Buf(np.float32, (5, 3), own=ys[0]), 3, 5] + mode.tail)
    assert _addr(ys[1]) == _addr(ys[0]) + 2 * 3 * 4


def test_call_list_form_mixed_dtypes_become_float64(rec):
    a, b = _pts((1, 3), np.float32, 1), _pts((2, 3), np.float64, 2)
    ys = _cal()([a, b], (1, 1))
    m = _Mode(False)
    _ret(ys[0], m, (1, 2), np.float64)
    _ret(ys[1], m, (2, 2), np.float64)
    _expect(rec, "cc_world2img_f64_aos_host", [
        m.h, INTR, Buf(np.float64, (2, 6), values=[VIEW[1], VIEW[1]]), 2, Buf(np.uint64, (3,), values=[0, 1, 3]),
        Buf(np.float64, (3, 3), values=np.concatenate([a.astype(np.float64), b])), 3,
        Buf(np.float64, (3, 2), own=ys[0]), 3])


def test_call_rejects(rec, mode):
    c = _cal()
    x = mode.to(_pts((4, 2)))
    _rejects(rec, TypeError, lambda: c(mode.to(_pts((4, 4))), 0))
    _rejects(rec, IndexError, lambda: c(x, 3))
    _rejects(rec, IndexError, lambda: c(x, -1))
    _rejects(rec, ValueError, lambda: c(x, "missing.png"))
    _rejects(rec, IndexError, lambda: _cal(["a", "b", "c"])(x, None))
    _rejects(rec, ValueError, lambda: c([x, x], [0]))
    _rejects(rec, TypeError, lambda: c([x, mode.to(_pts((4, 3)))], [0, 1]))
    _rejects(rec, TypeError, lambda: c([mode.to(_pts((4, 4)))], [0]))
    _rejects(rec, IndexError, lambda: c([x], [3]))
    if mode.cuda:
        _rejects(rec, TypeError, lambda: c(x.half(), 0))
    _rejects(rec, TypeError, lambda: c(torch.zeros((4, 2), dtype=torch.float64), 0))


# ---------------------------------------------------------------- img2world / world2img: one array per coordinate
@pytest.mark.parametrize("want_z", [True, False])
def test_img2world(rec, mode, want_z):
    row, col = mode.to(_pts((6,), seed=1)), mode.to(_pts((6,), seed=2))
    outs = _cal().img2world(row, col, "c.png", want_z=want_z)
    assert isinstance(outs, tuple) and len(outs) == (3 if want_z else 2)
    for o in outs:
        _ret(o, mode, (6,), np.float64)
    z = Buf(np.float64, (6,), own=outs[2]) if want_z else 0
    _expect(rec, mode.name("cc_img2world_f64"), [mode.h, INTR, VIEW[2], Buf(np.float64, (6,), own=row),
                                                 Buf(np.float64, (6,), own=col), Buf(np.float64, (6,), own=outs[0]),
                                                 Buf(np.float64, (6,), own=outs[1]), z, 6] + mode.tail)


@pytest.mark.parametrize("with_z", [True, False])
def test_world2img(rec, mode, with_z):
    x, y, z = (mode.to(_pts((5,), np.float32, s)) for s in (1, 2, 3))
    outs = _cal().world2img(x, y, z if with_z else None)          # extrinsic None: the first "extrinsic" file
    assert isinstance(outs, tuple) and len(outs) == 2
    for o in outs:
        _ret(o, mode, (5,), np.float32)
    _expect(rec, mode.name("cc_world2img_f32"), [
        mode.h, INTR, VIEW[1], Buf(np.float32, (5,), own=x), Buf(np.float32, (5,), own=y),
        Buf(np.float32, (5,), own=z) if with_z else 0, Buf(np.float32, (5,), own=outs[0]),
        Buf(np.float32, (5,), own=outs[1]), 5] + mode.tail)


def test_point_arrays_follow_the_first_numpy(rec):
    m = _Mode(False)
    row, col = _pts((2, 3), np.float32, 1), _pts((6,), np.float64, 2)
    outs = _cal().img2world(row, col, 0, want_z=False)
    _ret(outs[0], m, (6,), np.float32)
    _expect(rec, "cc_img2world_f32_host", [m.h, INTR, VIEW[0], Buf(np.float32, (2, 3), own=row),
                                           Buf(np.float32, (6,), copy_of=col), Buf(np.float32, (6,), own=outs[0]),
                                           Buf(np.float32, (6,), own=outs[1]), 0, 6])
    x, y = _pts((4,), np.int64, 1), _pts((8,), np.float32, 2)[::2]
    outs = _cal().world2img(x, y, None, 2)
    _ret(outs[1], m, (4,), np.float64)
    _expect(rec, "cc_world2img_f64_host", [m.h, INTR, VIEW[2], Buf(np.float64, (4,), copy_of=x),
                                           Buf(np.float64, (4,), copy_of=y), 0, Buf(np.float64, (4,), own=outs[0]),
                                           Buf(np.float64, (4,), own=outs[1]), 4])


def test_point_views(rec, mode):
    row, col = mode.to(_pts((6,), seed=1)), mode.to(_pts((6,), seed=2))
    outs = _cal().img2world_views(row, col, [2, "b_extrinsic.png", 2], [2, 0, 4])
    assert len(outs) == 3
    _expect(rec, mode.name("cc_img2world_f64_views"), [
        mode.h, INTR, Buf(np.float64, (3, 6), values=[VIEW[2], VIEW[1], VIEW[2]]), 3,
        Buf(np.uint64, (4,), values=[0, 2, 2, 6]), Buf(np.float64, (6,), own=row), Buf(np.float64, (6,), own=col),
        Buf(np.float64, (6,), own=outs[0]), Buf(np.float64, (6,), own=outs[1]), Buf(np.float64, (6,), own=outs[2])]
        + mode.tail)
    x, y = mode.to(_pts((3,), np.float32, 1)), mode.to(_pts((3,), np.float32, 2))
    outs = _cal().world2img_views(x, y, None, np.array([1, 0]), [3, 0])
    for o in outs:
        _ret(o, mode, (3,), np.float32)
    _expect(rec, mode.name("cc_world2img_f32_views"), [
        mode.h, INTR, Buf(np.float64, (2, 6), values=[VIEW[1], VIEW[0]]), 2, Buf(np.uint64, (3,), values=[0, 3, 3]),
        Buf(np.float32, (3,), own=x), Buf(np.float32, (3,), own=y), 0, Buf(np.float32, (3,), own=outs[0]),
        Buf(np.float32, (3,), own=outs[1])] + mode.tail)


def test_point_calls_reject(rec, mode):
    c = _cal()
    a4, a5 = mode.to(_pts((4,))), mode.to(_pts((5,)))
    _rejects(rec, ValueError, lambda: c.img2world(a4, a5, 0))
    _rejects(rec, ValueError, lambda: c.world2img(a4, a4, a5, 0))
    _rejects(rec, IndexError, lambda: c.img2world(a4, a4, 3))
    _rejects(rec, ValueError, lambda: c.img2world_views(a4, a4, [0, 1], [1, 2]))
    _rejects(rec, ValueError, lambda: c.img2world_views(a4, a4, [0, 1], [4]))
    _rejects(rec, ValueError, lambda: c.img2world_views(a4, a4, [], []))
    _rejects(rec, ValueError, lambda: c.img2world_views(a4, a4, [0, 1], [5, -1]))
    _rejects(rec, IndexError, lambda: c.img2world_views(a4, a4, [0, 3], [2, 2]))
    _rejects(rec, IndexError, lambda: c.world2img_views(a4, a4, None, [-1], [4]))
    _rejects(rec, ValueError, lambda: c.world2img_views(a4, a4, None, ["nope"], [4]))
    if mode.cuda:
        _rejects(rec, ValueError, lambda: c.img2world(a4, a4.float(), 0))
        _rejects(rec, TypeError, lambda: c.img2world(a4.half(), a4.half(), 0))
    _rejects(rec, TypeError, lambda: c.img2world(torch.zeros(4), torch.zeros(4), 0))


# ---------------------------------------------------------------- rectification(c, i)(pts)
@pytest.mark.parametrize("dtype", [np.float32, np.float64])
def test_rectification(rec, mode, dtype):
    x = mode.to(_pts((2, 4, 2), dtype))
    y = cal.rectification(_cal(), 2)(x)
    _ret(y, mode, (2, 4, 2), dtype)
    sfx = "f32" if dtype == np.float32 else "f64"
    _expect(rec, mode.name(f"cc_img2world_{sfx}_aos"), [mode.h, INTR, VIEW[2], 1, 0, Buf(dtype, (2, 4, 2), own=x),
                                                        Buf(dtype, (2, 4, 2), own=y), 2, 8] + mode.tail)


def test_rectification_takes_row_and_column_of_longer_points(rec, mode):
    base = _pts((5, 3), np.float32)
    x = mode.to(base)
    y = cal.rectification(_cal())(x)
    _ret(y, mode, (5, 2), np.float32)
    _expect(rec, mode.name("cc_img2world_f32_aos"), [mode.h, INTR, VIEW[1], 1, 0,
                                                     Buf(np.float32, (5, 2), copy_of=x[..., :2]),
                                                     Buf(np.float32, (5, 2), own=y), 2, 5] + mode.tail)


@pytest.mark.parametrize("dtype", [np.float16, np.int64])
def test_rectification_dtype_rule_numpy(rec, dtype):
    x = _pts((3, 2), dtype)
    y = cal.rectification(_cal(), 0)(x)
    m = _Mode(False)
    _ret(y, m, (3, 2), np.float64)
    _expect(rec, "cc_img2world_f64_aos_host", [m.h, INTR, VIEW[0], 1, 0, Buf(np.float64, (3, 2), copy_of=x),
                                               Buf(np.float64, (3, 2), own=y), 2, 3])


def test_rectification_rejects(rec, mode):
    _rejects(rec, IndexError, lambda: cal.rectification(_cal(), 3))
    _rejects(rec, IndexError, lambda: cal.rectification(_cal(), 0)(mode.to(_pts((3, 1)))))


# ---------------------------------------------------------------- warp / warp_views
def _frames(shape, dtype, seed=0):
    r = np.random.default_rng(seed)
    return r.integers(0, 256, shape).astype(np.uint8) if dtype == np.uint8 else r.random(shape).astype(dtype)


FLAGS = [("f64", "auto", 0), ("f32", "auto", 1), ("f64", "direct", 16), ("f32", "tma", 33)]


@pytest.mark.parametrize("coord, gather, flags", FLAGS)
@pytest.mark.parametrize("u8", [False, True])
@pytest.mark.parametrize("single", [False, True])
def test_warp(rec, mode, coord, gather, flags, u8, single):
    dt, kern = (np.uint8, "u8c3") if u8 else (np.float32, "f32c1")
    shape = ((6, 8) if single else (2, 6, 8)) + ((3,) if u8 else ())
    f = mode.to(_frames(shape, dt))
    y = cal.warp(_cal(), "b_extrinsic.png", f, 0.5, (-3, 4), coord=coord, gather=gather)
    _ret(y, mode, shape, dt)
    fill = [0, 0, 0] if u8 else NAN
    _expect(rec, mode.name(f"cc_rectify_{kern}"), [mode.h, INTR, VIEW[1], 0.5, [-3, 4], Buf(dt, shape, own=f),
                                                   Buf(dt, shape, own=y), 8, 6, 8, 48, 1 if single else 2, fill, flags]
            + mode.tail)


@pytest.mark.parametrize("u8", [False, True])
@pytest.mark.parametrize("single", [False, True])
def test_warp_out_and_fill(rec, mode, u8, single):
    dt, kern = (np.uint8, "u8c3") if u8 else (np.float32, "f32c1")
    shape = (1 if single else 3, 5, 7) + ((3,) if u8 else ())
    f = mode.to(_frames(shape[1:] if single else shape, dt))
    out = mode.to(np.zeros(shape, dt))
    y = cal.warp(_cal(), 2, f, 1.25, np.array([2, -1]), fill=(1, 2, 3) if u8 else 0.25, out=out)
    if single:
        _ret(y, mode, shape[1:], dt)
        assert _addr(y) == _addr(out)
    else:
        assert y is out
    _expect(rec, mode.name(f"cc_rectify_{kern}"), [
        mode.h, INTR, VIEW[2], 1.25, [2, -1], Buf(dt, shape[1:] if single else shape, own=f), Buf(dt, shape, own=out),
        7, 5, 7, 35, shape[0], [1, 2, 3] if u8 else 0.25, 0] + mode.tail)


@pytest.mark.parametrize("dtype", [np.float64, np.int16, np.uint16])
def test_warp_casts_numpy_frames_to_float32(rec, dtype):
    f = _frames((2, 4, 5), np.float64).astype(dtype) if dtype == np.float64 else np.arange(40, dtype=dtype).reshape(2, 4, 5)
    y = cal.warp(_cal(), 0, f, 1.0, (0, 0))
    m = _Mode(False)
    _ret(y, m, (2, 4, 5), np.float32)
    _expect(rec, "cc_rectify_f32c1_host", [m.h, INTR, VIEW[0], 1.0, [0, 0], Buf(np.float32, (2, 4, 5), copy_of=f),
                                           Buf(np.float32, (2, 4, 5), own=y), 5, 4, 5, 20, 2, NAN, 0])


def test_warp_copies_strided_frames(rec, mode):
    base = _frames((2, 4, 10), np.float32)
    f = mode.to(base)[:, :, ::2]
    y = cal.warp(_cal(), 0, f, 1.0, (0, 0))
    _ret(y, mode, (2, 4, 5), np.float32)
    _expect(rec, mode.name("cc_rectify_f32c1"), [mode.h, INTR, VIEW[0], 1.0, [0, 0],
                                                 Buf(np.float32, (2, 4, 5), copy_of=f),
                                                 Buf(np.float32, (2, 4, 5), own=y), 5, 4, 5, 20, 2, NAN, 0] + mode.tail)


@pytest.mark.parametrize("coord, gather, flags", FLAGS)
@pytest.mark.parametrize("u8", [False, True])
def test_warp_views(rec, mode, coord, gather, flags, u8):
    dt, kern = (np.uint8, "u8c3") if u8 else (np.float32, "f32c1")
    shape = (4, 6, 8) + ((3,) if u8 else ())
    f = mode.to(_frames(shape, dt))
    y = cal.warp_views(_cal(), [2, "a.png"], f, [0.5, 0.75], [(-3, 4), (1, -2)], coord=coord, gather=gather)
    _ret(y, mode, shape, dt)
    name = f"cc_rectify_{kern}_views" if mode.cuda else f"cc_rectify_views_{kern}_host"
    _expect(rec, name, [mode.h, INTR, [VIEW[2], VIEW[0]], 2, [0.5, 0.75], [-3, 4, 1, -2], Buf(dt, shape, own=f),
                        Buf(dt, shape, own=y), 8, 6, 8, 48, 2, [0, 0, 0] if u8 else NAN, flags] + mode.tail)


@pytest.mark.parametrize("u8", [False, True])
def test_warp_views_out_and_fill(rec, mode, u8):
    dt, kern = (np.uint8, "u8c3") if u8 else (np.float32, "f32c1")
    shape = (3, 5, 7) + ((3,) if u8 else ())
    f, out = mode.to(_frames(shape, dt)), mode.to(np.zeros(shape, dt))
    y = cal.warp_views(_cal(), ["c.png"], f, np.array([2.0]), np.array([[5, 6]]), fill=(9, 8, 7) if u8 else -1.5,
                       out=out)
    assert y is out
    name = f"cc_rectify_{kern}_views" if mode.cuda else f"cc_rectify_views_{kern}_host"
    _expect(rec, name, [mode.h, INTR, [VIEW[2]], 1, [2.0], [5, 6], Buf(dt, shape, own=f), Buf(dt, shape, own=out),
                        7, 5, 7, 35, 3, [9, 8, 7] if u8 else -1.5, 0] + mode.tail)


def test_warp_views_casts_numpy_frames_to_float32(rec):
    f = _frames((2, 3, 4), np.float64)[:, :, ::-1]
    y = cal.warp_views(_cal(), [0, 1], f, [1.0, 1.0], [(0, 0), (0, 0)])
    m = _Mode(False)
    _ret(y, m, (2, 3, 4), np.float32)
    _expect(rec, "cc_rectify_views_f32c1_host", [m.h, INTR, [VIEW[0], VIEW[1]], 2, [1.0, 1.0], [0, 0, 0, 0],
                                                 Buf(np.float32, (2, 3, 4), copy_of=f),
                                                 Buf(np.float32, (2, 3, 4), own=y), 4, 3, 4, 12, 1, NAN, 0])


def test_warp_rejects(rec, mode):
    c = _cal()
    f32, u8 = mode.to(_frames((2, 4, 5), np.float32)), mode.to(_frames((2, 4, 5, 3), np.uint8))
    _rejects(rec, IndexError, lambda: cal.warp(c, 3, f32, 1.0, (0, 0)))
    _rejects(rec, KeyError, lambda: cal.warp(c, 0, f32, 1.0, (0, 0), coord="f16"))
    _rejects(rec, KeyError, lambda: cal.warp(c, 0, f32, 1.0, (0, 0), gather="ldg"))
    _rejects(rec, ValueError, lambda: cal.warp(c, 0, f32[None], 1.0, (0, 0)))
    _rejects(rec, ValueError, lambda: cal.warp(c, 0, f32[0, 0], 1.0, (0, 0)))
    _rejects(rec, ValueError, lambda: cal.warp(c, 0, mode.to(_frames((2, 4, 5, 4), np.uint8)), 1.0, (0, 0)))
    _rejects(rec, ValueError, lambda: cal.warp(c, 0, u8[..., 0], 1.0, (0, 0)))
    _rejects(rec, TypeError, lambda: cal.warp(c, 0, torch.zeros((2, 4, 5)), 1.0, (0, 0)))
    _rejects(rec, IndexError, lambda: cal.warp_views(c, [0, 3], f32, [1.0, 1.0], [(0, 0), (0, 0)]))
    _rejects(rec, KeyError, lambda: cal.warp_views(c, [0, 1], f32, [1.0, 1.0], [(0, 0), (0, 0)], coord="f16"))
    _rejects(rec, KeyError, lambda: cal.warp_views(c, [0, 1], f32, [1.0, 1.0], [(0, 0), (0, 0)], gather="ldg"))
    _rejects(rec, ValueError, lambda: cal.warp_views(c, [0, 1, 2], f32, [1.0] * 3, [(0, 0)] * 3))
    _rejects(rec, ValueError, lambda: cal.warp_views(c, [], f32, [], []))
    _rejects(rec, ValueError, lambda: cal.warp_views(c, [0], f32[0], [1.0], [(0, 0)]))
    _rejects(rec, ValueError, lambda: cal.warp_views(c, [0], u8[..., 0], [1.0], [(0, 0)]))
    _rejects(rec, TypeError, lambda: cal.warp_views(c, [0, 1], torch.zeros((2, 4, 5)), [1.0, 1.0], [(0, 0), (0, 0)]))


# ---------------------------------------------------------------- the fit
NV, NC = 3, 4
FIT_INTR = (120.0, 100.0, 40.0, 50.0, -0.25, 0.5)


def test_reproj_jtj(rec, mode):
    views, obj, img = mode.to(_pts((NV, 6), seed=1)), mode.to(_pts((NC, 3), seed=2)), mode.to(_pts((NV, NC, 2), seed=3))
    pv, sh = cal.reproj_jtj(FIT_INTR, 1.25, views, obj, img)
    _ret(pv, mode, (NV, _lib.PER_VIEW), np.float64)
    _ret(sh, mode, (_lib.SHARED,), np.float64)
    _expect(rec, mode.name("cc_reproj_jtj_f64"), [
        mode.h, FIT_INTR, 1.25, Buf(np.float64, (NV, 6), own=views), NV, Buf(np.float64, (NC, 3), own=obj),
        Buf(np.float64, (NV, NC, 2), own=img), NC, Buf(np.float64, (NV, _lib.PER_VIEW), own=pv),
        Buf(np.float64, (_lib.SHARED,), own=sh)] + mode.tail)


def test_reproj_jtj_converts(rec, mode):
    views = mode.to(_pts((NV, 6), np.float32, 1))
    if not mode.cuda:
        views = views.reshape(-1)                 # a flat host array is read as (nv, 6)
    obj, img = mode.to(_pts((NC, 3), seed=2)), mode.to(_pts((NV, 2 * NC, 2), seed=3))[:, ::2]
    pv, sh = cal.reproj_jtj(np.array(FIT_INTR), 2.0, views, obj, img)
    _ret(pv, mode, (NV, _lib.PER_VIEW), np.float64)
    _expect(rec, mode.name("cc_reproj_jtj_f64"), [
        mode.h, FIT_INTR, 2.0, Buf(np.float64, (NV, 6), copy_of=views), NV,
        Buf(np.float64, (NC, 3), own=obj), Buf(np.float64, (NV, NC, 2), copy_of=img), NC,
        Buf(np.float64, (NV, _lib.PER_VIEW), own=pv), Buf(np.float64, (_lib.SHARED,), own=sh)] + mode.tail)


@pytest.mark.parametrize("with_distortion", [True, False])
def test_lm_fit_host(rec, with_distortion):
    views0, obj, img = _pts((NV, 6), seed=1), _pts((NC, 3), np.float32, 2), _pts((NV, NC, 2), seed=3)
    intr0 = (120.0, 100.0, 40.0, 50.0, -0.25)
    r = lm.lm_fit_host(intr0, views0, obj, img, checker_size=0.5, aspect=1.5, with_distortion=with_distortion,
                       max_iter=7, eps=1e-5)
    k = -0.25 if with_distortion else 0.0
    assert set(r) == {"intr", "views", "rms", "iterations"}
    assert r["intr"] == (150.0, 100.0, 40.0, 50.0, k) and r["rms"] == 0.0 and r["iterations"] == 0
    assert isinstance(r["views"], np.ndarray) and r["views"].shape == (NV, 6) and _addr(r["views"]) == _addr(views0)
    _expect(rec, "cc_lm_fit_f64_host", [
        _H, (150.0, 100.0, 40.0, 50.0, k, 0.5), 1.5, 15 if with_distortion else 7, Buf(np.float64, (NV, 6), own=views0),
        NV, Buf(np.float64, (NC, 3), copy_of=obj), Buf(np.float64, (NV, NC, 2), own=img), NC, 7, 1e-5, 0.0, 0])


def test_lm_fit_host_copies_other_views(rec):
    views0, obj, img = _pts((NV * 6,), seed=1).tolist(), _pts((NC, 3)), _pts((NV, NC, 2))
    r = lm.lm_fit_host((1.0, 2.0, 3.0, 4.0, 0.5), views0, obj, img, device=0)
    assert isinstance(r["views"], np.ndarray) and r["views"].shape == (NV, 6) and r["intr"] == (2.0, 2.0, 3.0, 4.0, 0.5)
    _expect(rec, "cc_lm_fit_f64_host", [_H, (2.0, 2.0, 3.0, 4.0, 0.5, 1.0), 1.0, 15,
                                        Buf(np.float64, (NV, 6), own=r["views"], values=np.reshape(views0, (NV, 6))),
                                        NV, Buf(np.float64, (NC, 3), own=obj), Buf(np.float64, (NV, NC, 2), own=img),
                                        NC, 30, 1e-3, 0.0, 0])


# ---------------------------------------------------------------- the board helpers
def test_get_ratio(rec):
    ip = _pts((3, 4, 2))
    assert cal.get_ratio(ip, 2.5) == 0.0
    _expect(rec, "cc_get_ratio", [Buf(np.float64, (12,), values=ip[:, :, 0].T.ravel()),
                                  Buf(np.float64, (12,), values=ip[:, :, 1].T.ravel()), 3, 4, 2.5, 0.0])
    flat = ip.transpose(1, 0, 2).reshape(12, 2)
    assert cal.get_ratio(flat.astype(np.float32), 1, n_corners=(3, 4)) == 0.0
    _expect(rec, "cc_get_ratio", [Buf(np.float64, (12,), values=ip[:, :, 0].T.ravel().astype(np.float32)),
                                  Buf(np.float64, (12,), values=ip[:, :, 1].T.ravel().astype(np.float32)), 3, 4, 1.0,
                                  0.0])
    _rejects(rec, ValueError, lambda: cal.get_ratio(flat, 1.0))
    _rejects(rec, ValueError, lambda: cal.get_ratio(flat, 1.0, n_corners=(4, 4)))


def test_get_axes(rec):
    assert cal.get_axes(0.75, 2, np.array([5, 8]), (375.0, 500)) == (0, 0)
    _expect(rec, "cc_get_axes", [0.75, 2.0, 5, 8, 375, 500, [0, 0]])


# ---------------------------------------------------------------- CUDA only: outputs are CUDA tensors
@pytest.mark.gpu
@pytest.mark.parametrize("coord", ["f64", "f32"])
def test_rectify_map(rec, cuda, coord):
    mr, mc = cal.rectify_map(_cal(), None, 0.5, (-3, 4), (8, 6), coord=coord)
    dt = np.float64 if coord == "f64" else np.float32
    _ret(mr, cuda, (6, 8), dt)
    _ret(mc, cuda, (6, 8), dt)
    _expect(rec, f"cc_rectify_map_{coord}", [cuda.h, INTR, VIEW[1], 0.5, [-3, 4], Buf(dt, (6, 8), own=mr),
                                             Buf(dt, (6, 8), own=mc), 8, 6, 8] + cuda.tail)
    mr, _ = cal.rectify_map(_cal(), 0, 2.0, (1, 1), (3, 2), device=cuda.device.index, coord=coord)
    _ret(mr, cuda, (2, 3), dt)
    assert rec.calls.pop().name == f"cc_rectify_map_{coord}"


@pytest.mark.gpu
def test_lm_steps(rec, cuda):
    pv = cuda.to(_pts((NV, _lib.PER_VIEW)))
    yz, schur = lm.lm_schur(pv, 0.125)
    _ret(yz, cuda, (NV, _lib.LM_YZ), np.float64)
    _ret(schur, cuda, (_lib.LM_SCHUR,), np.float64)
    _expect(rec, "cc_lm_schur_f64", [cuda.h, Buf(np.float64, pv.shape, own=pv), NV, 0.125,
                                     Buf(np.float64, (NV, _lib.LM_YZ), own=yz),
                                     Buf(np.float64, (_lib.LM_SCHUR,), own=schur)] + cuda.tail)
    yz0, _ = lm.lm_schur(pv[:0], 1.0)
    _ret(yz0, cuda, (1, _lib.LM_YZ), np.float64)
    rec.calls.clear()
    sh, views = cuda.to(_pts((_lib.SHARED,))), cuda.to(_pts((NV, 6)))
    out, delta = lm.lm_update(sh, schur, 0.5, lm.FREE_NO_K, yz, views)
    _ret(out, cuda, (NV, 6), np.float64)
    _ret(delta, cuda, (_lib.LM_DELTA,), np.float64)
    _expect(rec, "cc_lm_update_f64", [cuda.h, Buf(np.float64, sh.shape, own=sh), Buf(np.float64, schur.shape, own=schur),
                                      0.5, 7, Buf(np.float64, yz.shape, own=yz), Buf(np.float64, (NV, 6), own=views),
                                      NV, Buf(np.float64, (NV, 6), own=out),
                                      Buf(np.float64, (_lib.LM_DELTA,), own=delta)] + cuda.tail)


@pytest.mark.gpu
@pytest.mark.parametrize("views_kind", ["numpy", "cuda_f64", "cuda_f32"])
def test_lm_fit_device(rec, cuda, views_kind):
    v = _pts((NV, 6), seed=1)
    views0 = {"numpy": v, "cuda_f64": cuda.to(v), "cuda_f32": cuda.to(v.astype(np.float32))}[views_kind]
    before = _host(views0).copy()
    obj, img = cuda.to(_pts((NC, 3), seed=2)), _pts((NV, NC, 2), seed=3)
    r = lm.lm_fit_device((120.0, 100.0, 40.0, 50.0, -0.25), views0, obj, img, checker_size=0.5, aspect=1.5,
                         with_distortion=False, max_iter=9, eps=1e-4)
    assert set(r) == {"intr", "views", "views_device", "rms", "iterations"}
    assert r["intr"] == (150.0, 100.0, 40.0, 50.0, 0.0) and r["rms"] == 0.0 and r["iterations"] == 0
    _ret(r["views_device"], cuda, (NV, 6), np.float64)
    assert isinstance(r["views"], np.ndarray) and np.array_equal(r["views"], before.astype(np.float64))
    _expect(rec, "cc_lm_fit_f64", [
        cuda.h, (150.0, 100.0, 40.0, 50.0, 0.0, 0.5), 1.5, 7,
        Buf(np.float64, (NV, 6), own=r["views_device"], copy_of=views0), NV, Buf(np.float64, (NC, 3), own=obj),
        Buf(np.float64, (NV, NC, 2), copy_of=img), NC, 9, 1e-4, 0.0, 0] + cuda.tail)
    assert np.array_equal(_host(views0), before)                 # views0 itself is never written


@pytest.mark.gpu
def test_initial_guess_device(rec, cuda):
    obj, img = _pts((NC, 3), np.float32, 2), cuda.to(_pts((NV * NC, 2), seed=3))
    intr, views = lm.initial_guess_device(obj, img, (640, 480), aspect=0.5)
    assert intr == (1.0, 1.0, 0.0, 0.0, 0.0)
    _ret(views, cuda, (NV, 6), np.float64)
    _expect(rec, "cc_lm_initial_guess_f64", [cuda.h, Buf(np.float64, (NC, 3), copy_of=obj),
                                             Buf(np.float64, (NV, NC, 2), own=img.view(NV, NC, 2)), NV, NC, 640, 480,
                                             0.5, (1.0, 1.0, 0.0, 0.0, 0.0, 1.0), Buf(np.float64, (NV, 6), own=views)]
            + cuda.tail)
