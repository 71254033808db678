"""Argument errors of the rectification entry points.

Every single-fault case runs through all eight frame entry points (cc_rectify_{f32c1,u8c3}, their `_host` and
`_views` forms and cc_rectify_views_{f32c1,u8c3}_host), and the cases that apply to a map through
cc_rectify_map_{f64,f32}.  Each must return CC_ERR_INVALID_ARG with a message that names the fault, leave every output
byte at its sentinel and make no launch.  Zero views, zero frames per view and zero frames return 0 and write nothing.
"""
import ctypes as C
import re

import numpy as np
import pytest

torch = pytest.importorskip("torch")

from test_gpu_batching import F_FILL, F_SENT, U_FILL, U_SENT, _frames_f32, _frames_u8
from test_gpu_rectify_views_host import _Views

SZ = (64, 48)
NV, FPV = 3, 2                # the `_views` forms: 3 views of 2 frames; the single-view forms: view 1, 6 frames
FRAME_ENTRIES = [(fmt, form) for fmt in ("f32", "u8") for form in ("device", "host", "views", "views_host")]
BIG_PITCH = 1 << 25           # pitch * sz2 >= 2^30


@pytest.fixture(scope="module")
def cc():
    import cameracalibrations_b200 as m
    assert torch.cuda.is_available(), "GPU tests need a CUDA device"
    m.context(0)
    return m


@pytest.fixture(scope="module")
def vs(cc):
    return _Views(cc, NV, SZ, scale=0.021)


def _lib():
    from cameracalibrations_b200 import _lib as lib
    return lib


def _bad_intr(vs, **kv):
    intr = type(vs.c._intr).from_buffer_copy(vs.c._intr)
    for k, v in kv.items():
        setattr(intr, k, v)
    return intr


# name -> (arguments replaced, message pattern, forms it applies to: "frames" all eight, "views" the `_views` forms,
# "u8" the u8c3 forms, "map" the map entry points).  The single-view forms and the maps take view 1 of the arrays.
# Where the parent library worded a fault differently in its single-view and `_views` forms, the pattern accepts
# either wording.
def _cases(vs):
    bad_axs = (C.c_int64 * (2 * NV))(0, 0, 1 << 31, 0, 0, 0)
    bad_ratios = (C.c_double * NV)(vs.ratios[0], -1.0, vs.ratios[2])
    return {
        "ctx": (dict(ctx=None), r"NULL", "frames map"),
        "intr": (dict(intr=None), r"NULL", "frames map"),
        "view": (dict(views=None), r"NULL", "frames map"),
        "ratios": (dict(ratios=None), r"NULL", "views"),
        "axs": (dict(axs=None), r"NULL", "frames map"),
        "nviews<0": (dict(nviews=-1), r"bad counts", "views"),
        "frames<0": (dict(n=-1), r"bad counts|frame size must be positive", "frames"),
        "65536 frames": (dict(n=65536), r"at most 65535 frames", "frames"),
        "focal": (dict(intr=C.byref(_bad_intr(vs, frow=0.0))), r"focal lengths must be non-zero", "frames map"),
        "checker": (dict(intr=C.byref(_bad_intr(vs, checker_size=0.0))), r"checker_size must be non-zero", "frames map"),
        "ratio": (dict(ratios=bad_ratios), r"ratio must be positive", "frames map"),
        "axs range": (dict(axs=bad_axs), r"axs_min out of range", "frames map"),
        "sz1": (dict(sz1=0), r"frame size must be positive", "frames map"),
        "sz2": (dict(sz2=-4), r"frame size must be positive", "frames map"),
        "extent": (dict(sz2=1 << 22), r"frame extent must be < 2\^22", "frames map"),
        "pitch": (dict(pitch=SZ[0] - 1), r"pitch smaller than sz1", "frames map"),
        "overlap": (dict(stride=SZ[0] * SZ[1] - 1), r"frames overlap", "frames"),
        "too large": (dict(pitch=BIG_PITCH, stride=BIG_PITCH * SZ[1]), r"frame too large", "frames map"),
        "src": (dict(src=None), r"NULL frame pointer", "frames"),
        "dst": (dict(dst=None), r"NULL frame pointer", "frames"),
        "in place": (dict(src="dst"), r"in place", "frames"),
        "fill": (dict(fill=None), r"fill is NULL", "u8"),
        "map_row": (dict(map_row=None), r"NULL map pointer", "map"),
        "map_col": (dict(map_col=None), r"NULL map pointer", "map"),
    }


def _view1(a):
    """view, ratio and axes of view 1 of the arrays in a, for the single-view entry points"""
    def at(arr, t):                              # element 1 of a View array, pair 1 of an axes array
        return None if arr is None else C.cast(C.addressof(arr) + C.sizeof(t), C.POINTER(arr._type_))
    return [at(a["views"], _lib().View), a["ratios"][1], at(a["axs"], C.c_int64 * 2)]


def _common_args(cc, vs):
    lib = _lib()
    return dict(ctx=cc.context(0).handle, intr=C.byref(vs.c._intr),
                views=(lib.View * NV)(*[vs.c._views[i] for i in range(NV)]), nviews=NV,
                ratios=(C.c_double * NV)(*vs.ratios), axs=(C.c_int64 * (2 * NV))(*[x for am in vs.axss for x in am]))


class _Call:
    """One entry point with valid arguments on sentinel-filled outputs; call(**over) replaces arguments.  For the
    frame entry points n is nframes (single view) or frames per view (`_views` forms)."""

    def __init__(self, cc, vs, fmt, form, sz=SZ):
        lib = _lib()
        self.cc, self.vs, self.fmt, self.form, self.sz = cc, vs, fmt, form, sz
        self.many = form.startswith("views")
        self.on_host = form.endswith("host")
        n = NV * FPV
        frames = _frames_f32(n, sz, 4100) if fmt == "f32" else _frames_u8(n, sz, 4100)
        sent = np.array(F_SENT if fmt == "f32" else U_SENT, frames.dtype)
        self.src = frames if self.on_host else torch.from_numpy(frames).cuda()
        if self.on_host:
            self.out = np.empty_like(frames)
            self.out[...] = sent
        else:
            self.out = torch.empty_like(self.src)
            self.out[...] = torch.from_numpy(sent).cuda()
        self.ref = self._bytes()
        self.args = dict(_common_args(cc, vs), src=self._ptr(self.src), dst=self._ptr(self.out), sz1=sz[0],
                         sz2=sz[1], pitch=sz[0], stride=sz[0] * sz[1], n=FPV if self.many else n,
                         fill=C.c_float(F_FILL) if fmt == "f32" else (C.c_uint8 * 3)(*U_FILL), flags=lib.COORD_F64)
        name = "cc_rectify_" + ("views_" if form == "views_host" else "") + ("f32c1" if fmt == "f32" else "u8c3")
        name += {"device": "", "host": "_host", "views": "_views", "views_host": "_host"}[form]
        self.fn = getattr(lib.lib, name)

    @staticmethod
    def _ptr(a):
        return C.c_void_p(a.ctypes.data if isinstance(a, np.ndarray) else a.data_ptr())

    def _bytes(self):
        if not self.on_host:
            torch.cuda.synchronize()
        o = self.out if self.on_host else self.out.cpu().numpy()
        return o.tobytes()

    def __call__(self, **over):
        a = dict(self.args)
        a.update(over)
        if isinstance(a["src"], str):
            a["src"] = a[a["src"]]
        pos = [a["ctx"], a["intr"]]
        pos += [a["views"], a["nviews"], a["ratios"], a["axs"]] if self.many else _view1(a)
        pos += [a["src"], a["dst"], a["sz1"], a["sz2"], C.c_size_t(a["pitch"]), C.c_size_t(a["stride"]), a["n"],
                a["fill"], a["flags"]]
        if not self.on_host:
            pos.append(None)
        return self.fn(*pos)

    def untouched(self):
        return self._bytes() == self.ref


class _MapCall:
    """cc_rectify_map_{f64,f32} on sentinel-filled device maps"""

    def __init__(self, cc, vs, prec):
        dt = torch.float64 if prec == "f64" else torch.float32
        self.row = torch.full((SZ[1], SZ[0]), -777.0, dtype=dt, device="cuda")
        self.col = torch.full((SZ[1], SZ[0]), -555.0, dtype=dt, device="cuda")
        self.ref = self._bytes()
        self.args = dict(_common_args(cc, vs), map_row=C.c_void_p(self.row.data_ptr()),
                         map_col=C.c_void_p(self.col.data_ptr()), sz1=SZ[0], sz2=SZ[1], pitch=SZ[0])
        self.fn = _lib().lib.cc_rectify_map_f64 if prec == "f64" else _lib().lib.cc_rectify_map_f32

    def _bytes(self):
        torch.cuda.synchronize()
        return self.row.cpu().numpy().tobytes() + self.col.cpu().numpy().tobytes()

    def __call__(self, **over):
        a = dict(self.args)
        a.update(over)
        return self.fn(a["ctx"], a["intr"], *_view1(a), a["map_row"], a["map_col"], a["sz1"], a["sz2"],
                       C.c_size_t(a["pitch"]), None)

    def untouched(self):
        return self._bytes() == self.ref


def _check(cc, call, over, pattern, what):
    lib = _lib()
    n0 = cc.context(0).launch_count()
    rc = call(**over)
    msg = lib.last_error()
    assert rc == lib.CC_ERR_INVALID_ARG, (what, rc, msg)
    assert re.search(pattern, msg), (what, msg)
    assert call.untouched(), what
    assert cc.context(0).launch_count() == n0, what


@pytest.mark.gpu
@pytest.mark.parametrize("fmt,form", FRAME_ENTRIES)
def test_frame_entry_argument_errors(cc, vs, fmt, form):
    call = _Call(cc, vs, fmt, form)
    for what, (over, pattern, applies) in _cases(vs).items():
        if "frames" in applies or ("views" in applies and call.many) or ("u8" in applies and fmt == "u8"):
            if what == "65536 frames" and call.many:
                over = dict(n=65536 // NV + 1)
            _check(cc, call, over, pattern, what)


@pytest.mark.gpu
@pytest.mark.parametrize("prec", ["f64", "f32"])
def test_map_entry_argument_errors(cc, vs, prec):
    call = _MapCall(cc, vs, prec)
    for what, (over, pattern, applies) in _cases(vs).items():
        if "map" in applies:
            _check(cc, call, over, pattern, what)


@pytest.mark.gpu
@pytest.mark.parametrize("fmt,form", FRAME_ENTRIES)
def test_nothing_to_do(cc, vs, fmt, form):
    """zero views, zero frames per view, zero frames: status 0, nothing written, no launch"""
    call = _Call(cc, vs, fmt, form)
    for over in ((dict(nviews=0), dict(n=0)) if call.many else (dict(n=0),)):
        n0 = cc.context(0).launch_count()
        assert call(**over) == 0, (over, _lib().last_error())
        assert call.untouched(), over
        assert cc.context(0).launch_count() == n0, over


@pytest.mark.gpu
@pytest.mark.parametrize("form", ["host", "views_host"])
def test_gather_tma_unavailable(cc, form):
    """CC_GATHER_TMA on frames TMA cannot address (131 fp32 pixels per line: the slot lines are not 16-byte aligned)
    is an argument error the library reports; dst stays untouched"""
    sz = (131, 40)
    vs = _Views(cc, NV, sz, scale=0.023)
    call = _Call(cc, vs, "f32", form, sz=sz)
    _check(cc, call, dict(flags=_lib().GATHER_TMA | _lib().COORD_F64), r"TMA gather not available", "tma")
