"""Argument errors of the fit entry points.

Every single-fault case runs through both forms of cc_reproj_jtj_f64, cc_calculate_errors_f64 and cc_lm_fit_f64 (the
device form and `_host`), and the cases of the stepwise and initial-guess entry points (cc_lm_schur_f64,
cc_lm_update_f64, cc_lm_initial_guess_f64) through those.  Each must return CC_ERR_INVALID_ARG with a message that
names the fault, leave every output at its sentinel and make no launch.  The device forms also reject an img that is
not 16-byte aligned; a calculate_errors call over the kernel's shared-memory cap is rejected by both forms before
anything is uploaded.
"""
import ctypes as C
import re

import numpy as np
import pytest

torch = pytest.importorskip("torch")

from oracle import oracle_c as oc

INTR = (466.7, 466.7, 180.0, 320.0, -0.12, 1.0)    # frow, fcol, crow, ccol, k, checker_size
NV, N1, N2, NS = 3, 6, 5, 7                         # views, board corners, inverse samples per view
NC = N1 * N2
N2_BIG = 400                                        # N1 x N2_BIG corners: over the calc_errors shared-memory cap
PAIRS = [(entry, form) for entry in ("reproj_jtj", "calculate_errors", "lm_fit") for form in ("device", "host")]


@pytest.fixture(scope="module")
def cc():
    import cameracalibrations_b200 as m
    assert torch.cuda.is_available(), "GPU tests need a CUDA device"
    m.context(0)
    return m


@pytest.fixture(scope="module")
def prob():
    """NV views of an N1 x N2 board seen through INTR, with noisy image points and inverse samples.  obj and img
    have room for N1 x N2_BIG corners, so a call past the cap that were accepted would still stay in bounds."""
    rng = np.random.default_rng(11)
    a, b = np.meshgrid(np.arange(N1, dtype=np.float64), np.arange(N2, dtype=np.float64), indexing="ij")
    obj = np.zeros((N1 * N2_BIG, 3))
    obj[:NC, 0], obj[:NC, 1] = a.ravel(), b.ravel()
    views = np.zeros((NV, 6))
    img = np.zeros((NV, N1 * N2_BIG, 2))
    for v in range(NV):
        views[v, :3] = rng.normal(0.0, 0.05, 3)
        views[v, 3:] = (-2.5 + 0.3 * v, -2.0, 12.0 + v)
        row, col = oc.world2img_soa(oc.chain(INTR, views[v, :3], views[v, 3:]), obj[:NC, 0], obj[:NC, 1])
        img[v, :NC, 0] = row + rng.normal(0.0, 0.2, NC)
        img[v, :NC, 1] = col + rng.normal(0.0, 0.2, NC)
    inv = rng.uniform(1.0, 300.0, (2, NV, NS))
    return dict(views=views, obj=obj, img=img, inv_rows=inv[0].copy(), inv_cols=inv[1].copy())


def _lib():
    from cameracalibrations_b200 import _lib as lib
    return lib


def _intr(**kv):
    intr = _lib().make_intr(*INTR)
    for k, v in kv.items():
        setattr(intr, k, v)
    return intr


def _ptr(a, offset=0):
    return C.c_void_p((a.ctypes.data if isinstance(a, np.ndarray) else a.data_ptr()) + offset)


def _bytes(o):
    if torch.is_tensor(o):
        torch.cuda.synchronize()
        return o.cpu().numpy().tobytes()
    return o.tobytes() if isinstance(o, np.ndarray) else bytes(o)


class _Call:
    """One entry point with valid arguments: `names` the C parameters in order, `args` their values; outputs (and the
    in/out arrays) start at a sentinel.  call(**over) replaces arguments by name."""

    def __init__(self, cc, fn, names, args, outs):
        self.cc, self.fn, self.names, self.args, self.outs = cc, fn, names, args, outs
        self.ref = [_bytes(o) for o in outs]

    def __call__(self, **over):
        a = dict(self.args)
        a.update(over)
        return self.fn(*[a[n] for n in self.names])

    def untouched(self):
        return [_bytes(o) for o in self.outs] == self.ref


def _arrays(prob, host, names):
    """the named problem arrays on the host (numpy) or the device (torch), and sentinel-filled outputs"""
    if host:
        return {n: np.ascontiguousarray(prob[n]) for n in names}
    return {n: torch.from_numpy(np.ascontiguousarray(prob[n])).cuda() for n in names}


def _out(host, shape, value=-777.0):
    return np.full(shape, value) if host else torch.full(shape, value, dtype=torch.float64, device="cuda")


def _pair_call(cc, prob, entry, form):
    lib, host = _lib(), form == "host"
    ctx = cc.context(0).handle
    arr = _arrays(prob, host, ("views", "obj", "img", "inv_rows", "inv_cols"))
    intr = _intr()
    stream = [] if host else [None]
    if entry == "reproj_jtj":
        pv, sh = _out(host, (NV, lib.PER_VIEW)), _out(host, (lib.SHARED,))
        names = ["ctx", "intr", "aspect", "views", "nviews", "obj", "img", "ncorners", "per_view", "shared"]
        args = dict(ctx=ctx, intr=C.byref(intr), aspect=1.0, views=_ptr(arr["views"]), nviews=NV, obj=_ptr(arr["obj"]),
                    img=_ptr(arr["img"]), ncorners=NC, per_view=_ptr(pv), shared=_ptr(sh))
        outs = [pv, sh]
    elif entry == "calculate_errors":
        sums = _out(host, (4,))
        names = ["ctx", "intr", "views", "nviews", "obj", "img", "n1", "n2", "inv_rows", "inv_cols", "samples", "sums"]
        args = dict(ctx=ctx, intr=C.byref(intr), views=_ptr(arr["views"]), nviews=NV, obj=_ptr(arr["obj"]),
                    img=_ptr(arr["img"]), n1=N1, n2=N2, inv_rows=_ptr(arr["inv_rows"]), inv_cols=_ptr(arr["inv_cols"]),
                    samples=NS, sums=_ptr(sums))
        outs = [sums]
    else:
        rms, its = C.c_double(-777.0), C.c_int(-777)
        names = ["ctx", "intr", "aspect", "free_mask", "views", "nviews", "obj", "img", "ncorners", "max_iter", "eps",
                 "rms", "iterations"]
        args = dict(ctx=ctx, intr=C.byref(intr), aspect=1.0, free_mask=15, views=_ptr(arr["views"]), nviews=NV,
                    obj=_ptr(arr["obj"]), img=_ptr(arr["img"]), ncorners=NC, max_iter=5, eps=0.0, rms=C.byref(rms),
                    iterations=C.byref(its))
        outs = [arr["views"], intr, rms, its]
    name = {"reproj_jtj": "cc_reproj_jtj_f64", "calculate_errors": "cc_calculate_errors_f64",
            "lm_fit": "cc_lm_fit_f64"}[entry] + ("_host" if host else "")
    fn = getattr(lib.lib, name)
    call = _Call(cc, lambda *a: fn(*a, *stream), names, args, outs)
    call.keep = (arr, intr)                          # the arguments' memory lives as long as the call
    return call


# entry -> [(name, arguments replaced, message pattern, forms it applies to)]; "img+8" is img 8 bytes past its start
NULL_PTR = r"NULL (device|host) pointer"
PAIR_CASES = {
    "reproj_jtj": [
        ("ctx", dict(ctx=None), r"NULL argument", "device host"),
        ("intr", dict(intr=None), r"NULL argument", "device host"),
        ("nviews<0", dict(nviews=-1), r"bad sizes", "device host"),
        ("ncorners", dict(ncorners=0), r"bad sizes", "device host"),
        ("shared", dict(shared=None), r"shared is NULL", "device host"),
        ("views", dict(views=None), NULL_PTR, "device host"),
        ("obj", dict(obj=None), NULL_PTR, "device host"),
        ("img", dict(img=None), NULL_PTR, "device host"),
        ("per_view", dict(per_view=None), NULL_PTR, "device host"),
        ("checker", dict(intr="checker0"), r"checker_size must be non-zero", "device host"),
        ("img align", dict(img="img+8"), r"img must be 16-byte aligned", "device"),
    ],
    "calculate_errors": [
        ("ctx", dict(ctx=None), r"NULL argument", "device host"),
        ("intr", dict(intr=None), r"NULL argument", "device host"),
        ("sums", dict(sums=None), r"NULL argument", "device host"),
        ("nviews<0", dict(nviews=-1), r"bad sizes", "device host"),
        ("n1", dict(n1=0), r"bad sizes", "device host"),
        ("n2", dict(n2=0), r"bad sizes", "device host"),
        ("samples<0", dict(samples=-1), r"bad sizes", "device host"),
        ("views", dict(views=None), NULL_PTR, "device host"),
        ("obj", dict(obj=None), NULL_PTR, "device host"),
        ("img", dict(img=None), NULL_PTR, "device host"),
        ("inv_rows", dict(inv_rows=None), r"NULL sample pointer", "device host"),
        ("inv_cols", dict(inv_cols=None), r"NULL sample pointer", "device host"),
        ("frow", dict(intr="frow0"), r"bad intrinsics", "device host"),
        ("fcol", dict(intr="fcol0"), r"bad intrinsics", "device host"),
        ("checker", dict(intr="checker0"), r"bad intrinsics", "device host"),
        ("img align", dict(img="img+8"), r"img must be 16-byte aligned", "device"),
        ("smem cap", dict(n2=N2_BIG), r"too many corners per view", "device host"),
    ],
    "lm_fit": [
        ("ctx", dict(ctx=None), r"NULL argument", "device host"),
        ("intr", dict(intr=None), r"NULL argument", "device host"),
        ("obj", dict(obj=None), r"NULL argument", "device host"),
        ("views", dict(views=None), r"NULL", "device host"),
        ("img", dict(img=None), r"NULL", "device host"),
        ("nviews<0", dict(nviews=-1), r"bad sizes", "device host"),
        ("nviews=0", dict(nviews=0), r"bad sizes", "host"),
        ("ncorners", dict(ncorners=0), r"bad sizes", "device host"),
        ("free_mask 0", dict(free_mask=0), r"free_mask", "device host"),
        ("free_mask 16", dict(free_mask=16), r"free_mask", "device host"),
        ("max_iter", dict(max_iter=-1), r"bad stopping rule", "device host"),
        ("eps", dict(eps=-1.0), r"bad stopping rule", "device host"),
        ("aspect", dict(aspect=0.0), r"bad starting intrinsics", "device host"),
        ("fcol", dict(intr="fcol0"), r"bad starting intrinsics", "device host"),
        ("checker", dict(intr="checker0"), r"bad starting intrinsics", "device host"),
        ("img align", dict(img="img+8"), r"img must be 16-byte aligned", "device"),
    ],
}
BAD_INTR = {"frow0": dict(frow=0.0), "fcol0": dict(fcol=0.0), "checker0": dict(checker_size=0.0)}


def _resolve(call, over):
    """symbolic replacements: a bad copy of the intrinsics, img 8 bytes past its start"""
    over = dict(over)
    if isinstance(over.get("intr"), str):
        bad = _intr(**BAD_INTR[over["intr"]])
        call.keep = call.keep + (bad,)
        over["intr"] = C.byref(bad)
    if over.get("img") == "img+8":
        over["img"] = _ptr(call.keep[0]["img"], 8)
    return over


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
@pytest.mark.parametrize("entry,form", PAIRS)
def test_fit_pair_argument_errors(cc, prob, entry, form):
    call = _pair_call(cc, prob, entry, form)
    for what, over, pattern, forms in PAIR_CASES[entry]:
        if form in forms.split():
            _check(cc, call, _resolve(call, over), pattern, what)


def _stepwise_calls(cc):
    """cc_lm_schur_f64, cc_lm_update_f64 and cc_lm_initial_guess_f64 with valid device arguments"""
    lib = _lib()
    ctx = cc.context(0).handle
    d = lambda *shape: torch.zeros(shape, dtype=torch.float64, device="cuda")
    pv, yz, schur, shared = d(NV, lib.PER_VIEW), _out(False, (NV, lib.LM_YZ)), _out(False, (lib.LM_SCHUR,)), d(lib.SHARED)
    schur_in, vin, vout, delta = d(lib.LM_SCHUR), d(NV, 6), _out(False, (NV, 6)), _out(False, (lib.LM_DELTA,))
    obj, img, views = d(NC, 3), d(NV, NC, 2), _out(False, (NV, 6))
    intr = _intr()
    p = _ptr
    schur_call = _Call(cc, lambda *a: lib.lib.cc_lm_schur_f64(*a, None),
                       ["ctx", "per_view", "nviews", "lambda", "yz", "schur"],
                       dict(ctx=ctx, per_view=p(pv), nviews=NV, **{"lambda": 1e-3}, yz=p(yz), schur=p(schur)),
                       [yz, schur])
    update_call = _Call(cc, lambda *a: lib.lib.cc_lm_update_f64(*a, None),
                        ["ctx", "shared", "schur", "lambda", "free_mask", "yz", "views_in", "nviews", "views_out",
                         "delta"],
                        dict(ctx=ctx, shared=p(shared), schur=p(schur_in), **{"lambda": 1e-3}, free_mask=15, yz=p(yz),
                             views_in=p(vin), nviews=NV, views_out=p(vout), delta=p(delta)),
                        [vout, delta])
    guess_call = _Call(cc, lambda *a: lib.lib.cc_lm_initial_guess_f64(*a, None),
                       ["ctx", "obj", "img", "nviews", "ncorners", "sz1", "sz2", "aspect", "intr", "views"],
                       dict(ctx=ctx, obj=p(obj), img=p(img), nviews=NV, ncorners=NC, sz1=360, sz2=640, aspect=1.0,
                            intr=C.byref(intr), views=p(views)),
                       [intr, views])
    for c in (schur_call, update_call, guess_call):
        c.keep = (pv, yz, schur, shared, schur_in, vin, vout, delta, obj, img, views, intr)
    return dict(lm_schur=schur_call, lm_update=update_call, initial_guess=guess_call)


STEPWISE_CASES = {
    "lm_schur": [
        ("ctx", dict(ctx=None), r"NULL argument"),
        ("schur", dict(schur=None), r"NULL argument"),
        ("nviews<0", dict(nviews=-1), r"bad sizes"),
        ("per_view", dict(per_view=None), r"NULL device pointer"),
        ("yz", dict(yz=None), r"NULL device pointer"),
        ("lambda<0", {"lambda": -1.0}, r"lambda must be non-negative"),
        ("lambda nan", {"lambda": float("nan")}, r"lambda must be non-negative"),
    ],
    "lm_update": [
        ("ctx", dict(ctx=None), r"NULL argument"),
        ("shared", dict(shared=None), r"NULL argument"),
        ("schur", dict(schur=None), r"NULL argument"),
        ("delta", dict(delta=None), r"NULL argument"),
        ("nviews<0", dict(nviews=-1), r"bad sizes"),
        ("yz", dict(yz=None), r"NULL device pointer"),
        ("views_in", dict(views_in=None), r"NULL device pointer"),
        ("views_out", dict(views_out=None), r"NULL device pointer"),
        ("lambda<0", {"lambda": -1.0}, r"lambda must be non-negative"),
        ("lambda nan", {"lambda": float("nan")}, r"lambda must be non-negative"),
        ("free_mask 0", dict(free_mask=0), r"free_mask"),
        ("free_mask 16", dict(free_mask=16), r"free_mask"),
    ],
    "initial_guess": [
        ("ctx", dict(ctx=None), r"NULL argument"),
        ("intr", dict(intr=None), r"NULL argument"),
        ("obj", dict(obj=None), r"NULL argument"),
        ("nviews<0", dict(nviews=-1), r"bad sizes"),
        ("ncorners", dict(ncorners=3), r"bad sizes"),
        ("sz1", dict(sz1=0), r"bad sizes"),
        ("sz2", dict(sz2=0), r"bad sizes"),
        ("views", dict(views=None), r"NULL view / image-point array"),
        ("img", dict(img=None), r"NULL view / image-point array"),
    ],
}


@pytest.mark.gpu
@pytest.mark.parametrize("entry", list(STEPWISE_CASES))
def test_fit_stepwise_argument_errors(cc, entry):
    call = _stepwise_calls(cc)[entry]
    for what, over, pattern in STEPWISE_CASES[entry]:
        _check(cc, call, over, pattern, what)


@pytest.mark.gpu
@pytest.mark.parametrize("form", ["device", "host"])
def test_calculate_errors_no_views_needs_no_arrays(cc, prob, form):
    """nviews == 0 reads no array: NULL views, points and samples are accepted with inverse_samples > 0, and the four
    sums are 0"""
    call = _pair_call(cc, prob, "calculate_errors", form)
    rc = call(nviews=0, views=None, obj=None, img=None, inv_rows=None, inv_cols=None)
    assert rc == 0, _lib().last_error()
    sums = call.outs[0]
    sums = sums if isinstance(sums, np.ndarray) else sums.cpu().numpy()
    assert np.array_equal(sums, np.zeros(4))


@pytest.mark.gpu
def test_calculate_errors_host_is_the_device_form(cc, prob):
    """cc_calculate_errors_f64_host returns the device form's four raw sums bit for bit"""
    dev = _pair_call(cc, prob, "calculate_errors", "device")
    host = _pair_call(cc, prob, "calculate_errors", "host")
    assert dev() == 0 and host() == 0, _lib().last_error()
    a, b = dev.outs[0].cpu().numpy(), host.outs[0]
    assert np.all(np.isfinite(a)) and np.all(a > 0.0)
    assert a.tobytes() == b.tobytes(), (a, b)
