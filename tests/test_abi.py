"""CPU tests of the boundary: the C-ABI library loads, exports every symbol that
include/camcal_b200.h declares, fails loudly without a device, and the host-only helpers agree
with the oracle.  No compute entry point is called here."""
import ctypes as C
import json
import os
import re

import numpy as np
import pytest

from conftest import ROOT
from oracle import oracle_c as oc


@pytest.fixture(scope="module")
def cc():
    import cameracalibrations_b200 as m
    return m


def _header_params():
    """{name: ["ptr" | "scalar" per parameter]} of every function include/camcal_b200.h declares"""
    hdr = open(os.path.join(ROOT, "include", "camcal_b200.h")).read()
    hdr = re.sub(r"/\*.*?\*/", "", hdr, flags=re.S)
    out = {}
    for name, params in re.findall(r"\b(cc_[a-z0-9_]+)\s*\(([^)]*)\)\s*;", hdr):
        ps = [p.strip() for p in params.split(",") if p.strip() and p.strip() != "void"]
        out[name] = ["ptr" if ("*" in p or "[" in p) else "scalar" for p in ps]
    return out


def _julia_ccalls():
    """[(name, ["ptr" | "scalar" per argument])] of every ccall into libcamcal in the Julia shim"""
    src = open(os.path.join(ROOT, "julia", "CameraCalibrationsB200.jl")).read()
    calls = []
    for m in re.finditer(r"ccall\(\(:(cc_[a-z0-9_]+),\s*libcamcal\),\s*\w+,\s*\(", src):
        i, depth = m.end(), 1                   # the argument-type tuple: up to its matching ')'
        j = i
        while depth:
            depth += {"(": 1, ")": -1}.get(src[j], 0)
            j += 1
        types, depth, cur = [], 0, ""
        for ch in src[i:j - 1]:
            if ch in "({":
                depth += 1
            elif ch in ")}":
                depth -= 1
            if ch == "," and depth == 0:
                types.append(cur.strip())
                cur = ""
            else:
                cur += ch
        if cur.strip():
            types.append(cur.strip())
        calls.append((m.group(1), ["ptr" if re.match(r"(Ptr|Ref)\{", t) else "scalar" for t in types]))
    return calls


def test_library_exports_every_declared_symbol(cc):
    from cameracalibrations_b200 import _lib
    names = sorted(_header_params())
    assert len(names) >= 30
    for n in names:
        assert hasattr(_lib.lib, n), f"{n} declared in include/camcal_b200.h but not exported"
    assert set(names) == set(_lib.EXPORTS)          # the ctypes table binds all of them
    assert _lib.lib.cc_abi_version() == 1


def test_bindings_pass_pointers_where_the_header_takes_them(cc):
    """Every ctypes signature and every Julia ccall passes a pointer exactly where include/camcal_b200.h declares
    one, and a scalar everywhere else."""
    from cameracalibrations_b200 import _lib
    hdr = _header_params()
    for name, (_, args) in _lib._SIGS.items():
        kinds = ["ptr" if a in (C.c_void_p, C.c_char_p) or issubclass(a, C._Pointer) else "scalar" for a in args]
        assert kinds == hdr[name], (name, kinds, hdr[name])
    calls = _julia_ccalls()
    assert len(calls) >= 29
    for name, kinds in calls:
        assert name in hdr and kinds == hdr[name], (name, kinds, hdr.get(name))


def test_no_cpu_fallback(cc):
    import torch
    if torch.cuda.is_available():
        pytest.skip("a device is present")
    with pytest.raises(cc.CamcalError) as e:
        cc.Context(0)
    assert e.value.status == -2                     # CC_ERR_NO_DEVICE
    c = cc.Calibration((100.0, 100.0, 50.0, 50.0), [((0, 0, 0), (0, 0, 1.0))], 1.0, 0.0, ["extrinsic.png"])
    with pytest.raises(cc.CamcalError):
        c(np.zeros((4, 2)))                          # host entry point: still needs the GPU


def test_argument_errors_are_status_codes(cc):
    from cameracalibrations_b200 import _lib
    out = C.c_double()
    assert _lib.lib.cc_get_ratio(None, None, 5, 8, 1.0, C.byref(out)) == -1
    assert b"NULL" in _lib.lib.cc_last_error_string()
    assert _lib.lib.cc_ctx_create(0, None) == -1
    n = C.c_uint64()
    assert _lib.lib.cc_ctx_launch_count(None, C.byref(n)) == -1
    assert _lib.lib.cc_ctx_destroy(None) == 0


def test_get_ratio_get_axes_match_oracle(cc, example_fit):
    n1, n2 = example_fit["n_corners"]
    for vi in range(6):
        ip = example_fit["corners_np"][vi].reshape(n2, n1, 2).transpose(1, 0, 2)
        r = cc.get_ratio(ip, 1.0)
        assert r == oc.get_ratio(ip, 1.0)
        assert cc.get_axes(r, 1.0, (n1, n2), example_fit["sz"]) == oc.get_axes(r, 1.0, (n1, n2), example_fit["sz"])
    ip = example_fit["corners_np"][0].reshape(n2, n1, 2).transpose(1, 0, 2)
    assert cc.get_axes(cc.get_ratio(ip, 1.0), 1.0, (n1, n2), (375, 500)) == (-112, -119)   # SURVEY Appendix A


def test_calibration_object_and_json_round_trip(cc, tmp_path, example_fit):
    """test/runtests.jl:88-98: save -> load preserves files (and here also the numbers)."""
    rng = np.random.default_rng(0)
    for _ in range(20):
        org = cc.Calibration(rng.random(4), [(rng.random(3), rng.random(3)) for _ in range(5)],
                             rng.random(), rng.random(), ["".join(rng.choice(list("abcdefgh"), 5)) for _ in range(5)])
        f = tmp_path / "calibration.json"
        cc.save(f, org)
        copy = cc.load(f)
        assert org.files == copy.files
        assert org.intrinsic == copy.intrinsic and org.extrinsics == copy.extrinsics
        assert org.scale == copy.scale and org.k == copy.k
    d = json.load(open(f))
    assert set(d) == {"intrinsic", "extrinsics", "scale", "k", "files"}      # CalibrationIO, src/io.jl:9-15
    # a rotation stored as a 3x3 matrix (column-major) loads to the same rotation vector
    from oracle import oracle_np as on
    rv = np.array([0.3, -0.2, 0.5])
    d["extrinsics"][0]["linear"] = on.rodrigues(rv).T.ravel().tolist()
    json.dump(d, open(f, "w"))
    np.testing.assert_allclose(cc.load(f).extrinsics[0][0], rv, atol=1e-12)


def test_view_index_semantics(cc):
    c = cc.Calibration((1.0, 1.0, 0.0, 0.0), [((0, 0, 0), (0, 0, 1.0))] * 3, 1.0, 0.0, ["a.png", "x_extrinsic_1.png", "b.png"])
    assert c._index(None) == 1 and c._index("b.png") == 2 and c._index(0) == 0
    with pytest.raises(IndexError):
        c._index(3)
    with pytest.raises(ValueError):
        c._index("missing.png")
    assert c.checker_size == 1.0


def test_ingest_and_group_entry_points_fail_loudly_without_a_device(cc):
    """No CPU decode path, no silent success: without a CUDA device the JPEG ingest and the multi-device
    context return status codes; bad arguments are rejected before anything else."""
    import torch
    from cameracalibrations_b200 import _lib
    assert _lib.lib.cc_jpeg_info(None, 0, None, None, None) == -1
    assert _lib.lib.cc_jpeg_decode_u8c3(None, None, None, 1, None, 4, 4, 4, 16, None) == -1
    assert _lib.lib.cc_ctx_create_group(0, None, None) == -1
    assert _lib.lib.cc_allreduce_shared_group(None, 0, None, 0, None) == -1
    if torch.cuda.is_available():
        return
    with pytest.raises(cc.CamcalError):
        cc.jpeg_info(b"\xff\xd8\xff\xe0 definitely not a complete jpeg")
    devs = (C.c_int * 1)(0)
    ctxs = (C.c_void_p * 1)()
    assert _lib.lib.cc_ctx_create_group(1, devs, ctxs) == -2 and not ctxs[0]      # CC_ERR_NO_DEVICE


def test_draw_crosses_is_the_reference_rule():
    """draw_crosses!, src/plot_calibration.jl:24-28: radius = round(|ij[1] - ij[n1]| / n1 / 5), a horizontal and a
    vertical bar of +-radius through every rounded corner, clipped at the frame."""
    from cameracalibrations_b200.plotting import _draw_crosses
    frame = np.zeros((40, 60, 3), dtype=np.uint8)              # frame layout [c][r]: sz1 = 60 rows, sz2 = 40 columns
    pts = np.array([[10.2, 5.4], [30.0, 5.0], [50.4, 5.0], [59.6, 39.7]])     # (row, col), 1-based; n1 = 3
    _draw_crosses(frame, pts, 3, (255, 0, 0))
    radius = int(np.rint(np.hypot(10 - 50, 0) / 3 / 5))        # = 3
    assert radius == 3
    assert np.all(frame[4, 9 - 3:9 + 4, 0] == 255) and frame[4, 9 - 4, 0] == 0 and frame[4, 9 + 4, 0] == 0    # along the rows
    assert np.all(frame[4 - 3:4 + 4, 9, 0] == 255) and frame[4 + 4, 9, 0] == 0                               # along the columns
    assert np.all(frame[39, 56:60, 0] == 255) and np.all(frame[36:40, 59, 0] == 255)                          # clipped at the corner
    assert frame[..., 1].max() == 0 and frame[..., 2].max() == 0


def _build_c_consumer(tmp_path):
    import shutil
    import subprocess
    if shutil.which("gcc") is None:
        pytest.skip("no gcc")
    libdir = os.path.join(ROOT, "cameracalibrations_b200")
    exe = str(tmp_path / "abi_consumer")
    r = subprocess.run(["gcc", "-std=c99", "-Wall", "-Wextra", "-pedantic", "-Werror", "-I", os.path.join(ROOT, "include"),
                        os.path.join(ROOT, "tests", "c", "abi_consumer.c"), "-o", exe, "-L", libdir, "-lcamcal_b200", "-lm",
                        "-Wl,-rpath," + libdir], capture_output=True, text=True)
    assert r.returncode == 0, r.stderr                    # the header is valid strict C99 and every symbol links
    return subprocess.run([exe], capture_output=True, text=True)


def test_plain_c_consumer_of_the_abi(tmp_path):
    """include/camcal_b200.h + the .so from C, no Python or torch in between: the host helpers work, and a box
    without a GPU gets CC_ERR_NO_DEVICE (printed as 'no device'), never a CPU result."""
    import torch
    r = _build_c_consumer(tmp_path)
    assert r.returncode == 0, r.stdout + r.stderr
    assert r.stdout.strip() == ("ok" if torch.cuda.is_available() else "no device")
