"""Reference of the rectification into output axes of any size (tests/c/rectify_axes_ref.c), for the tests of
cc_rectify_axes_*.  TEST INFRASTRUCTURE ONLY.  The C file is compiled on first use into a temporary directory with
the oracle's flags (oracle/Makefile: only the explicit fma() calls fuse) and linked against the oracle, whose
cco_rectify_coord gives every output index its source coordinate.  Chains are oracle.oracle_c.chain()."""
import ctypes as C
import os
import shutil
import subprocess
import tempfile

import numpy as np

from oracle import oracle_c as oc

_HERE = os.path.dirname(os.path.abspath(__file__))
_ORACLE = os.path.join(os.path.dirname(_HERE), "oracle")
_lib = None


def lib():
    global _lib
    if _lib is None:
        so = oc.build()                                     # the oracle the reference links against
        cc = shutil.which("/usr/bin/gcc") or shutil.which("gcc")
        assert cc, "the rectification reference needs gcc"
        out = os.path.join(tempfile.mkdtemp(prefix="camcal_ref_"), "librectify_axes_ref.so")
        subprocess.check_call([cc, "-O2", "-std=c99", "-fPIC", "-ffp-contract=off", "-mfma", "-fno-fast-math",
                               "-Wall", "-Wextra", "-shared", "-I", _ORACLE,
                               os.path.join(_HERE, "c", "rectify_axes_ref.c"), "-o", out,
                               "-L", _ORACLE, "-l:" + os.path.basename(so), "-Wl,-rpath," + _ORACLE, "-lm"])
        C.CDLL(so, mode=C.RTLD_GLOBAL)
        _lib = C.CDLL(out)
        shutil.rmtree(os.path.dirname(out), ignore_errors=True)     # loaded: the file is no longer needed
    return _lib


def rectify_f32c1(ch, inv_ratio, axs_min, src, out_sz, fill=np.nan):
    """src: float32 (nframes, sz2, sz1); returns (nframes, out_sz2, out_sz1), dense"""
    src = np.ascontiguousarray(src, dtype=np.float32)
    nf, sz2, sz1 = src.shape
    o1, o2 = int(out_sz[0]), int(out_sz[1])
    dst = np.empty((nf, o2, o1), dtype=np.float32)
    lib().ref_rectify_f32c1_axes(C.byref(ch), C.c_double(inv_ratio), (C.c_longlong * 2)(*map(int, axs_min)),
                                 src.ctypes.data_as(C.POINTER(C.c_float)), sz1, sz2, C.c_size_t(sz1),
                                 C.c_size_t(sz1 * sz2), dst.ctypes.data_as(C.POINTER(C.c_float)), o1, o2,
                                 C.c_size_t(o1), C.c_size_t(o1 * o2), nf, C.c_float(fill))
    return dst


def rectify_u8c3(ch, inv_ratio, axs_min, src, out_sz, fill=(0, 0, 0)):
    """src: uint8 (nframes, sz2, sz1, 3); returns (nframes, out_sz2, out_sz1, 3), dense"""
    src = np.ascontiguousarray(src, dtype=np.uint8)
    nf, sz2, sz1, _ = src.shape
    o1, o2 = int(out_sz[0]), int(out_sz[1])
    dst = np.empty((nf, o2, o1, 3), dtype=np.uint8)
    lib().ref_rectify_u8c3_axes(C.byref(ch), C.c_double(inv_ratio), (C.c_longlong * 2)(*map(int, axs_min)),
                                src.ctypes.data_as(C.POINTER(C.c_uint8)), sz1, sz2, C.c_size_t(sz1),
                                C.c_size_t(sz1 * sz2), dst.ctypes.data_as(C.POINTER(C.c_uint8)), o1, o2,
                                C.c_size_t(o1), C.c_size_t(o1 * o2), nf, (C.c_uint8 * 3)(*[int(v) for v in fill]))
    return dst
