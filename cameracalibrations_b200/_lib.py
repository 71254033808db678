"""ctypes binding of libcamcal_b200.so (the C ABI in include/camcal_b200.h).

There is no CPU fallback anywhere in this package: if the shared library is missing
(`python __graft_entry__.py build` / `make -C cameracalibrations_b200/csrc` builds it)
importing this module raises, and every compute entry point fails with CC_ERR_NO_DEVICE
when no B200 is visible.
"""
from __future__ import annotations

import ctypes as C
import os

_HERE = os.path.dirname(os.path.abspath(__file__))
# CAMCAL_B200_LIB: load another build of the same ABI (the bounds-checked build, or another commit's for an A/B)
LIB_PATH = os.environ.get("CAMCAL_B200_LIB") or os.path.join(_HERE, "libcamcal_b200.so")

CC_OK = 0
CC_ERR_INVALID_ARG = -1
CC_ERR_NO_DEVICE = -2
CC_ERR_CUDA = -3
CC_ERR_UNSUPPORTED = -4
CC_ERR_NOMEM = -5

COORD_F64 = 0
COORD_F32 = 1
GATHER_AUTO = 0
GATHER_DIRECT = 16
GATHER_TMA = 32

PER_VIEW = 66
SHARED = 21
LM_YZ = 30
LM_SCHUR = 21
LM_DELTA = 8
COMM_ID_BYTES = 128


class CamcalError(RuntimeError):
    def __init__(self, status: int, message: str):
        super().__init__(f"libcamcal_b200 status {status}: {message}")
        self.status = status


class Intr(C.Structure):
    _fields_ = [(n, C.c_double) for n in ("frow", "fcol", "crow", "ccol", "k", "checker_size")]


class View(C.Structure):
    _fields_ = [("rvec", C.c_double * 3), ("tvec", C.c_double * 3)]


if not os.path.exists(LIB_PATH):
    raise ImportError(
        f"{LIB_PATH} not found: build it with `python -c 'import __graft_entry__ as g; g.build()'` "
        "(needs nvcc). cameracalibrations_b200 has no CPU fallback.")

lib = C.CDLL(LIB_PATH)

_vp, _sz, _i, _u, _d, _f = C.c_void_p, C.c_size_t, C.c_int, C.c_uint, C.c_double, C.c_float
_pI, _pV = C.POINTER(Intr), C.POINTER(View)
_i64p = C.POINTER(C.c_int64)
_u8p = C.POINTER(C.c_uint8)

_SIGS = {
    "cc_abi_version": (_i, []),
    "cc_last_error_string": (C.c_char_p, []),
    "cc_device_count": (_i, [C.POINTER(_i)]),
    "cc_ctx_create": (_i, [_i, C.POINTER(_vp)]),
    "cc_ctx_destroy": (_i, [_vp]),
    "cc_ctx_device": (_i, [_vp, C.POINTER(_i)]),
    "cc_ctx_synchronize": (_i, [_vp]),
    "cc_ctx_launch_count": (_i, [_vp, C.POINTER(C.c_uint64)]),
    "cc_host_alloc": (_i, [C.POINTER(_vp), _sz]),
    "cc_host_free": (_i, [_vp]),
    "cc_host_register": (_i, [_vp, _sz]),
    "cc_host_unregister": (_i, [_vp]),
    "cc_img2world_f64": (_i, [_vp, _pI, _pV, _vp, _vp, _vp, _vp, _vp, _sz, _vp]),
    "cc_img2world_f32": (_i, [_vp, _pI, _pV, _vp, _vp, _vp, _vp, _vp, _sz, _vp]),
    "cc_img2world_f64_host": (_i, [_vp, _pI, _pV, _vp, _vp, _vp, _vp, _vp, _sz]),
    "cc_img2world_f32_host": (_i, [_vp, _pI, _pV, _vp, _vp, _vp, _vp, _vp, _sz]),
    "cc_world2img_f64": (_i, [_vp, _pI, _pV, _vp, _vp, _vp, _vp, _vp, _sz, _vp]),
    "cc_world2img_f32": (_i, [_vp, _pI, _pV, _vp, _vp, _vp, _vp, _vp, _sz, _vp]),
    "cc_world2img_f64_host": (_i, [_vp, _pI, _pV, _vp, _vp, _vp, _vp, _vp, _sz]),
    "cc_world2img_f32_host": (_i, [_vp, _pI, _pV, _vp, _vp, _vp, _vp, _vp, _sz]),
    "cc_img2world_f64_views": (_i, [_vp, _pI, _vp, _i, _vp, _vp, _vp, _vp, _vp, _vp, _vp]),
    "cc_img2world_f32_views": (_i, [_vp, _pI, _vp, _i, _vp, _vp, _vp, _vp, _vp, _vp, _vp]),
    "cc_world2img_f64_views": (_i, [_vp, _pI, _vp, _i, _vp, _vp, _vp, _vp, _vp, _vp, _vp]),
    "cc_world2img_f32_views": (_i, [_vp, _pI, _vp, _i, _vp, _vp, _vp, _vp, _vp, _vp, _vp]),
    "cc_img2world_f64_views_host": (_i, [_vp, _pI, _vp, _i, _vp, _vp, _vp, _vp, _vp, _vp]),
    "cc_img2world_f32_views_host": (_i, [_vp, _pI, _vp, _i, _vp, _vp, _vp, _vp, _vp, _vp]),
    "cc_world2img_f64_views_host": (_i, [_vp, _pI, _vp, _i, _vp, _vp, _vp, _vp, _vp, _vp]),
    "cc_world2img_f32_views_host": (_i, [_vp, _pI, _vp, _i, _vp, _vp, _vp, _vp, _vp, _vp]),
    "cc_img2world_f64_aos": (_i, [_vp, _pI, _vp, _i, _vp, _vp, _vp, _i, _sz, _vp]),
    "cc_img2world_f32_aos": (_i, [_vp, _pI, _vp, _i, _vp, _vp, _vp, _i, _sz, _vp]),
    "cc_world2img_f64_aos": (_i, [_vp, _pI, _vp, _i, _vp, _vp, _i, _vp, _sz, _vp]),
    "cc_world2img_f32_aos": (_i, [_vp, _pI, _vp, _i, _vp, _vp, _i, _vp, _sz, _vp]),
    "cc_img2world_f64_aos_host": (_i, [_vp, _pI, _vp, _i, _vp, _vp, _vp, _i, _sz]),
    "cc_img2world_f32_aos_host": (_i, [_vp, _pI, _vp, _i, _vp, _vp, _vp, _i, _sz]),
    "cc_world2img_f64_aos_host": (_i, [_vp, _pI, _vp, _i, _vp, _vp, _i, _vp, _sz]),
    "cc_world2img_f32_aos_host": (_i, [_vp, _pI, _vp, _i, _vp, _vp, _i, _vp, _sz]),
    "cc_rectify_f32c1": (_i, [_vp, _pI, _pV, _d, _i64p, _vp, _vp, _i, _i, _sz, _sz, _i, _f, _u, _vp]),
    "cc_rectify_u8c3": (_i, [_vp, _pI, _pV, _d, _i64p, _vp, _vp, _i, _i, _sz, _sz, _i, _u8p, _u, _vp]),
    "cc_rectify_f32c1_host": (_i, [_vp, _pI, _pV, _d, _i64p, _vp, _vp, _i, _i, _sz, _sz, _i, _f, _u]),
    "cc_rectify_u8c3_host": (_i, [_vp, _pI, _pV, _d, _i64p, _vp, _vp, _i, _i, _sz, _sz, _i, _u8p, _u]),
    "cc_rectify_f32c1_views": (_i, [_vp, _pI, _vp, _i, _vp, _vp, _vp, _vp, _i, _i, _sz, _sz, _i, _f, _u, _vp]),
    "cc_rectify_u8c3_views": (_i, [_vp, _pI, _vp, _i, _vp, _vp, _vp, _vp, _i, _i, _sz, _sz, _i, _u8p, _u, _vp]),
    "cc_rectify_views_f32c1_host": (_i, [_vp, _pI, _vp, _i, _vp, _vp, _vp, _vp, _i, _i, _sz, _sz, _i, _f, _u]),
    "cc_rectify_views_u8c3_host": (_i, [_vp, _pI, _vp, _i, _vp, _vp, _vp, _vp, _i, _i, _sz, _sz, _i, _u8p, _u]),
    "cc_rectify_map_f64": (_i, [_vp, _pI, _pV, _d, _i64p, _vp, _vp, _i, _i, _sz, _vp]),
    "cc_rectify_map_f32": (_i, [_vp, _pI, _pV, _d, _i64p, _vp, _vp, _i, _i, _sz, _vp]),
    "cc_jpeg_info": (_i, [_vp, _sz, C.POINTER(_i), C.POINTER(_i), C.POINTER(_i)]),
    "cc_jpeg_decode_u8c3": (_i, [_vp, _vp, _vp, _i, _vp, _i, _i, _sz, _sz, _vp]),
    "cc_get_ratio": (_i, [_vp, _vp, _i, _i, _d, C.POINTER(_d)]),
    "cc_get_axes": (_i, [_d, _d, _i, _i, _i, _i, _i64p]),
    "cc_reproj_jtj_f64": (_i, [_vp, _pI, _d, _vp, _i, _vp, _vp, _i, _vp, _vp, _vp]),
    "cc_reproj_jtj_f64_host": (_i, [_vp, _pI, _d, _vp, _i, _vp, _vp, _i, _vp, _vp]),
    "cc_calculate_errors_f64": (_i, [_vp, _pI, _vp, _i, _vp, _vp, _i, _i, _vp, _vp, _i, _vp, _vp]),
    "cc_calculate_errors_f64_host": (_i, [_vp, _pI, _vp, _i, _vp, _vp, _i, _i, _vp, _vp, _i, _vp]),
    "cc_lm_schur_f64": (_i, [_vp, _vp, _i, _d, _vp, _vp, _vp]),
    "cc_lm_update_f64": (_i, [_vp, _vp, _vp, _d, _u, _vp, _vp, _i, _vp, _vp, _vp]),
    "cc_lm_fit_f64_host": (_i, [_vp, _pI, _d, _u, _vp, _i, _vp, _vp, _i, _i, _d, C.POINTER(_d), C.POINTER(_i)]),
    "cc_lm_fit_f64": (_i, [_vp, _pI, _d, _u, _vp, _i, _vp, _vp, _i, _i, _d, C.POINTER(_d), C.POINTER(_i), _vp]),
    "cc_lm_initial_guess_f64": (_i, [_vp, _vp, _vp, _i, _i, _i, _i, _d, _pI, _vp, _vp]),
    "cc_comm_unique_id": (_i, [_vp]),
    "cc_comm_init_rank": (_i, [_vp, _i, _i, _vp]),
    "cc_comm_destroy": (_i, [_vp]),
    "cc_comm_size": (_i, [_vp, C.POINTER(_i), C.POINTER(_i)]),
    "cc_comm_nccl_version": (_i, [C.POINTER(_i)]),
    "cc_allreduce_shared": (_i, [_vp, _vp, _sz, _vp]),
    "cc_ctx_create_group": (_i, [_i, C.POINTER(_i), C.POINTER(_vp)]),
    "cc_ctx_destroy_group": (_i, [_i, C.POINTER(_vp)]),
    "cc_allreduce_shared_group": (_i, [C.POINTER(_vp), _i, C.POINTER(_vp), _sz, C.POINTER(_vp)]),
    "cc_ctx_collective_count": (_i, [_vp, C.POINTER(C.c_uint64)]),
}

EXPORTS = tuple(_SIGS)

for _name, (_res, _args) in _SIGS.items():
    _fn = getattr(lib, _name)  # AttributeError here = header/library mismatch
    _fn.restype = _res
    _fn.argtypes = _args


def last_error() -> str:
    return lib.cc_last_error_string().decode("utf-8", "replace")


def check(status: int) -> None:
    if status != CC_OK:
        raise CamcalError(status, last_error())


def make_intr(frow, fcol, crow, ccol, k, checker_size) -> Intr:
    return Intr(float(frow), float(fcol), float(crow), float(ccol), float(k), float(checker_size))


def make_view(rvec, tvec) -> View:
    v = View()
    v.rvec[:] = [float(x) for x in rvec]
    v.tvec[:] = [float(x) for x in tvec]
    return v


class Context:
    """cc_ctx for one device (per-device scratch + host pipeline)."""

    def __init__(self, device: int = 0):
        h = _vp()
        check(lib.cc_ctx_create(int(device), C.byref(h)))
        self._h = h
        self.device = int(device)

    @property
    def handle(self):
        return self._h

    def synchronize(self):
        check(lib.cc_ctx_synchronize(self._h))

    def launch_count(self) -> int:
        n = C.c_uint64()
        check(lib.cc_ctx_launch_count(self._h, C.byref(n)))
        return int(n.value)

    def collective_count(self) -> int:
        n = C.c_uint64()
        check(lib.cc_ctx_collective_count(self._h, C.byref(n)))
        return int(n.value)

    # -- NCCL communicator of this context (csrc/comm.cu) ------------------------------------
    def comm_size(self):
        n, r = _i(1), _i(0)
        check(lib.cc_comm_size(self._h, C.byref(n), C.byref(r)))
        return int(n.value), int(r.value)

    def comm_init(self, nranks: int, rank: int, unique_id: bytes | None):
        """cc_comm_init_rank: `unique_id` = the 128 bytes rank 0 got from comm_unique_id()."""
        buf = C.create_string_buffer(unique_id, COMM_ID_BYTES) if unique_id is not None else None
        check(lib.cc_comm_init_rank(self._h, int(nranks), int(rank), buf))

    def comm_init_from_torch(self, group=None):
        """Bootstrap over an initialised torch.distributed group (any backend): rank 0 creates the
        NCCL unique id, the group broadcasts its 128 bytes, every rank joins.  torch only carries
        the id; the all-reduces of the hot path then run inside libcamcal_b200 on raw NCCL."""
        import torch.distributed as dist
        if self.comm_size()[0] > 1:
            return
        world, rank = dist.get_world_size(group), dist.get_rank(group)
        if world == 1:
            return
        box = [comm_unique_id() if rank == 0 else None]
        dist.broadcast_object_list(box, src=dist.get_global_rank(group, 0) if group is not None else 0, group=group)
        self.comm_init(world, rank, box[0])

    def allreduce(self, t):
        """in-place sum of a float64 CUDA tensor over the ranks (cc_allreduce_shared), torch's current stream"""
        import torch
        assert t.is_cuda and t.dtype == torch.float64 and t.is_contiguous()
        st = C.c_void_p(torch.cuda.current_stream(t.device.index).cuda_stream)
        check(lib.cc_allreduce_shared(self._h, C.c_void_p(t.data_ptr()), C.c_size_t(t.numel()), st))
        return t

    def close(self):
        if getattr(self, "_h", None):
            lib.cc_ctx_destroy(self._h)
            self._h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass


_contexts: dict[int, Context] = {}


def context(device: int = 0) -> Context:
    ctx = _contexts.get(device)
    if ctx is None:
        ctx = _contexts[device] = Context(device)
    return ctx


def comm_unique_id() -> bytes:
    buf = C.create_string_buffer(COMM_ID_BYTES)
    check(lib.cc_comm_unique_id(buf))
    return buf.raw


def device_count() -> int:
    n = _i(0)
    check(lib.cc_device_count(C.byref(n)))
    return int(n.value)
