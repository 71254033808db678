"""Wall time of rectifying many views' frames from pinned host memory (the reference's plot loop from a host
program such as the Julia shim): 256 views x 1 frame, 1080p f32, 1080p and 4K u8c3, exact and fast coordinates.

  views_host warm   cc_rectify_views_*_host, second call with the same views (group plans cached)
  views_host cold   the same with views never seen before (every group plan built during the call)
  plan              host planning of those views alone: cold minus warm of the device call cc_rectify_*_views
  per_view_loop     one cc_rectify_*_host call per view (what the Julia shim did before the many-view call)
  one_view          cc_rectify_*_host over the same frames with ONE view: the pipeline's link-bound ceiling
  link              pinned host<->device copy rate in the same run, both directions at once (profiles/pcie_bw.py)

Usage: python profiles/rectify_views_host.py [--views 256] [--reps 3] [--out results/rectify_views_host.json]
"""
import argparse
import ctypes as C
import json
import os
import subprocess
import sys
import time

import numpy as np

sys.path.insert(0, os.path.join(os.path.dirname(os.path.abspath(__file__)), ".."))
sys.path.insert(0, os.path.join(os.path.dirname(os.path.abspath(__file__)), "..", "tests"))
import torch  # noqa: E402

import cameracalibrations_b200 as cc  # noqa: E402
from cameracalibrations_b200 import _lib  # noqa: E402
from conftest import BENCH_VIEW, camera_for  # noqa: E402
from oracle import oracle_c as oc  # noqa: E402


def views_for(n, salt):
    """n distinct near-frontal views; salt makes a family no earlier call has planned"""
    return [((BENCH_VIEW[0][0] + 0.0004 * i + 1e-7 * salt, BENCH_VIEW[0][1] - 0.0003 * i, BENCH_VIEW[0][2]),
             (BENCH_VIEW[1][0] + 0.003 * i, BENCH_VIEW[1][1] - 0.002 * i, BENCH_VIEW[1][2] + 0.01 * i))
            for i in range(n)]


def ratio_axes(intr, sz, view):
    n1, n2 = 20, 14
    ch = oc.chain(intr, *view)
    a, b = np.meshgrid(np.arange(n1, dtype=np.float64), np.arange(n2, dtype=np.float64), indexing="ij")
    row, col = oc.world2img_soa(ch, (a * intr[5]).ravel(), (b * intr[5]).ravel())
    ip = np.stack([row, col], axis=-1).reshape(n1, n2, 2)
    ratio = oc.get_ratio(ip, intr[5])
    return ratio, oc.get_axes(ratio, intr[5], (n1, n2), sz)


class Setup:
    def __init__(self, intr, sz, views):
        self.c = cc.Calibration(intr[:4], views, 1.0 / intr[5], intr[4], [f"{i}.png" for i in range(len(views))])
        ra = [ratio_axes(intr, sz, v) for v in views]
        self.nv = len(views)
        self.ratios = (C.c_double * self.nv)(*[r for r, _ in ra])
        self.axs = (C.c_int64 * (2 * self.nv))(*[x for _, am in ra for x in am])
        self.vw = (_lib.View * self.nv)(*[self.c._views[i] for i in range(self.nv)])


def timed(fn):
    torch.cuda.synchronize()
    t = time.perf_counter()
    fn()
    torch.cuda.synchronize()
    return time.perf_counter() - t


def link_rate(nbytes=1 << 30, reps=3):
    h1 = torch.empty(nbytes, dtype=torch.uint8).pin_memory()
    h2 = torch.empty(nbytes, dtype=torch.uint8).pin_memory()
    d1 = torch.empty(nbytes, dtype=torch.uint8, device="cuda")
    d2 = torch.empty(nbytes, dtype=torch.uint8, device="cuda")
    s1, s2 = torch.cuda.Stream(), torch.cuda.Stream()

    def both():
        for _ in range(reps):
            with torch.cuda.stream(s1):
                d1.copy_(h1, non_blocking=True)
            with torch.cuda.stream(s2):
                h2.copy_(d2, non_blocking=True)
    both()
    dt = timed(both)
    return nbytes * reps / dt / 1e9               # GB/s each direction


def run_case(fmt, sz, coord, nviews, reps, gbps, salt):
    ctx = cc.context(0).handle
    intr = camera_for(sz)
    pxb = 4 if fmt == "f32" else 3
    shape = (nviews, sz[1], sz[0]) + (() if fmt == "f32" else (3,))
    dt = torch.float32 if fmt == "f32" else torch.uint8
    src = torch.empty(shape, dtype=dt).pin_memory()
    dst = torch.empty(shape, dtype=dt).pin_memory()
    # a frame's content does not change the work: one random frame, repeated
    src[:] = (torch.rand(shape[1:]) if fmt == "f32" else torch.randint(0, 256, shape[1:], dtype=dt))
    fill = C.c_float(0.0) if fmt == "f32" else (C.c_uint8 * 3)(0, 0, 0)
    flags = _lib.COORD_F32 if coord == "f32" else _lib.COORD_F64
    ps, pd = C.c_void_p(src.data_ptr()), C.c_void_p(dst.data_ptr())
    geom = (sz[0], sz[1], C.c_size_t(sz[0]), C.c_size_t(sz[0] * sz[1]))
    many = _lib.lib.cc_rectify_views_f32c1_host if fmt == "f32" else _lib.lib.cc_rectify_views_u8c3_host
    one = _lib.lib.cc_rectify_f32c1_host if fmt == "f32" else _lib.lib.cc_rectify_u8c3_host
    dev_views = _lib.lib.cc_rectify_f32c1_views if fmt == "f32" else _lib.lib.cc_rectify_u8c3_views
    frame_b = sz[0] * sz[1] * pxb

    def call_many(s):
        _lib.check(many(ctx, C.byref(s.c._intr), s.vw, s.nv, s.ratios, s.axs, ps, pd, *geom, 1, fill, flags))

    # warm: the same views again
    s = Setup(intr, sz, views_for(nviews, salt))
    call_many(s)
    warm = min(timed(lambda: call_many(s)) for _ in range(reps))
    # cold: a new family of views per repetition
    cold = []
    for r in range(reps):
        s2 = Setup(intr, sz, views_for(nviews, salt + 1 + r))
        cold.append(timed(lambda: call_many(s2)))
    # host planning alone: the device call on device-resident frames, cold minus warm
    dsrc, ddst = src.cuda(), torch.empty(shape, dtype=dt, device="cuda")
    plan = []
    for r in range(reps):
        s3 = Setup(intr, sz, views_for(nviews, salt + 100 + r))
        call = lambda: _lib.check(dev_views(ctx, C.byref(s3.c._intr), s3.vw, s3.nv, s3.ratios, s3.axs,  # noqa: E731
                                            C.c_void_p(dsrc.data_ptr()), C.c_void_p(ddst.data_ptr()), *geom, 1, fill,
                                            flags, None))
        t_cold = timed(call)
        t_warm = min(timed(call) for _ in range(2))
        plan.append(t_cold - t_warm)
    del dsrc, ddst
    # today's per-view loop (the Julia shim before): warm after one pass
    def loop():
        for v in range(nviews):
            off = v * frame_b
            _lib.check(one(ctx, C.byref(s.c._intr), C.byref(s.c._views[v]), s.ratios[v],
                           (C.c_int64 * 2)(s.axs[2 * v], s.axs[2 * v + 1]), C.c_void_p(src.data_ptr() + off),
                           C.c_void_p(dst.data_ptr() + off), *geom, 1, fill, flags))
    loop()
    per_view = min(timed(loop) for _ in range(reps))
    # ONE view over all the frames: the link-bound ceiling of the pipeline
    def single():
        _lib.check(one(ctx, C.byref(s.c._intr), C.byref(s.c._views[0]), s.ratios[0], (C.c_int64 * 2)(s.axs[0], s.axs[1]),
                       ps, pd, *geom, nviews, fill, flags))
    single()
    one_view = min(timed(single) for _ in range(reps))
    gpix = nviews * sz[0] * sz[1] / 1e9
    transfer = nviews * frame_b / (gbps * 1e9)
    plan_t = float(np.median(plan))
    cold_t = float(np.median(cold))
    return {
        "fmt": fmt, "sz": list(sz), "coord": coord, "views": nviews,
        "warm_ms": warm * 1e3, "warm_gpix_s": gpix / warm,
        "cold_ms": cold_t * 1e3, "cold_gpix_s": gpix / cold_t,
        "plan_ms": plan_t * 1e3, "transfer_ms": transfer * 1e3,
        "cold_over_max_plan_transfer": cold_t / max(plan_t, transfer),
        "per_view_loop_ms": per_view * 1e3, "per_view_loop_gpix_s": gpix / per_view,
        "one_view_ms": one_view * 1e3, "one_view_gpix_s": gpix / one_view,
        "warm_over_one_view": one_view / warm, "warm_speedup_over_loop": per_view / warm,
    }


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--views", type=int, default=256)
    ap.add_argument("--reps", type=int, default=3)
    ap.add_argument("--out", default="")
    a = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("needs a CUDA device")
    smi = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"],
                         capture_output=True, text=True).stdout.strip()
    gbps = link_rate()
    res = {"gpu": smi, "link_gb_s_each_direction": gbps, "cases": []}
    print(f"# {smi}; host link {gbps:.1f} GB/s each direction, both at once")
    salt = int(time.time()) % 100000
    for fmt, sz in (("f32", (1080, 1920)), ("u8", (1080, 1920)), ("u8", (2160, 3840))):
        for coord in ("f64", "f32"):
            r = run_case(fmt, sz, coord, a.views, a.reps, gbps, salt)
            salt += 1000
            res["cases"].append(r)
            print(f"{fmt} {sz[0]}x{sz[1]} {coord}: warm {r['warm_ms']:.1f} ms ({r['warm_gpix_s']:.2f} Gpix/s) "
                  f"cold {r['cold_ms']:.1f} ms (plan {r['plan_ms']:.1f}, transfer {r['transfer_ms']:.1f}, "
                  f"x{r['cold_over_max_plan_transfer']:.2f} of the max) | per-view loop {r['per_view_loop_ms']:.1f} ms "
                  f"({r['warm_speedup_over_loop']:.2f}x) | one view {r['one_view_ms']:.1f} ms "
                  f"(warm = {r['warm_over_one_view']:.2f}x of it)", flush=True)
    if a.out:
        os.makedirs(os.path.dirname(a.out) or ".", exist_ok=True)
        with open(a.out, "w") as f:
            json.dump(res, f, indent=1)


if __name__ == "__main__":
    main()
