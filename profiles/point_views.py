"""Point maps over many views: the one-launch cc_*_views kernels against the single-view kernel, and the per-call
cost of mapping the C5 shape (10 000 views x 280 corners) view by view.

  python profiles/point_views.py [--reps 20] [--out DIR]

Prints the card and its power limit, then one JSON line per measurement (and writes them to DIR/point_views.json
when --out is given).
  c4_*   100 M points (inputs and outputs 2-4 GB: far larger than L2), split into 1, 64 and 10 000 equal segments
         with different views.  CUDA events over `reps` back-to-back calls give the rate of each call, table upload
         included; a torch.profiler pass over the same calls splits it into kernel time and the table's
         host-to-device copy.  The single-view kernel runs on the same points in the same process.
  c5_*   10 000 x 280 FP64 points (22-45 MB: L2-resident after the first pass).  Wall time of one _views call
         against a loop of 10 000 single-view calls through the C ABI with prebuilt arguments, device form (torch
         tensors, one stream synchronisation at the end) and host form (numpy arrays, the *_host entry points).
"""
import argparse
import ctypes as C
import json
import os
import subprocess
import sys
import time

ROOT = os.path.join(os.path.dirname(os.path.abspath(__file__)), "..")
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))
import numpy as np
import torch

import cameracalibrations_b200 as cc
from cameracalibrations_b200 import _lib
from conftest import C3_INTR, SYN_VIEW


def card():
    name = torch.cuda.get_device_name(0)
    try:
        pl = subprocess.run(["nvidia-smi", "--query-gpu=power.limit", "--format=csv,noheader", "-i", "0"],
                            capture_output=True, text=True, timeout=30).stdout.strip()
    except Exception as e:          # the number is still reported, without its power limit
        pl = f"unknown ({e})"
    return name, pl


def poses(n, seed):
    rng = np.random.default_rng(seed)
    r0, t0 = np.asarray(SYN_VIEW[0]), np.asarray(SYN_VIEW[1])
    return [(tuple(r0 + rng.uniform(-0.15, 0.15, 3)), tuple(t0 + rng.uniform(-3, 3, 3))) for _ in range(n)]


def events_ms(fn, reps):
    fn()
    torch.cuda.synchronize()
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record()
    for _ in range(reps):
        fn()
    b.record()
    torch.cuda.synchronize()
    return a.elapsed_time(b) / reps


def profiled_split(fn, reps):
    """mean per call: kernel time by kernel name, and host-to-device copy time (the table upload)"""
    from torch.profiler import ProfilerActivity, profile
    fn()
    torch.cuda.synchronize()
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        for _ in range(reps):
            fn()
        torch.cuda.synchronize()
    kern, h2d = 0.0, 0.0
    for e in prof.events():
        if e.device_type != torch.autograd.DeviceType.CUDA:
            continue
        name = e.name
        dur = e.device_time_total if hasattr(e, "device_time_total") else e.cuda_time_total
        if "kernel" in name and ("img2world" in name or "world2img" in name):
            kern += dur
        elif "HtoD" in name or "Memcpy HtoD" in name:
            h2d += dur
    return kern / reps / 1e3, h2d / reps / 1e3


def c4(out, reps):
    n = 100_000_000
    c = cc.Calibration(C3_INTR[:4], poses(64, 3), 1.0 / C3_INTR[5], C3_INTR[4], [f"{i}.png" for i in range(64)])
    rng = np.random.default_rng(0)
    for dt, name in ((torch.float64, "f64"), (torch.float32, "f32")):
        g = torch.Generator(device="cuda").manual_seed(99)
        row = torch.rand(n, dtype=dt, device="cuda", generator=g) * 2160
        col = torch.rand(n, dtype=dt, device="cuda", generator=g) * 3840
        x, y, z = c.img2world(row, col, 0)
        calls = {"img2world": (lambda vs, cs: c.img2world_views(row, col, vs, cs), lambda: c.img2world(row, col, 0)),
                 "world2img": (lambda vs, cs: c.world2img_views(x, y, z, vs, cs), lambda: c.world2img(x, y, z, 0))}
        for kind, (views_call, single_call) in calls.items():
            ms1 = events_ms(single_call, reps)
            k1, _ = profiled_split(single_call, 5)
            for nseg in (1, 64, 10_000):
                vs = rng.integers(0, 64, nseg).tolist()
                cs = [n // nseg + (1 if s < n % nseg else 0) for s in range(nseg)]
                f = lambda: views_call(vs, cs)
                ms = events_ms(f, reps)
                kv, up = profiled_split(f, 5)
                rec = dict(case=f"c4_{kind}_{name}_100M_{nseg}seg", single_gpt_s=n / ms1 / 1e6, single_kernel_ms=k1,
                           views_gpt_s=n / ms / 1e6, views_call_ms=ms, views_kernel_ms=kv, table_upload_ms=up,
                           views_kernel_gpt_s=n / kv / 1e6 if kv else None,
                           kernel_ratio=(k1 / kv) if kv else None, call_ratio=ms1 / ms)
                print(json.dumps(rec), flush=True)
                out.append(rec)
        del row, col, x, y, z
        torch.cuda.empty_cache()


def c5(out, reps):
    nv, nc = 10_000, 280
    n = nv * nc
    c = cc.Calibration(C3_INTR[:4], poses(nv, 5), 1.0 / C3_INTR[5], C3_INTR[4], [f"{i}.png" for i in range(nv)])
    rng = np.random.default_rng(1)
    row_h, col_h = rng.uniform(1, 2160, n), rng.uniform(1, 3840, n)
    x_h, y_h, z_h = (np.empty(n) for _ in range(3))
    row, col = torch.from_numpy(row_h).cuda(), torch.from_numpy(col_h).cuda()
    x, y, z = (torch.empty(n, dtype=torch.float64, device="cuda") for _ in range(3))
    h = _lib.context(0).handle
    ci = C.byref(c._intr)
    views = (_lib.View * nv)(*c._views)
    offs = (C.c_size_t * (nv + 1))(*range(0, n + 1, nc))
    st = C.c_void_p(torch.cuda.current_stream().cuda_stream)
    P = lambda t, i: C.c_void_p(t.data_ptr() + 8 * i)
    Q = lambda a, i: C.c_void_p(a.ctypes.data + 8 * i)
    single_dev = [(h, ci, C.byref(c._views[v]), P(row, v * nc), P(col, v * nc), P(x, v * nc), P(y, v * nc),
                   P(z, v * nc), C.c_size_t(nc), st) for v in range(nv)]
    single_host = [(h, ci, C.byref(c._views[v]), Q(row_h, v * nc), Q(col_h, v * nc), Q(x_h, v * nc),
                    Q(y_h, v * nc), Q(z_h, v * nc), C.c_size_t(nc)) for v in range(nv)]
    views_dev = (h, ci, views, nv, offs, P(row, 0), P(col, 0), P(x, 0), P(y, 0), P(z, 0), st)
    views_host = (h, ci, views, nv, offs, Q(row_h, 0), Q(col_h, 0), Q(x_h, 0), Q(y_h, 0), Q(z_h, 0))
    L = _lib.lib

    def wall(fn, r):
        fn()
        torch.cuda.synchronize()
        t = time.perf_counter()
        for _ in range(r):
            fn()
        torch.cuda.synchronize()
        return (time.perf_counter() - t) / r * 1e3

    def loop(f, args):
        def run():
            for a in args:
                f(*a)
        return run

    recs = [
        ("device_one_views_call", wall(lambda: L.cc_img2world_f64_views(*views_dev), reps)),
        ("device_10000_single_calls", wall(loop(L.cc_img2world_f64, single_dev), 3)),
        ("host_one_views_call", wall(lambda: L.cc_img2world_f64_views_host(*views_host), reps)),
        ("host_10000_single_calls", wall(loop(L.cc_img2world_f64_host, single_host), 3)),
    ]
    # the same results either way
    L.cc_img2world_f64_views_host(*views_host)
    xv = x_h.copy()
    loop(L.cc_img2world_f64_host, single_host)()
    assert np.array_equal(xv, x_h)
    for name, ms in recs:
        rec = dict(case=f"c5_img2world_f64_10000x280_{name}", ms=ms, points=n, note="L2-resident")
        print(json.dumps(rec), flush=True)
        out.append(rec)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=20)
    ap.add_argument("--out")
    args = ap.parse_args()
    assert torch.cuda.is_available(), "point_views.py measures on a CUDA device"
    name, pl = card()
    print(f"card: {name}, power limit {pl}", flush=True)
    out = [dict(card=name, power_limit=pl)]
    c4(out, args.reps)
    c5(out, args.reps)
    if args.out:
        os.makedirs(args.out, exist_ok=True)
        with open(os.path.join(args.out, "point_views.json"), "w") as f:
            json.dump(out, f, indent=1)


if __name__ == "__main__":
    main()
