"""Point maps on interleaved points: the cc_*_aos kernels against the SoA kernels, and what the interleaved entry
points save the Python layer.

  python profiles/point_aos.py [--reps 10] [--out DIR]

Prints the card and its power limit, then one JSON line per measurement (and writes them to DIR/point_aos.json
when --out is given).  100 M points throughout (inputs and outputs 1.6-4 GB: far larger than L2).
  kernel_*  kernel time (torch.profiler) of every map at both output / input dims: pixel->world with out_dim 3
            (c(::RowCol, i)) and 2 (rectification), world->pixel with in_dim 3 and 2 (z = 0).  SoA and AoS over one
            view (the SINGLE kernel) and over 64 and 10 000 equal segments with different views (TABLE).  The
            algorithmic bytes are the same in both layouts.
  python_*  Calibration.__call__ on CUDA tensors, events around back-to-back calls: the AoS call against the path it
            replaces (one .contiguous() copy per input coordinate, the SoA entry point, torch.stack), rebuilt here.
  host_*    the same on numpy arrays (the *_host entry points), against the host link rate measured in the same run
            (pinned torch copies, each way).
"""
import argparse
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
from conftest import C3_INTR, SYN_VIEW

N = 100_000_000


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


def kernel_ms(fn, reps):
    """mean kernel time per call of the point-map kernels"""
    from torch.profiler import ProfilerActivity, profile
    fn()
    torch.cuda.synchronize()
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        for _ in range(reps):
            fn()
        torch.cuda.synchronize()
    t = 0.0
    for e in prof.events():
        if e.device_type == torch.autograd.DeviceType.CUDA and ("img2world" in e.name or "world2img" in e.name):
            t += e.device_time_total if hasattr(e, "device_time_total") else e.cuda_time_total
    return t / reps / 1e3


def emit(out, rec):
    print(json.dumps(rec), flush=True)
    out.append(rec)


def kernels(c, out, reps):
    rng = np.random.default_rng(0)
    segs = {}
    for nseg in (64, 10_000):
        segs[nseg] = (rng.integers(0, 64, nseg).tolist(), [N // nseg + (1 if s < N % nseg else 0) for s in range(nseg)])
    for dt, name in ((torch.float64, "f64"), (torch.float32, "f32")):
        esz = 8 if dt == torch.float64 else 4
        g = torch.Generator(device="cuda").manual_seed(99)
        rc = torch.stack([torch.rand(N, dtype=dt, device="cuda", generator=g) * 2160,
                          torch.rand(N, dtype=dt, device="cuda", generator=g) * 3840], -1)
        xyz = c(rc, 0)
        row, col = rc[:, 0].contiguous(), rc[:, 1].contiguous()
        x, y, z = (xyz[:, d].contiguous() for d in range(3))
        for kind, dim in (("img2world", 3), ("img2world", 2), ("world2img", 3), ("world2img", 2)):
            if kind == "img2world":
                soa1 = lambda: c.img2world(row, col, 0, want_z=dim == 3)
                soav = lambda vs, cs: c.img2world_views(row, col, vs, cs, want_z=dim == 3)
                pts, aos_nv = rc, lambda vs, cs: cc.calibration._aos_call(kind, c, c._segments(vs, cs), rc, dim)
                aos1 = (lambda: cc.calibration._aos_call(kind, c, 0, rc, 3)) if dim == 3 else \
                       (lambda: cc.rectification(c, 0)(rc))
                nbytes = (2 + dim) * esz
            else:
                zz = z if dim == 3 else None
                pts = xyz if dim == 3 else xyz[:, :2].contiguous()
                soa1 = lambda: c.world2img(x, y, zz, 0)
                soav = lambda vs, cs: c.world2img_views(x, y, zz, vs, cs)
                aos1 = lambda: cc.calibration._aos_call(kind, c, 0, pts, 2)
                aos_nv = lambda vs, cs: cc.calibration._aos_call(kind, c, c._segments(vs, cs), pts, 2)
                nbytes = (dim + 2) * esz
            rows = [("1", kernel_ms(soa1, reps), kernel_ms(aos1, reps))]
            for nseg, (vs, cs) in segs.items():
                rows.append((str(nseg), kernel_ms(lambda: soav(vs, cs), reps), kernel_ms(lambda: aos_nv(vs, cs), reps)))
            for nseg, ks, ka in rows:
                emit(out, dict(case=f"kernel_{kind}_{name}_dim{dim}_100M_{nseg}seg", soa_kernel_ms=ks,
                               aos_kernel_ms=ka, soa_gpt_s=N / ks / 1e6, aos_gpt_s=N / ka / 1e6,
                               aos_tb_s=N * nbytes / ka / 1e9, aos_over_soa=ks / ka))
            del pts
        del rc, xyz, row, col, x, y, z
        torch.cuda.empty_cache()


def python_calls(c, out, reps):
    """c(pts, i) on CUDA tensors: the AoS call against the former column copies + SoA call + stack"""
    for dt, name in ((torch.float64, "f64"), (torch.float32, "f32")):
        g = torch.Generator(device="cuda").manual_seed(7)
        rc = torch.stack([torch.rand(N, dtype=dt, device="cuda", generator=g) * 2160,
                          torch.rand(N, dtype=dt, device="cuda", generator=g) * 3840], -1)
        xyz = c(rc, 0)
        before = {"img2world": lambda: torch.stack(c.img2world(rc[..., 0].contiguous(), rc[..., 1].contiguous(), 0), -1),
                  "world2img": lambda: torch.stack(c.world2img(*(xyz[..., d].contiguous() for d in range(3)), 0), -1)}
        after = {"img2world": lambda: c(rc, 0), "world2img": lambda: c(xyz, 0)}
        for kind in ("img2world", "world2img"):
            assert torch.equal(before[kind](), after[kind]())
            mb, ma = events_ms(before[kind], reps), events_ms(after[kind], reps)
            emit(out, dict(case=f"python_{kind}_{name}_cuda_100M", before_ms=mb, after_ms=ma, speedup=mb / ma,
                           after_gpt_s=N / ma / 1e6))
        del rc, xyz
        torch.cuda.empty_cache()


def link_gb_s():
    """pinned host <-> device copy rate, each way, 1 GB"""
    h = torch.empty(1 << 30, dtype=torch.uint8).pin_memory()
    d = torch.empty(1 << 30, dtype=torch.uint8, device="cuda")
    h2d = events_ms(lambda: d.copy_(h, non_blocking=True), 5)
    d2h = events_ms(lambda: h.copy_(d, non_blocking=True), 5)
    return (1 << 30) / h2d / 1e6, (1 << 30) / d2h / 1e6


def host_calls(c, out, reps):
    """numpy points through the *_host entry points: AoS against the former split + SoA host call + np.stack"""
    h2d, d2h = link_gb_s()
    emit(out, dict(case="host_link_pinned", h2d_gb_s=h2d, d2h_gb_s=d2h))
    rng = np.random.default_rng(3)
    for dt, name in ((np.float64, "f64"), (np.float32, "f32")):
        rc = np.stack([rng.uniform(1, 2160, N), rng.uniform(1, 3840, N)], -1).astype(dt)
        xyz = c(rc, 0)
        esz = np.dtype(dt).itemsize
        before = {"img2world": lambda: np.stack(c.img2world(np.ascontiguousarray(rc[:, 0]),
                                                             np.ascontiguousarray(rc[:, 1]), 0), -1),
                  "world2img": lambda: np.stack(c.world2img(*(np.ascontiguousarray(xyz[:, d]) for d in range(3)), 0), -1)}
        after = {"img2world": lambda: c(rc, 0), "world2img": lambda: c(xyz, 0)}
        for kind in ("img2world", "world2img"):
            assert np.array_equal(before[kind](), after[kind]())
            res = {}
            for label, fn in (("before", before[kind]), ("after", after[kind])):
                fn()
                t = time.perf_counter()
                for _ in range(reps):
                    fn()
                res[label] = (time.perf_counter() - t) / reps * 1e3
            inb, outb = (2 * esz, 3 * esz) if kind == "img2world" else (3 * esz, 2 * esz)
            # the link moves inb one way and outb the other; at the measured rates that takes at least:
            link_ms = max(N * inb / h2d, N * outb / d2h) / 1e6
            emit(out, dict(case=f"host_{kind}_{name}_numpy_100M", before_ms=res["before"], after_ms=res["after"],
                           speedup=res["before"] / res["after"], link_bound_ms=link_ms,
                           after_over_link=link_ms / res["after"]))
        del rc, xyz


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=10)
    ap.add_argument("--out")
    args = ap.parse_args()
    assert torch.cuda.is_available(), "point_aos.py measures on a CUDA device"
    name, pl = card()
    print(f"card: {name}, power limit {pl}", flush=True)
    out = [dict(card=name, power_limit=pl)]
    c = cc.Calibration(C3_INTR[:4], poses(64, 3), 1.0 / C3_INTR[5], C3_INTR[4], [f"{i}.png" for i in range(64)])
    kernels(c, out, args.reps)
    python_calls(c, out, args.reps)
    host_calls(c, out, max(2, args.reps // 4))
    if args.out:
        os.makedirs(args.out, exist_ok=True)
        with open(os.path.join(args.out, "point_aos.json"), "w") as f:
            json.dump(out, f, indent=1)


if __name__ == "__main__":
    main()
