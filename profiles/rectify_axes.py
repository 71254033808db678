"""Rectification into output axes of any size (cc_rectify_axes_*, warp(..., out_size=)): kernel time, output rate,
path and HBM fraction of the workloads a user resamples a calibrated camera with.

  64 x 1080p fp32 -> 540 x 960  (ratio / 2, the same world window), exact and fast coordinates
  64 x 1080p fp32 -> 2160 x 3840 (ratio x 2), exact and fast
  16 x 4K u8 RGB  -> 1080p, exact and fast
  64 views x 1080p fp32 -> 540 x 960 in one views call, exact and fast
  same size: cc_rectify_f32c1 against cc_rectify_axes_f32c1 on 64 x 1080p, alternated

Every working set is larger than the 126 MB L2.  Times are CUDA events around `reps` calls after warm-ups, the
median of `windows` windows.  HBM bytes = output bytes + the source bytes the taps touch (the distinct 2 x 2 tap
texels of every in-frame pixel, counted on the host from the FP64 map of the oracle), over 7.7 TB/s.  The card's
name and power limit are read in the same run.  Prints one JSON line per workload; --out also writes them all.
"""
import argparse
import json
import os
import subprocess
import sys
import tempfile

ROOT = os.path.join(os.path.dirname(os.path.abspath(__file__)), "..")
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))

import numpy as np
import torch

import cameracalibrations_b200 as cc
from conftest import BENCH_VIEW, C2_INTR, C3_INTR
from oracle import oracle_c as oc

HBM = 7.7e12


def rect_params(intr, sz, view):
    n1, n2 = 20, 14
    ch = oc.chain(intr, *view)
    a, b = np.meshgrid(np.arange(n1, dtype=np.float64), np.arange(n2, dtype=np.float64), indexing="ij")
    row, col = oc.world2img_soa(ch, (a * intr[5]).ravel(), (b * intr[5]).ravel())
    ratio = oc.get_ratio(np.stack([row, col], -1).reshape(n1, n2, 2), intr[5])
    return ratio, oc.get_axes(ratio, intr[5], (n1, n2), sz)


def views(n):
    return [((BENCH_VIEW[0][0] + 0.004 * i, BENCH_VIEW[0][1] - 0.003 * i, BENCH_VIEW[0][2] + 0.002 * i),
             (BENCH_VIEW[1][0] + 0.03 * i, BENCH_VIEW[1][1] - 0.02 * i, BENCH_VIEW[1][2] + 0.1 * i)) for i in range(n)]


def touched_texels(intr, view, ratio, axs, out_sz, sz):
    """distinct source texels the bilinear taps of one output frame read (FP64 map, the oracle's rule)"""
    mr, mc = oc.rectify_map(oc.chain(intr, *view), 1.0 / ratio, axs, out_sz)
    inb = (mr >= 1) & (mr <= sz[0]) & (mc >= 1) & (mc <= sz[1])
    i1 = np.minimum(np.floor(mr[inb]), sz[0] - 1).astype(np.int64) - 1
    i2 = np.minimum(np.floor(mc[inb]), sz[1] - 1).astype(np.int64) - 1
    lin = np.concatenate([(i2 + d2) * sz[0] + i1 + d1 for d1 in (0, 1) for d2 in (0, 1)])
    return int(np.unique(lin).size)


class Stderr:
    """C-level stderr of the block (the library's CAMCAL_DEBUG lines)"""

    def __enter__(self):
        self.f = tempfile.TemporaryFile(mode="w+")
        sys.stderr.flush()
        self.saved = os.dup(2)
        os.dup2(self.f.fileno(), 2)
        return self

    def __exit__(self, *a):
        sys.stderr.flush()
        os.dup2(self.saved, 2)
        os.close(self.saved)
        self.f.seek(0)
        self.text = self.f.read()
        self.f.close()


def path_of(fn):
    """launches and staged launches of one call"""
    ctx = cc.context(0)
    n0 = ctx.launch_count()
    os.environ["CAMCAL_DEBUG"] = "1"
    try:
        with Stderr() as e:
            fn()
            torch.cuda.synchronize()
    finally:
        os.environ.pop("CAMCAL_DEBUG", None)
    launches = ctx.launch_count() - n0
    staged = e.text.count("[camcal] staged:")
    return {"launches": launches, "staged": staged, "path": "staged" if staged == launches else
            ("direct" if staged == 0 else "mixed")}


def time_ms(fn, reps, windows, warmup=3):
    for _ in range(warmup):
        fn()
    torch.cuda.synchronize()
    ts = []
    for _ in range(windows):
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        for _ in range(reps):
            fn()
        b.record()
        torch.cuda.synchronize()
        ts.append(a.elapsed_time(b) / reps)
    return float(np.median(ts)), float(min(ts)), float(max(ts))


def card():
    name = torch.cuda.get_device_name(0)
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader", "-i", "0"],
                           capture_output=True, text=True, timeout=30).stdout.strip()
    except Exception as e:                       # the query is informative only
        q = f"unavailable: {e}"
    return {"torch_name": name, "nvidia_smi": q}


def workload(name, fn, frames_out_px, pxb, nframes, texels_per_frame, reps, windows):
    p = path_of(fn)
    med, lo, hi = time_ms(fn, reps, windows)
    out_bytes = frames_out_px * pxb
    bytes_ = out_bytes + texels_per_frame * pxb * nframes
    r = {"workload": name, "ms": med, "ms_min": lo, "ms_max": hi, "gpix_s": frames_out_px / med / 1e6,
         "hbm_bytes": bytes_, "hbm_fraction": bytes_ / (med * 1e-3) / HBM, **p}
    print(json.dumps(r), flush=True)
    return r


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=10)
    ap.add_argument("--windows", type=int, default=5)
    ap.add_argument("--out", default=None, help="also write the results to this JSON file")
    args = ap.parse_args()
    assert torch.cuda.is_available(), "needs a CUDA device"
    res = {"card": card(), "workloads": []}
    print(json.dumps(res["card"]), flush=True)
    W = res["workloads"]
    rng = np.random.default_rng(0)

    # 64 x 1080p fp32, one view
    sz = (1080, 1920)
    ratio, axs = rect_params(C2_INTR, sz, BENCH_VIEW)
    c = cc.Calibration(C2_INTR[:4], [BENCH_VIEW], 1.0 / C2_INTR[5], C2_INTR[4], ["v.png"])
    f = torch.from_numpy(rng.random((64, sz[1], sz[0]), dtype=np.float32)).cuda()
    for label, scale, out_sz in (("down2 540x960", 0.5, (540, 960)), ("up2 2160x3840", 2.0, (2160, 3840))):
        r_s, a_s = ratio * scale, (int(round(axs[0] * scale)), int(round(axs[1] * scale)))
        tex = touched_texels(C2_INTR, BENCH_VIEW, r_s, a_s, out_sz, sz)
        out = torch.empty((64, out_sz[1], out_sz[0]), dtype=torch.float32, device="cuda")
        for coord in ("f64", "f32"):
            fn = lambda: cc.warp(c, 0, f, r_s, a_s, coord=coord, out=out, out_size=out_sz)
            W.append(workload(f"64x1080p fp32 -> {label}, {coord}", fn, 64 * out_sz[0] * out_sz[1], 4, 64, tex,
                              args.reps, args.windows))
        del out

    # same size: old symbol against new, alternated
    tex = touched_texels(C2_INTR, BENCH_VIEW, ratio, axs, sz, sz)
    out = torch.empty_like(f)
    for rnd in range(3):
        for coord in ("f64", "f32"):
            W.append(workload(f"same size A/B round {rnd}: cc_rectify_f32c1, {coord}",
                              lambda: cc.warp(c, 0, f, ratio, axs, coord=coord, out=out),
                              64 * sz[0] * sz[1], 4, 64, tex, args.reps, args.windows))
            W.append(workload(f"same size A/B round {rnd}: cc_rectify_axes_f32c1, {coord}",
                              lambda: cc.warp(c, 0, f, ratio, axs, coord=coord, out=out, out_size=sz),
                              64 * sz[0] * sz[1], 4, 64, tex, args.reps, args.windows))
    del out

    # 64 views x 1080p -> 540 x 960, one views call
    vs = views(64)
    cv = cc.Calibration(C2_INTR[:4], vs, 1.0 / C2_INTR[5], C2_INTR[4], [f"{i}.png" for i in range(64)])
    rs, as_ = [], []
    tex = 0
    for v in vs:
        r, a = rect_params(C2_INTR, sz, v)
        rs.append(r / 2)
        as_.append((int(round(a[0] / 2)), int(round(a[1] / 2))))
        tex += touched_texels(C2_INTR, v, rs[-1], as_[-1], (540, 960), sz)
    out = torch.empty((64, 960, 540), dtype=torch.float32, device="cuda")
    for coord in ("f64", "f32"):
        fn = lambda: cc.warp_views(cv, list(range(64)), f, rs, as_, coord=coord, out=out, out_size=(540, 960))
        W.append(workload(f"64 views x 1080p fp32 -> 540x960, one call, {coord}", fn, 64 * 540 * 960, 4, 1, tex,
                          args.reps, args.windows))
    del out, f

    # 16 x 4K u8 RGB -> 1080p
    sz4 = (2160, 3840)
    ratio4, axs4 = rect_params(C3_INTR, sz4, BENCH_VIEW)
    c4 = cc.Calibration(C3_INTR[:4], [BENCH_VIEW], 1.0 / C3_INTR[5], C3_INTR[4], ["v.png"])
    f8 = torch.from_numpy(rng.integers(0, 256, (16, sz4[1], sz4[0], 3), dtype=np.uint8)).cuda()
    r_s, a_s = ratio4 / 2, (int(round(axs4[0] / 2)), int(round(axs4[1] / 2)))
    tex = touched_texels(C3_INTR, BENCH_VIEW, r_s, a_s, sz, sz4)
    out = torch.empty((16, sz[1], sz[0], 3), dtype=torch.uint8, device="cuda")
    for coord in ("f64", "f32"):
        fn = lambda: cc.warp(c4, 0, f8, r_s, a_s, coord=coord, out=out, out_size=sz)
        W.append(workload(f"16x4K u8 RGB -> 1080p, {coord}", fn, 16 * sz[0] * sz[1], 3, 16, tex, args.reps, args.windows))

    if args.out:
        with open(args.out, "w") as fh:
            json.dump(res, fh, indent=1)


if __name__ == "__main__":
    main()
