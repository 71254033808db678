"""Where the time of cc_rectify_f32c1_views goes: 64 x 1080p frames, 64 different views, one call.
Per coordinate type: host enqueue time (wall clock of the call, no synchronisation) against the device
time (CUDA events)."""
import os, sys, time
sys.path.insert(0, os.path.join(os.path.dirname(os.path.abspath(__file__)), ".."))
import numpy as np
import torch
import bench
import cameracalibrations_b200 as cc

wl = bench.WORKLOADS["c2"]
sz = wl["sz"]
BV = bench.BENCH_VIEW
vlist = [((BV[0][0] + 0.002 * i, BV[0][1], BV[0][2] + 0.001 * i),
          (BV[1][0] + 0.01 * i, BV[1][1], BV[1][2] + 0.05 * i)) for i in range(64)]
calv = cc.Calibration(wl["intr"][:4], vlist, 1.0, wl["intr"][4], [f"{i}.png" for i in range(64)])
ratio = cc.get_ratio(bench.geometry(wl), 1.0)
axs = cc.get_axes(ratio, 1.0, bench.N_CORNERS, sz)
src = torch.rand((64, sz[1], sz[0]), dtype=torch.float32, device="cuda")
dst = torch.empty_like(src)
peak = bench.measured_peak()[0]
npx = 64 * sz[0] * sz[1]


def run(coord, nviews=64, reps=20):
    idx = list(range(nviews))
    f = lambda: cc.warp_views(calv, idx, src[:nviews], [ratio] * nviews, [axs] * nviews, coord=coord, out=dst[:nviews])
    for _ in range(3):
        f()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    host = 0.0
    e0.record()
    for _ in range(reps):
        t0 = time.perf_counter()
        f()
        host += time.perf_counter() - t0
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) / reps, host / reps * 1e3


# cold call: 64 views nobody has planned yet (host footprints + upload + launch), wall clock
vcold = [((BV[0][0] - 0.003 * i, BV[0][1] + 0.001 * i, BV[0][2]), (BV[1][0] - 0.02 * i, BV[1][1], BV[1][2] + 0.03 * i)) for i in range(1, 65)]
calc = cc.Calibration(wl["intr"][:4], vcold, 1.0, wl["intr"][4], [f"c{i}.png" for i in range(64)])
torch.cuda.synchronize()
t0 = time.perf_counter()
cc.warp_views(calc, list(range(64)), src, [ratio] * 64, [axs] * 64, coord="f32", out=dst)
torch.cuda.synchronize()
print(f"cold call, 64 new views x 1080p: {(time.perf_counter() - t0) * 1e3:.2f} ms", flush=True)
SHORT = len(sys.argv) > 1 and sys.argv[1] == "short"
for coord in ("f32", "f64"):
    ms, host_ms = run(coord)
    print(f"views 64x1080p {coord}: device {ms:.4f} ms  host enqueue {host_ms:.4f} ms  "
          f"frac {8 * npx / (ms * 1e-3) / 1e9 / peak:.3f}", flush=True)
if SHORT:
    sys.exit(0)
# the same 64 frames with ONE view (map shared by the frames of a unit) and as 64 single-frame calls of one view
cal1 = cc.Calibration(wl["intr"][:4], [BV], 1.0, wl["intr"][4], ["extrinsic.png"])
for coord in ("f32", "f64"):
    f = lambda: [cc.warp(cal1, 0, src[i:i + 1], ratio, axs, coord=coord, out=dst[i:i + 1]) for i in range(64)]
    for _ in range(3):
        f()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    t0 = time.perf_counter()
    for _ in range(10):
        f()
    host_ms = (time.perf_counter() - t0) / 10 * 1e3
    e1.record()
    torch.cuda.synchronize()
    ms = e0.elapsed_time(e1) / 10
    print(f"64 single-frame calls, one view, one stream {coord}: device {ms:.4f} ms  host enqueue {host_ms:.4f} ms", flush=True)
