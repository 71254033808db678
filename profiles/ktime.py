"""Device-resident kernel timing of the rectification workloads (tuning loop; bench.py is the
judged measurement).   python profiles/ktime.py [c2|c3] [f64|f32] [auto|tma|direct] [steps]
Honors CAMCAL_B200_LIB (another build of the library, e.g. the parent commit's for an A/B)."""
import os, sys
sys.path.insert(0, os.path.join(os.path.dirname(os.path.abspath(__file__)), ".."))
import torch
import bench
import cameracalibrations_b200 as cc

def run(wname, coord, gather="auto", steps=30):
    wl = bench.WORKLOADS[wname]
    sz = wl["sz"]
    ip = bench.geometry(wl)
    ratio = cc.get_ratio(ip, wl["intr"][5])
    axs = cc.get_axes(ratio, wl["intr"][5], bench.N_CORNERS, sz)
    c = cc.Calibration(wl["intr"][:4], [bench.BENCH_VIEW], 1.0 / wl["intr"][5], wl["intr"][4], ["extrinsic.png"])
    g = torch.Generator(device="cuda").manual_seed(wl["seed"])
    if wl["u8"]:
        fr = torch.randint(0, 256, (wl["frames"], sz[1], sz[0], 3), device="cuda", dtype=torch.uint8, generator=g)
    else:
        fr = torch.rand((wl["frames"], sz[1], sz[0]), device="cuda", generator=g)
    out = torch.empty_like(fr)
    f = lambda: cc.warp(c, 0, fr, ratio, axs, coord=coord, gather=gather, out=out)
    for _ in range(5):
        f()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(steps):
        f()
    e1.record()
    torch.cuda.synchronize()
    ms = e0.elapsed_time(e1) / steps
    npx = wl["frames"] * sz[0] * sz[1]
    gbs = npx * wl["bytes_per_px"] / ms / 1e6
    return ms, gbs / bench.measured_peak()[0], npx / ms / 1e6

if __name__ == "__main__":
    w = sys.argv[1] if len(sys.argv) > 1 else "c2"
    coords = [sys.argv[2]] if len(sys.argv) > 2 else ["f64", "f32"]
    gather = sys.argv[3] if len(sys.argv) > 3 else "auto"
    steps = int(sys.argv[4]) if len(sys.argv) > 4 else 30
    tag = os.path.basename(os.environ.get("CAMCAL_B200_LIB", "default"))
    for cd in coords:
        ms, frac, gpix = run(w, cd, gather, steps)
        print(f"{tag:28s} {w} {cd} {gather:6s} {ms:8.4f} ms  frac {frac:5.3f}  {gpix:7.1f} Gpix/s", flush=True)
