#!/usr/bin/env python
"""bench.py -- headline benchmark of the hot path (BASELINE.json): rectified Mpix/s.

    python bench.py --gpus N --steps K --warmup W            # this framework, N B200s
    python bench.py --impl reference --gpus N --steps K ...  # CPU arm (oracle port of the reference)
    torchrun ... bench.py --gpus N ...                        # one rank per GPU (N > 1)
    python bench.py ... --dump-outputs DIR                    # also save the last timed step's output

The frames of the timed workload are seeded: the same arguments give the same frames on every run.

A step = one pass of full-frame rectification over one batch of synthetic frames:
  workload c2 (default): 64 frames 1080x1920 single-channel fp32 (BASELINE configs[1])
  workload c3:           16 frames 2160x3840 u8 RGB per step (ring slice of configs[2])
`value`  : whole-job Mpix/s with the batch resident in HBM (CUDA events, max over ranks)
`e2e`    : the same metric through the host entry point of the C ABI (pinned host buffers,
           H2D + D2H inside the timed region)
`roofline`: algorithmic bytes / kernel time against the measured HBM copy bandwidth
`cpu_baseline`: the oracle port of the reference's path on this box's host cores (rank 0, N=1)
One JSON line on stdout (rank 0).
"""
from __future__ import annotations

import argparse
import ctypes as C
import json
import os
import statistics
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

import numpy as np

N_CORNERS = (20, 14)
BENCH_VIEW = ((0.05, -0.04, 0.02), (-9.3, -6.4, 30.0))   # >= 99 % of output pixels in bounds
WORKLOADS = {
    # name: (sz1, sz2, frames per step, channels, bytes/px algorithmic, intr)
    "c2": dict(sz=(1080, 1920), frames=64, u8=False, bytes_per_px=8,
               intr=(1400.0, 1400.0, 540.0, 960.0, -0.12, 1.0), seed=1234,
               name="64 x 1080x1920 fp32 gray frames, full-frame rectification (BASELINE configs[1])"),
    "c4k": dict(sz=(2160, 3840), frames=16, u8=False, bytes_per_px=8,
                intr=(2800.0, 2800.0, 1080.0, 1920.0, -0.12, 1.0), seed=1234,
                name="16 x 2160x3840 fp32 gray frames, full-frame rectification (4K variant of configs[1])"),
    "c3": dict(sz=(2160, 3840), frames=16, u8=True, bytes_per_px=6,
               intr=(2800.0, 2800.0, 1080.0, 1920.0, -0.12, 1.0), seed=4321,
               name="16 x 2160x3840 u8 RGB frames per step (ring slice of BASELINE configs[2])"),
}


def measured_peak():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        try:
            return float(json.load(open(p))["hbm_gbs"]), "measured (MEASURED_PEAKS.json)"
        except Exception:
            pass
    return 6650.0, "fallback (B200_PROFILING.md)"


def recorded_traffic(key):
    """per-launch dram bytes from the committed ncu --set full capture, if any"""
    p = os.path.join(ROOT, "profiles", "traffic.json")
    if os.path.exists(p):
        try:
            return json.load(open(p)).get(key)
        except Exception:
            return None
    return None


def geometry(wl):
    """ratio / axs of the rectified output, from the synthetic board seen by the bench view.
    Pure host arithmetic on 280 corners (numpy): parameters, not the measured path."""
    intr, (rv, tv) = wl["intr"], BENCH_VIEW
    th = np.linalg.norm(rv)
    n = np.asarray(rv) / th
    K = np.array([[0, -n[2], n[1]], [n[2], 0, -n[0]], [-n[1], n[0], 0]])
    R = np.cos(th) * np.eye(3) + (1 - np.cos(th)) * np.outer(n, n) + np.sin(th) * K
    n1, n2 = N_CORNERS
    a, b = np.meshgrid(np.arange(n1, dtype=np.float64), np.arange(n2, dtype=np.float64), indexing="ij")
    P = np.stack([a.ravel(), b.ravel(), np.zeros(a.size)], 1) @ R.T + np.asarray(tv)
    uv = P[:, :2] / P[:, 2:3]
    uv = uv * (1 + intr[4] * np.sum(uv * uv, 1, keepdims=True))
    rc = uv * np.array(intr[:2]) + np.array(intr[2:4])
    return rc.reshape(n1, n2, 2)


def project_np(intr, views, obj):
    """World -> pixel of every board corner in every view, vectorised numpy: INPUT synthesis for the
    residual / fit workloads (parameters of the benchmark, not the measured path)."""
    rv, tv = views[:, :3], views[:, 3:]
    th = np.linalg.norm(rv, axis=1)
    n = rv / np.maximum(th, 1e-300)[:, None]
    K = np.zeros((len(views), 3, 3))
    K[:, 0, 1], K[:, 0, 2], K[:, 1, 0] = -n[:, 2], n[:, 1], n[:, 2]
    K[:, 1, 2], K[:, 2, 0], K[:, 2, 1] = -n[:, 0], -n[:, 1], n[:, 0]
    c, s_ = np.cos(th)[:, None, None], np.sin(th)[:, None, None]
    R = c * np.eye(3) + (1 - c) * n[:, :, None] * n[:, None, :] + s_ * K
    P = np.einsum("vij,cj->vci", R, obj / intr[5]) + tv[:, None, :]
    uv = P[..., :2] / P[..., 2:3]
    uv = uv * (1 + intr[4] * np.sum(uv * uv, -1, keepdims=True))
    return np.ascontiguousarray(uv * np.array(intr[:2]) + np.array(intr[2:4]))


class ClockSampler:
    """SM clock + throttle reasons via NVML while the timed region runs."""

    def __init__(self, index):
        self.samples, self.reasons, self.max_mhz = [], set(), None
        self._stop = threading.Event()
        self._t = None
        try:
            import pynvml
            pynvml.nvmlInit()
            self.nv = pynvml
            self.h = pynvml.nvmlDeviceGetHandleByIndex(index)
            self.max_mhz = pynvml.nvmlDeviceGetMaxClockInfo(self.h, pynvml.NVML_CLOCK_SM)
        except Exception:
            self.nv = None

    def _run(self):
        nv = self.nv
        names = {"hw_slowdown": 0x8, "sw_power_cap": 0x4, "hw_thermal_slowdown": 0x40,
                 "sw_thermal_slowdown": 0x20, "hw_power_brake": 0x80}
        while not self._stop.is_set():
            try:
                self.samples.append(nv.nvmlDeviceGetClockInfo(self.h, nv.NVML_CLOCK_SM))
                r = nv.nvmlDeviceGetCurrentClocksEventReasons(self.h)
                for k, bit in names.items():
                    if r & bit:
                        self.reasons.add(k)
            except Exception:
                pass
            time.sleep(0.0002)

    def start(self):
        if self.nv:
            self._t = threading.Thread(target=self._run, daemon=True)
            self._t.start()

    def stop(self):
        self._stop.set()
        if self._t:
            self._t.join()
        if not self.samples:
            return {"sm_mhz": None, "sm_max_mhz": self.max_mhz, "reasons": []}
        return {"sm_mhz": statistics.median(self.samples), "sm_max_mhz": self.max_mhz,
                "reasons": sorted(self.reasons), "samples": len(self.samples)}


def pinned_array(cc, shape, dtype):
    """numpy view of cudaHostAlloc'ed memory (cc_host_alloc)"""
    from cameracalibrations_b200 import _lib
    nbytes = int(np.prod(shape)) * np.dtype(dtype).itemsize
    p = C.c_void_p()
    _lib.check(_lib.lib.cc_host_alloc(C.byref(p), C.c_size_t(nbytes)))
    buf = (C.c_uint8 * nbytes).from_address(p.value)
    return np.frombuffer(buf, dtype=dtype).reshape(shape), p


DUMP_MAX_ELEMS = 4 << 20        # 16 MB of float32 per dumped file


def dump_outputs(out_dir, outputs):
    """--dump-outputs: every array as <out_dir>/<name>.npy in float32, flattened.  One larger than
    DUMP_MAX_ELEMS is reduced to a fixed sample (seed 0, sorted flat indices), the same for every run
    of the same workload, so that the outputs of two builds can be compared element for element.
    Every file holds finite numbers only: a NaN (the fill of a float frame's pixels that map outside
    the source) is written as 0, and <name>_nonfinite.npy is 1.0 where the output was not finite."""
    import torch
    os.makedirs(out_dir, exist_ok=True)
    for name, t in outputs.items():
        flat = t.reshape(-1)
        if flat.numel() > DUMP_MAX_ELEMS:
            idx = np.sort(np.random.default_rng(0).integers(0, flat.numel(), DUMP_MAX_ELEMS))
            flat = flat[torch.from_numpy(idx).to(flat.device)]
        vals = flat.float().cpu().numpy()
        bad = ~np.isfinite(vals)
        np.save(os.path.join(out_dir, name + ".npy"), np.where(bad, np.float32(0), vals))
        np.save(os.path.join(out_dir, name + "_nonfinite.npy"), bad.astype(np.float32))


def cpu_port(wl, nframes, nthreads, ratio, axs, steps=1, warmup=0):
    """The oracle restatement of the reference's warp on the host cores (checker code used
    only as the reported CPU baseline)."""
    from oracle import oracle_c as oc
    oc.build()
    sz = wl["sz"]
    ch = oc.chain(wl["intr"], *BENCH_VIEW)
    rng = np.random.default_rng(wl["seed"])
    if wl["u8"]:
        frames = rng.integers(0, 256, (nframes, sz[1], sz[0], 3), dtype=np.uint8)
        run = lambda: oc.rectify_u8c3(ch, 1.0 / ratio, axs, frames, nthreads=nthreads)
    else:
        frames = rng.random((nframes, sz[1], sz[0]), dtype=np.float32)
        run = lambda: oc.rectify_f32c1(ch, 1.0 / ratio, axs, frames, fill=np.nan, nthreads=nthreads)
    for _ in range(warmup):
        run()
    t0 = time.perf_counter()
    for _ in range(steps):
        run()
    dt = (time.perf_counter() - t0) / steps
    return nframes * sz[0] * sz[1] / dt / 1e6, dt


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=100)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--workload", default="c2", choices=sorted(WORKLOADS))
    ap.add_argument("--coord", default="f64", choices=["f64", "f32"],
                    help="coordinate arithmetic of the map (f64 = the reference's precision)")
    ap.add_argument("--gather", default="auto", choices=["auto", "direct", "tma"])
    ap.add_argument("--no-extras", action="store_true", help="skip the secondary workloads")
    ap.add_argument("--no-cpu", action="store_true", help="skip the cpu_baseline leg")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="write the output of the last timed step to DIR/rectified.npy (float32; a fixed "
                         "sample of 4M elements of rank 0's frames, non-finite values as 0) and where it was "
                         "not finite to DIR/rectified_nonfinite.npy")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "b200":
        ap.error("--dump-outputs needs --impl b200 (the reference arm sizes its sample from the host's speed)")
    args.warmup = max(args.warmup, 3)
    wl = WORKLOADS[args.workload]
    sz = wl["sz"]
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    ncores = len(os.sched_getaffinity(0))

    ip = geometry(wl)
    metric, unit = "rectified_mpix_per_s", "Mpix/s"
    config = {"workload": wl["name"], "frame": f"{sz[0]}x{sz[1]}", "frames_per_step_per_gpu": wl["frames"],
              "pixel": "u8x3" if wl["u8"] else "f32x1", "view": BENCH_VIEW, "intr": wl["intr"],
              "coord": args.coord, "parallelism": f"frame-sharded x{args.gpus} (no data-path collective)",
              "l2": "inputs+outputs per step exceed the 126 MB L2 (no flush needed)",
              "map_reuse": "the rectification map is built once per tile per group of <= 12 (f64) / 4 (f32) "
                           "frames of the batch and reused; every frame is read and written once per step"}
    if args.impl == "reference":
        config["coord"] = "f64"

    # ------------------------------------------------------------------ CPU arm
    if args.impl == "reference":
        if rank != 0:
            return
        from oracle import oracle_c as oc
        oc.build()
        ip_ratio = oc.get_ratio(ip, wl["intr"][5])
        axs = oc.get_axes(ip_ratio, wl["intr"][5], N_CORNERS, sz)
        # bounded sample per step: sized from one timed frame so the run ends within minutes
        _, per_frame = cpu_port(wl, 2, ncores, ip_ratio, axs)
        per_frame /= 2
        budget = 120.0 / (args.steps + args.warmup)
        nfr = max(1, min(wl["frames"], int(budget / max(per_frame, 1e-9))))
        v, dt = cpu_port(wl, nfr, ncores, ip_ratio, axs, steps=args.steps, warmup=args.warmup)
        sample = f"{nfr} of {wl['frames']} frames per step, {args.steps} steps, {ncores} OpenMP threads"
        print(json.dumps({
            "impl": "reference", "metric": metric, "value": v, "unit": unit, "n_gpus": args.gpus,
            "steps": args.steps, "warmup": args.warmup, "ms_per_step": dt * 1e3, "higher_is_better": True,
            "scaling": "weak", "vs_baseline": None, "dtype": "f64", "data": "synthetic", "config": config,
            "cpu_baseline": {"value": v, "unit": unit, "cores": ncores, "kind": "port", "sample": sample,
                             "note": "C restatement of the reference's Julia path (Julia is not "
                                     "installed on this image); faster than the Julia code would be"},
            "e2e": {"value": v, "unit": unit, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
            "gpu_launches": 0}))
        return

    # ------------------------------------------------------------------ B200 arm
    import torch
    import cameracalibrations_b200 as cc
    from cameracalibrations_b200 import _lib

    assert torch.cuda.is_available(), "bench.py needs a CUDA device (no CPU fallback)"
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    if world > 1:
        import torch.distributed as dist
        dist.init_process_group("nccl", device_id=dev)
    ctx = cc.context(local_rank)
    c = cc.Calibration(wl["intr"][:4], [BENCH_VIEW], 1.0 / wl["intr"][5], wl["intr"][4], ["extrinsic.png"])
    ratio = cc.get_ratio(ip, wl["intr"][5])
    axs = cc.get_axes(ratio, wl["intr"][5], N_CORNERS, sz)
    nfr = wl["frames"]
    npx = nfr * sz[0] * sz[1]

    g = torch.Generator(device=dev).manual_seed(wl["seed"] + rank)
    if wl["u8"]:
        src = torch.randint(0, 256, (nfr, sz[1], sz[0], 3), dtype=torch.uint8, device=dev, generator=g)
    else:
        src = torch.rand((nfr, sz[1], sz[0]), dtype=torch.float32, device=dev, generator=g)
    dst = torch.empty_like(src)
    step = lambda: cc.warp(c, 0, src, ratio, axs, coord=args.coord, gather=args.gather, out=dst)

    def barrier():
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
            torch.cuda.synchronize()

    for _ in range(args.warmup):
        step()
    barrier()
    sampler = ClockSampler(local_rank)
    sampler.start()
    l0 = ctx.launch_count()
    ev = [torch.cuda.Event(enable_timing=True) for _ in range(args.steps + 1)]
    ev[0].record()
    for i in range(args.steps):
        step()
        ev[i + 1].record()
    barrier()
    total_ms = ev[0].elapsed_time(ev[-1])
    launches = ctx.launch_count() - l0
    clocks = sampler.stop()
    per_step_ms = [ev[i].elapsed_time(ev[i + 1]) for i in range(args.steps)]
    kern_ms = statistics.mean(per_step_ms)          # one kernel launch per step
    tmax = torch.tensor([total_ms], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(tmax, op=dist.ReduceOp.MAX)
    total_ms = float(tmax.item())
    value = world * npx * args.steps / (total_ms * 1e-3) / 1e6
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, {"rectified": dst})

    # in-bounds fraction of the output (what share of the counted source bytes is really read)
    if wl["u8"]:
        inb = float((cc.warp(c, 0, torch.full_like(src[:1], 255), ratio, axs, coord=args.coord)[0, :, :, 0] == 255)
                    .float().mean().item())
    else:
        inb = float((~torch.isnan(dst[0])).float().mean().item())
    observed = {"in_bounds_fraction": round(inb, 4)}

    peak, peak_src = measured_peak()
    achieved = wl["bytes_per_px"] * npx / (kern_ms * 1e-3) / 1e9
    kname = ("rectify_u8c3" if wl["u8"] else "rectify_f32c1") + "_" + args.coord
    roofline = {"bound": "hbm", "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak,
                "traffic": recorded_traffic(f"{args.workload}_{args.coord}"), "peak_source": peak_src,
                "kernel": kname, "kernel_ms": kern_ms,
                "algorithmic_bytes_per_launch": wl["bytes_per_px"] * npx}

    # ---- e2e: host entry point of the C ABI, pinned host buffers, copies in the timed region
    # Bind this rank to the CPUs next to its GPU first, so that the pinned buffers (first touch) and
    # the enqueueing thread sit on the GPU's NUMA node; restored before the CPU baseline leg.
    cpus_before = os.sched_getaffinity(0)
    try:
        import pynvml
        pynvml.nvmlInit()
        pynvml.nvmlDeviceSetCpuAffinity(pynvml.nvmlDeviceGetHandleByIndex(local_rank))
        observed["e2e_cpu_affinity"] = f"nvml ideal cpus of gpu {local_rank} ({len(os.sched_getaffinity(0))} of {len(cpus_before)})"
    except Exception as ex:       # no NVML / not permitted: run unbound
        observed["e2e_cpu_affinity"] = f"unbound ({type(ex).__name__})"
    px_bytes = 3 if wl["u8"] else 4
    shape = tuple(src.shape)
    h_src, p1 = pinned_array(cc, shape, np.uint8 if wl["u8"] else np.float32)
    h_dst, p2 = pinned_array(cc, shape, np.uint8 if wl["u8"] else np.float32)
    h_src[...] = src.cpu().numpy()
    e2e_steps = max(3, min(args.steps, 10))
    for _ in range(2):
        cc.warp(c, 0, h_src, ratio, axs, coord=args.coord, gather=args.gather, out=h_dst)
    barrier()
    t0 = time.perf_counter()
    for _ in range(e2e_steps):
        cc.warp(c, 0, h_src, ratio, axs, coord=args.coord, gather=args.gather, out=h_dst)
    barrier()
    e2e_s = time.perf_counter() - t0
    te = torch.tensor([e2e_s], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(te, op=dist.ReduceOp.MAX)
    e2e_val = world * npx * e2e_steps / float(te.item()) / 1e6
    same = bool(np.array_equal(np.nan_to_num(h_dst[0], nan=-1.0),
                               np.nan_to_num(dst[0].cpu().numpy(), nan=-1.0)))
    dist = torch.distributed if world > 1 else None
    # what the host link can carry with every rank copying at once: pinned duplex memcpy, same buffers
    link = link_ceiling(torch, dist if world > 1 else None, dev, h_src, h_dst, src, dst)
    link_pix = world * link["duplex_gbs_per_dir_per_gpu"] * 1e9 / px_bytes / 1e6      # Mpix/s if only the copies ran
    e2e = {"value": e2e_val, "unit": unit, "link_ceiling": link, "link_frac": e2e_val / link_pix,
           "h2d_bytes_per_step": npx * px_bytes,
           "d2h_bytes_per_step": npx * px_bytes, "steps": e2e_steps,
           "api": "cc_rectify_%s_host via cameracalibrations_b200.warp(numpy)" % ("u8c3" if wl["u8"] else "f32c1"),
           "matches_device_path": same}
    _lib.lib.cc_host_free(p1)
    _lib.lib.cc_host_free(p2)
    del h_src, h_dst
    try:
        os.sched_setaffinity(0, cpus_before)
    except Exception:
        pass

    out = {"metric": metric, "value": value, "unit": unit, "n_gpus": world, "steps": args.steps,
           "warmup": args.warmup, "ms_per_step": total_ms / args.steps, "higher_is_better": True,
           "scaling": "weak", "vs_baseline": None, "dtype": args.coord, "data": "synthetic", "config": config,
           "roofline": roofline, "e2e": e2e, "gpu_launches": int(launches), "clocks": clocks, "observed": observed}

    if not args.no_extras:
        if world == 1:
            out["extras"] = extras(cc, torch, dev, c, args)
        sh = extras_sharded(cc, torch, dev, rank, world, args)          # collective: every rank takes part
        out.setdefault("extras", {}).update(sh)
    if rank == 0 and world == 1 and not args.no_cpu:
        nthreads = ncores
        from oracle import oracle_c as oc
        oc.build()
        # bounded sample: the whole batch, repeated for ~2 s of wall time on all host cores
        # (~30 core-seconds on 16 cores), sized from one untimed-quality pass
        _, dt1 = cpu_port(wl, nfr, nthreads, ratio, axs, steps=1, warmup=1)
        passes = int(min(50, max(3, np.ceil(2.0 / max(dt1, 1e-6)))))
        v, dt = cpu_port(wl, nfr, nthreads, ratio, axs, steps=passes, warmup=0)
        out["cpu_baseline"] = {"value": v, "unit": unit, "cores": nthreads, "kind": "port",
                               "sample": f"{nfr} of {nfr} frames x {passes} timed passes ({dt:.2f} s each, "
                                         f"{passes * dt * nthreads:.0f} core-seconds), {nthreads} OpenMP threads",
                               "note": "C restatement of the reference's Julia path (Julia is not installed "
                                       "on this image); faster than the Julia code would be"}
    if rank == 0:
        print(json.dumps(out))
    if world > 1:
        dist.destroy_process_group()


def link_ceiling(torch, dist, dev, h_src, h_dst, d_src, d_dst, reps=3):
    """Pinned host <-> device copies of the e2e buffers, both directions at once on two streams, all
    ranks at the same time: GB/s per direction per GPU (max time over ranks)."""
    hs, hd = torch.from_numpy(h_src), torch.from_numpy(h_dst)
    s1, s2 = torch.cuda.Stream(dev), torch.cuda.Stream(dev)
    nbytes = hs.numel() * hs.element_size()

    def run():
        torch.cuda.synchronize()
        if dist is not None:
            dist.barrier()
        t0 = time.perf_counter()
        for _ in range(reps):
            with torch.cuda.stream(s1):
                d_src.copy_(hs, non_blocking=True)
            with torch.cuda.stream(s2):
                hd.copy_(d_dst, non_blocking=True)
        torch.cuda.synchronize()
        t = torch.tensor([time.perf_counter() - t0], dtype=torch.float64, device=dev)
        if dist is not None:
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item()) / reps
    run()
    dt = run()
    return {"duplex_gbs_per_dir_per_gpu": nbytes / dt / 1e9, "bytes_per_dir": nbytes,
            "how": "cudaMemcpyAsync pinned<->device, H2D and D2H concurrently on two streams, every rank at once"}


def _time_ms(torch, fn, steps, warmup=3):
    for _ in range(warmup):
        fn()
    torch.cuda.synchronize()
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record()
    for _ in range(steps):
        fn()
    b.record()
    torch.cuda.synchronize()
    return a.elapsed_time(b) / steps


def extras(cc, torch, dev, c2cal, args):
    """Secondary workloads on ONE GPU (device-resident, CUDA events): every variant of the
    rectification kernels, and the whole fit of 100 views against OpenCV's calibrateCamera.  The
    workloads BASELINE.json names for 1/2/4/8 GPUs are in extras_sharded()."""
    peak, _ = measured_peak()
    ex = {}
    # the other variants of the rectification kernels
    for wname in ("c2", "c4k", "c3"):
        wl = WORKLOADS[wname]
        sz, nfr = wl["sz"], wl["frames"]
        cal = cc.Calibration(wl["intr"][:4], [BENCH_VIEW], 1.0, wl["intr"][4], ["extrinsic.png"])
        ratio = cc.get_ratio(geometry(wl), 1.0)
        axs = cc.get_axes(ratio, 1.0, N_CORNERS, sz)
        if wl["u8"]:
            src = torch.randint(0, 256, (nfr, sz[1], sz[0], 3), dtype=torch.uint8, device=dev)
        else:
            src = torch.rand((nfr, sz[1], sz[0]), dtype=torch.float32, device=dev)
        dst = torch.empty_like(src)
        for coord in ("f64", "f32"):
            if wname == args.workload and coord == args.coord:
                continue
            ms = _time_ms(torch, lambda: cc.warp(cal, 0, src, ratio, axs, coord=coord, gather=args.gather, out=dst), 20)
            npx = nfr * sz[0] * sz[1]
            gbs = wl["bytes_per_px"] * npx / (ms * 1e-3) / 1e9
            ex[f"rectify_{wname}_{coord}"] = {"mpix_per_s": npx / (ms * 1e-3) / 1e6, "ms": ms, "gb_per_s": gbs,
                                              "hbm_frac": gbs / peak}
        del src, dst
    # the reference's plot loop: every frame with its OWN view (src/plot_calibration.jl:36-42) -- 64 frames,
    # 64 views, one call of cc_rectify_f32c1_views; no map reuse is possible (one frame per view)
    wl = WORKLOADS["c2"]
    sz = wl["sz"]
    rngv = np.random.default_rng(3)
    vlist = [((BENCH_VIEW[0][0] + 0.002 * i, BENCH_VIEW[0][1], BENCH_VIEW[0][2] + 0.001 * i),
              (BENCH_VIEW[1][0] + 0.01 * i, BENCH_VIEW[1][1], BENCH_VIEW[1][2] + 0.05 * i)) for i in range(64)]
    calv = cc.Calibration(wl["intr"][:4], vlist, 1.0, wl["intr"][4], [f"{i}.png" for i in range(64)])
    ratio = cc.get_ratio(geometry(wl), 1.0)
    axs = cc.get_axes(ratio, 1.0, N_CORNERS, sz)
    src = torch.rand((64, sz[1], sz[0]), dtype=torch.float32, device=dev)
    dst = torch.empty_like(src)
    for coord in ("f64", "f32"):
        t0 = time.perf_counter()
        cc.warp_views(calv, list(range(64)), src, [ratio] * 64, [axs] * 64, coord=coord, out=dst)
        torch.cuda.synchronize()
        first_ms = (time.perf_counter() - t0) * 1e3
        ms = _time_ms(torch, lambda: cc.warp_views(calv, list(range(64)), src, [ratio] * 64, [axs] * 64, coord=coord, out=dst), 10)
        npx = 64 * sz[0] * sz[1]
        ex[f"rectify_views_64x1080p_{coord}"] = {
            "mpix_per_s": npx / (ms * 1e-3) / 1e6, "ms": ms, "hbm_frac": 8 * npx / (ms * 1e-3) / 1e9 / peak,
            "first_call_ms": first_ms,
            "note": "64 frames, 64 different views, one call = ONE launch (rectify_f32c1_views_kernel; tile plans cached after the first call); "
                    "first_call_ms includes building and uploading the 64 tile plans on the host"}
    del src, dst
    # the same loop on what the reference's plot actually warps: RGB{N0f8} images, here 16 views x 4K u8 RGB
    wl3 = WORKLOADS["c3"]
    sz3 = wl3["sz"]
    v16 = vlist[:16]
    cal3 = cc.Calibration(wl3["intr"][:4], v16, 1.0, wl3["intr"][4], [f"{i}.png" for i in range(16)])
    ratio3 = cc.get_ratio(geometry(wl3), 1.0)
    axs3 = cc.get_axes(ratio3, 1.0, N_CORNERS, sz3)
    src3 = torch.randint(0, 256, (16, sz3[1], sz3[0], 3), dtype=torch.uint8, device=dev)
    dst3 = torch.empty_like(src3)
    for coord in ("f64", "f32"):
        ms = _time_ms(torch, lambda: cc.warp_views(cal3, list(range(16)), src3, [ratio3] * 16, [axs3] * 16, coord=coord, out=dst3), 10)
        npx = 16 * sz3[0] * sz3[1]
        ex[f"rectify_views_16x4k_u8_{coord}"] = {
            "mpix_per_s": npx / (ms * 1e-3) / 1e6, "ms": ms, "hbm_frac": 6 * npx / (ms * 1e-3) / 1e9 / peak,
            "note": "16 u8 RGB 4K frames, 16 different views, one call = one launch (rectify_u8c3_views_kernel)"}
    del src3, dst3
    # ingest (SURVEY 8f rank 4): compressed JPEG bytes -> device frames -> the views call, nothing returns to
    # the host in between (the reference: FileIO.load + warp per file, src/plot_calibration.jl:36-42)
    try:
        import cv2
        yy, xx = np.mgrid[0:sz[0], 0:sz[1]]
        stills = [np.clip(np.stack([127 + 100 * np.sin(xx / (37.0 + i)) * np.cos(yy / 53.0), 127 + 90 * np.cos(xx / 71.0 + i),
                                    60 + 0.09 * xx + 0 * yy], -1), 0, 255).astype(np.uint8) for i in range(8)]
        blobs = [cv2.imencode(".jpg", im, [cv2.IMWRITE_JPEG_QUALITY, 92])[1].tobytes() for im in stills]
        fr8 = cc.load_jpegs(blobs)
        out8 = torch.empty_like(fr8)
        def ingest():
            cc.load_jpegs(blobs, out=fr8)
            cc.warp_views(calv, list(range(8)), fr8, [ratio] * 8, [axs] * 8, coord="f64", out=out8)
        for _ in range(2):
            ingest()
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        for _ in range(5):
            ingest()
        torch.cuda.synchronize()
        dt = (time.perf_counter() - t0) / 5
        ex["ingest_jpeg_8x1080p"] = {"mpix_per_s": 8 * sz[0] * sz[1] / dt / 1e6, "ms": dt * 1e3,
                                     "compressed_mb": sum(len(b) for b in blobs) / 1e6,
                                     "api": "cc_jpeg_decode_u8c3 (nvJPEG + transposition kernel) -> cc_rectify_u8c3_views, wall clock",
                                     "note": "decode-bound (nvJPEG hybrid backend: Huffman on the host); library code, not a roofline line"}
        del fr8, out8
    except Exception as e:                    # cv2 or libnvjpeg missing: the ingest line is optional
        ex["ingest_jpeg_8x1080p"] = {"unavailable": str(e)[:120]}
    wl = WORKLOADS["c3"]
    rng = np.random.default_rng(7)
    nv, nc = 10_000, 280
    views = np.concatenate([rng.normal(0, 0.3, (nv, 3)), np.array([-10.0, -7.0, 40.0]) + rng.normal(0, 2.0, (nv, 3))], 1)
    obj = np.array([[a, b, 0.0] for b in range(14) for a in range(20)], dtype=np.float64)
    to = torch.from_numpy(obj).to(dev)
    from cameracalibrations_b200 import lm
    # the whole fit (starting values on the host + device LM, CRITERIA 30 / 1e-3) on 100 noisy synthetic
    # views, and OpenCV's calibrateCamera -- the call the reference makes -- on the same corners (CPU)
    nvf = 100
    vf = views[:nvf]
    c100 = cc.Calibration(wl["intr"][:4], [(v[:3], v[3:]) for v in vf[:1]], 1.0, wl["intr"][4], ["extrinsic.png"])
    imgs = np.empty((nvf, nc, 2))
    for i in range(nvf):
        ci = cc.Calibration(wl["intr"][:4], [(vf[i, :3], vf[i, 3:])], 1.0, wl["intr"][4], ["extrinsic.png"])
        r_, q_ = ci.world2img(to[:, 0].contiguous(), to[:, 1].contiguous(), to[:, 2].contiguous(), 0)
        imgs[i, :, 0], imgs[i, :, 1] = r_.cpu().numpy(), q_.cpu().numpy()
    imgs += rng.normal(0, 0.1, imgs.shape)
    ti = torch.from_numpy(imgs).to(dev)
    for _ in range(2):                                   # warm: workspace of the context, NCCL not involved (1 rank)
        i0, v0 = lm.initial_guess_device(to, ti, (2160, 3840), 1.0)
        fit = lm.lm_fit_device(i0, v0, to, ti)
    torch.cuda.synchronize()
    samples = []                                         # wall clock of single calls: the median of 7
    for _ in range(7):
        t0 = time.perf_counter()
        i0, v0 = lm.initial_guess_device(to, ti, (2160, 3840), 1.0)
        torch.cuda.synchronize()
        t1 = time.perf_counter()
        fit = lm.lm_fit_device(i0, v0, to, ti)           # CRITERIA of the reference: 30 iterations, 1e-3
        torch.cuda.synchronize()
        t2 = time.perf_counter()
        samples.append((t2 - t0, t1 - t0, t2 - t1))
    samples.sort()
    tot_s, init_s, lm_s = samples[len(samples) // 2]
    th0 = time.perf_counter()
    lm.initial_guess(obj, imgs, (2160, 3840), 1.0)
    th1 = time.perf_counter()
    ex["fit_100_views"] = {"init_device_ms": init_s * 1e3, "lm_device_ms": lm_s * 1e3,
                           "total_ms": tot_s * 1e3, "total_ms_min_max": [samples[0][0] * 1e3, samples[-1][0] * 1e3],
                           "init_host_numpy_ms": (th1 - th0) * 1e3,
                           "rms_px": fit["rms"], "iterations": fit["iterations"],
                           "api": "cc_lm_initial_guess_f64 + cc_lm_fit_f64 (device arrays in, device-resident loop)"}
    try:
        import cv2
        flags = cv2.CALIB_ZERO_TANGENT_DIST + cv2.CALIB_FIX_K3 + cv2.CALIB_FIX_K2 + cv2.CALIB_FIX_ASPECT_RATIO
        crit = (cv2.TERM_CRITERIA_EPS + cv2.TERM_CRITERIA_MAX_ITER, 30, 0.001)
        t3 = time.perf_counter()
        rms = cv2.calibrateCamera([obj.astype(np.float32)] * nvf, [c_.astype(np.float32).reshape(-1, 1, 2) for c_ in imgs],
                                  (2160, 3840), np.eye(3), np.zeros(5), flags=flags, criteria=crit)[0]
        ex["fit_100_views"].update({"cv2_calibrateCamera_ms": (time.perf_counter() - t3) * 1e3, "cv2_rms_px": float(rms)})
    except Exception as e:          # cv2 missing: the comparison is optional
        ex["fit_100_views"]["cv2"] = f"unavailable ({type(e).__name__})"
    return ex


# FP64 arithmetic of reproj_jtj_kernel per corner (csrc/residual.cu, counted from the source; an FMA = 2):
# corner_jac ~ 150 (projection 22, distortion / chain-rule terms 40, rotation-derivative products 75,
# intrinsic columns 8) + normal-equation accumulation 2 rows x 66 FMAs = 264  ->  ~414 flop
FLOP_PER_CORNER = 414.0
# measured FP64 FMA issue rate of one B200 (profiles/r1_ubench_pipes.txt: 1.89 warp-DFMA / clk / SM)
FP64_PEAK_GFLOPS = 1.89 * 32 * 2 * 148 * 1.965


def extras_sharded(cc, torch, dev, rank, world, args):
    """The workloads BASELINE.json names for 1/2/4/8 GPUs, sharded over the ranks of this run
    (world == 1: one shard).  Device-side times are CUDA events, max over ranks; values are
    whole-job aggregates.
      c3_stream   configs[2]: 4096 frames 3840x2160 u8 RGB, frame-sharded, streamed from pinned host
                  memory through the host entry point of the C ABI (ring of device buffers,
                  H2D / kernel / D2H overlapped) -- end to end -- and the kernel alone on a
                  device-resident ring slice
      c4_points   configs[3]: 100 M random RowCol -> world (FP64 and FP32), point-sharded
      c5_*        configs[4]: residual + J'J over 10k views x 280 corners, view-sharded, with the NCCL
                  all-reduce of the normal-equation block inside the timed region (cc_allreduce_shared),
                  and full LM iterations of cc_lm_fit_f64 (two all-reduces each, no host sync)"""
    from cameracalibrations_b200 import lm, _lib
    from cameracalibrations_b200.shard import shard_range
    dist = torch.distributed if world > 1 else None
    peak, _ = measured_peak()
    ctx = cc.context(dev.index)
    if dist is not None:
        ctx.comm_init_from_torch()
    ex = {}

    def tmax(ms):
        t = torch.tensor([ms], dtype=torch.float64, device=dev)
        if dist is not None:
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item())

    def sync_all():
        torch.cuda.synchronize()
        if dist is not None:
            dist.barrier()
            torch.cuda.synchronize()

    def timed(fn, steps, warmup=3):
        for _ in range(warmup):
            fn()
        sync_all()
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        for _ in range(steps):
            fn()
        b.record()
        torch.cuda.synchronize()
        return tmax(a.elapsed_time(b) / steps)

    # ---- c3: 4K u8 RGB stream, frame-sharded
    wl = WORKLOADS["c3"]
    sz = wl["sz"]
    cal = cc.Calibration(wl["intr"][:4], [BENCH_VIEW], 1.0, wl["intr"][4], ["extrinsic.png"])
    ratio = cc.get_ratio(geometry(wl), 1.0)
    axs = cc.get_axes(ratio, 1.0, N_CORNERS, sz)
    total_frames = 4096
    lo, hi = shard_range(total_frames, rank, world)
    chunk = 64                                           # frames per host call: 1.6 GB in, 1.6 GB out, pinned
    h_src, p1 = pinned_array(cc, (chunk, sz[1], sz[0], 3), np.uint8)
    h_dst, p2 = pinned_array(cc, (chunk, sz[1], sz[0], 3), np.uint8)
    h_src[...] = np.random.default_rng(wl["seed"] + rank).integers(0, 256, h_src.shape, dtype=np.uint8)
    for coord in ("f64", "f32"):
        cc.warp(cal, 0, h_src[:16], ratio, axs, coord=coord, out=h_dst[:16])         # warm: plan, staging buffers
        sync_all()
        t0 = time.perf_counter()
        done = lo
        while done < hi:
            n = min(chunk, hi - done)
            cc.warp(cal, 0, h_src[:n], ratio, axs, coord=coord, out=h_dst[:n])       # cc_rectify_u8c3_host
            done += n
        torch.cuda.synchronize()
        dt = tmax((time.perf_counter() - t0) * 1e3) * 1e-3
        npx = total_frames * sz[0] * sz[1]
        ex[f"c3_stream_{coord}"] = {"frames": total_frames, "frames_per_rank": hi - lo, "mpix_per_s_e2e": npx / dt / 1e6,
                                    "seconds": dt, "host_gb_per_s_each_way": 3 * npx / dt / 1e9,
                                    "api": "cc_rectify_u8c3_host, 64-frame pinned chunks, 4-slot device ring"}
    _lib.lib.cc_host_free(p1)
    _lib.lib.cc_host_free(p2)
    del h_src, h_dst
    nfr = wl["frames"]
    src = torch.randint(0, 256, (nfr, sz[1], sz[0], 3), dtype=torch.uint8, device=dev)
    dst = torch.empty_like(src)
    for coord in ("f64", "f32"):
        ms = timed(lambda: cc.warp(cal, 0, src, ratio, axs, coord=coord, out=dst), 20)
        npx = world * nfr * sz[0] * sz[1]
        ex[f"c3_device_{coord}"] = {"mpix_per_s": npx / (ms * 1e-3) / 1e6, "ms": ms,
                                    "hbm_frac_per_gpu": wl["bytes_per_px"] * npx / world / (ms * 1e-3) / 1e9 / peak,
                                    "note": "16-frame ring slice resident in HBM per GPU (weak: every rank its own slice)"}
    del src, dst

    # ---- c4: 100 M points, point-sharded
    n_all = 100_000_000
    lo, hi = shard_range(n_all, rank, world)
    n = hi - lo
    for dt_, name, bpp in ((torch.float64, "f64", 40), (torch.float32, "f32", 20)):
        g = torch.Generator(device=dev).manual_seed(99 + rank)
        row = torch.rand(n, dtype=dt_, device=dev, generator=g) * 2160
        col = torch.rand(n, dtype=dt_, device=dev, generator=g) * 3840
        ms = timed(lambda: cal.img2world(row, col, 0), 10)
        x, y, z = cal.img2world(row, col, 0)
        ex[f"c4_img2world_{name}_100M"] = {"gpt_per_s": n_all / (ms * 1e-3) / 1e9, "ms": ms, "points_per_rank": n,
                                           "hbm_frac_per_gpu": bpp * n / (ms * 1e-3) / 1e9 / peak}
        ms = timed(lambda: cal.world2img(x, y, z, 0), 10)
        ex[f"c4_world2img_{name}_100M"] = {"gpt_per_s": n_all / (ms * 1e-3) / 1e9, "ms": ms, "points_per_rank": n,
                                           "hbm_frac_per_gpu": bpp * n / (ms * 1e-3) / 1e9 / peak}
        del row, col, x, y, z

    # ---- c5: 10k views x 280 corners, view-sharded, all-reduce inside the timed region
    rng = np.random.default_rng(7)
    nv_all, nc = 10_000, 280
    views = np.concatenate([rng.normal(0, 0.3, (nv_all, 3)),
                            np.array([-10.0, -7.0, 40.0]) + rng.normal(0, 2.0, (nv_all, 3))], 1)
    obj = np.array([[a, b, 0.0] for b in range(14) for a in range(20)], dtype=np.float64)
    lo, hi = shard_range(nv_all, rank, world)
    tv = torch.from_numpy(views[lo:hi]).to(dev)
    to = torch.from_numpy(obj).to(dev)
    ti = torch.from_numpy(project_np(wl["intr"], views[lo:hi], obj)).to(dev)     # synthetic detections: projection + noise
    ti += torch.randn(ti.shape, dtype=torch.float64, device=dev, generator=torch.Generator(device=dev).manual_seed(7 + rank)) * 0.25
    c0 = ctx.collective_count()
    ms = timed(lambda: cc.reproj_jtj(wl["intr"], 1.0, tv, to, ti), 20)
    flop = FLOP_PER_CORNER * nv_all * nc
    ex["c5_reproj_jtj_10k_views"] = {
        "views_per_s": nv_all / (ms * 1e-3), "ms": ms, "views_per_rank": hi - lo,
        "gb_per_s": 4936 * nv_all / (ms * 1e-3) / 1e9, "hbm_frac": 4936 * nv_all / world / (ms * 1e-3) / 1e9 / peak,
        "gflop_per_s": flop / (ms * 1e-3) / 1e9, "fp64_peak_gflop_per_s_per_gpu": FP64_PEAK_GFLOPS,
        "fp64_frac": flop / world / (ms * 1e-3) / 1e9 / FP64_PEAK_GFLOPS, "flop_per_corner": FLOP_PER_CORNER,
        "allreduce": "cc_allreduce_shared (NCCL, 21 doubles) inside the timed region" if world > 1 else "world of one",
        "collectives_per_call": (ctx.collective_count() - c0) / 23.0}
    # full LM iterations from a perturbed start: eps = 0 never stops early, so max_iter iterations run
    start = tv + 1e-3
    iters = 8
    intr0 = (wl["intr"][0] * 1.01, wl["intr"][1] * 1.01, wl["intr"][2] + 2.0, wl["intr"][3] - 2.0, 0.0)

    def fit():
        return lm.lm_fit_device(intr0, start, to, ti, max_iter=iters, eps=0.0)
    fit()
    sync_all()
    c0 = ctx.collective_count()
    t0 = time.perf_counter()
    r = fit()
    torch.cuda.synchronize()
    ms = tmax((time.perf_counter() - t0) * 1e3)
    ex["c5_lm_iterations_10k_views"] = {
        "us_per_iteration": ms * 1e3 / iters, "iterations": r["iterations"], "ms_total": ms, "rms_px": r["rms"],
        "collectives_per_iteration": max(0, ctx.collective_count() - c0 - 1) / iters,
        "what": "cc_lm_fit_f64: Schur + update + candidate residual/J'J + decision per iteration, state on the "
                "device, two all-reduces (21 + 23 doubles) and no host synchronisation; wall clock of the whole call "
                "(one first evaluation + 8 iterations + final read-back) / 8"}
    return ex


if __name__ == "__main__":
    main()
