"""bench.py's command line and JSON line.  The reference arm runs on the CPU (oracle port); the B200 arm
and its --dump-outputs need a GPU."""
import json
import os
import subprocess
import sys

import pytest

from conftest import ROOT


def test_reference_arm_json_contract():
    p = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--steps", "1",
                        "--warmup", "0"], capture_output=True, text=True, timeout=600, cwd=ROOT)
    assert p.returncode == 0, p.stderr[-2000:]
    d = json.loads(p.stdout.strip().splitlines()[-1])
    assert d["impl"] == "reference" and d["metric"] == "rectified_mpix_per_s" and d["unit"] == "Mpix/s"
    assert d["higher_is_better"] is True and d["value"] > 0 and d["steps"] == 1 and d["n_gpus"] == 1
    assert d["config"]["workload"].startswith("64 x 1080x1920 fp32")
    cb = d["cpu_baseline"]
    assert cb["kind"] == "port" and cb["cores"] >= 1 and cb["value"] == d["value"] and "frames" in cb["sample"]
    assert d["e2e"] == {"value": d["value"], "unit": "Mpix/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}


def test_reference_arm_other_ranks_are_silent():
    env = dict(os.environ, RANK="1", WORLD_SIZE="2", LOCAL_RANK="1")
    p = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--gpus", "2",
                        "--steps", "1", "--warmup", "0"], capture_output=True, text=True, timeout=120, cwd=ROOT, env=env)
    assert p.returncode == 0 and p.stdout.strip() == ""


def test_bench_rejects_zero_steps_and_dumps_of_the_reference_arm(tmp_path):
    for extra in (["--steps", "0"], ["--impl", "reference", "--dump-outputs", str(tmp_path)]):
        p = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py")] + extra, capture_output=True, text=True,
                           timeout=120, cwd=ROOT)
        assert p.returncode == 2 and p.stdout == "", extra
    assert not any(tmp_path.iterdir())


def test_dump_outputs_writes_finite_values_and_where_they_were_not_finite(tmp_path):
    """A NaN fill is stored as 0 in <name>.npy and as 1.0 in <name>_nonfinite.npy: finite files, nothing lost."""
    import numpy as np
    import torch

    import bench
    t = torch.arange(24, dtype=torch.float32).reshape(2, 3, 4)
    t[0, 1, 2] = float("nan")
    t[1, 0, 0] = float("-inf")
    bench.dump_outputs(str(tmp_path), {"out": t})
    vals, bad = np.load(tmp_path / "out.npy"), np.load(tmp_path / "out_nonfinite.npy")
    assert vals.dtype == np.float32 and bad.dtype == np.float32 and np.isfinite(vals).all()
    ref = t.reshape(-1).numpy()
    assert np.array_equal(bad, (~np.isfinite(ref)).astype(np.float32))
    assert np.array_equal(np.where(bad == 1, np.nan, vals), np.where(np.isfinite(ref), ref, np.nan), equal_nan=True)


def test_dump_outputs_samples_a_large_array_at_seeded_sorted_indices(tmp_path):
    """An array larger than DUMP_MAX_ELEMS is dumped as the elements at np.sort(default_rng(0).integers(0, n, k)):
    on t = arange(n) every dumped value is its own flat index."""
    import numpy as np
    import torch

    import bench
    n, k = bench.DUMP_MAX_ELEMS + 3 * 4096, bench.DUMP_MAX_ELEMS
    assert n < 1 << 24                                   # every index is exact in float32
    bench.dump_outputs(str(tmp_path), {"out": torch.arange(n, dtype=torch.float32).reshape(-1, 4096)})
    vals, bad = np.load(tmp_path / "out.npy"), np.load(tmp_path / "out_nonfinite.npy")
    assert vals.shape == (k,) and bad.shape == (k,) and not bad.any()
    assert np.all(np.diff(vals) >= 0) and vals[0] >= 0 and vals[-1] < n
    assert np.array_equal(vals, np.sort(np.random.default_rng(0).integers(0, n, k)).astype(np.float32))


@pytest.mark.gpu
def test_dump_outputs_is_the_output_of_the_timed_path(tmp_path):
    """--dump-outputs DIR: rectified.npy and rectified_nonfinite.npy hold what the timed steps computed
    (the seed-0 sample of cc.warp on the same seeded frames, bit for bit), finite, within 64 MB, and the
    same whatever the number of steps."""
    import numpy as np
    import torch

    import bench
    import cameracalibrations_b200 as cc
    names = ["rectified.npy", "rectified_nonfinite.npy"]
    dumps = []
    for steps in (1, 3):
        d = tmp_path / f"steps{steps}"
        p = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--steps", str(steps), "--warmup", "0",
                            "--no-extras", "--no-cpu", "--dump-outputs", str(d)],
                           capture_output=True, text=True, timeout=600, cwd=ROOT)
        assert p.returncode == 0, p.stderr[-2000:]
        assert json.loads(p.stdout.strip().splitlines()[-1])["steps"] == steps
        assert sorted(f.name for f in d.iterdir()) == names
        assert sum(f.stat().st_size for f in d.iterdir()) <= 64 << 20
        dumps.append([np.load(d / n) for n in names])
    for a in dumps[0]:
        assert a.dtype == np.float32 and np.isfinite(a).all()
    assert all(np.array_equal(a, b) for a, b in zip(dumps[0], dumps[1]))

    wl = bench.WORKLOADS["c2"]
    sz = wl["sz"]
    c = cc.Calibration(wl["intr"][:4], [bench.BENCH_VIEW], 1.0 / wl["intr"][5], wl["intr"][4], ["extrinsic.png"])
    ratio = cc.get_ratio(bench.geometry(wl), wl["intr"][5])
    axs = cc.get_axes(ratio, wl["intr"][5], bench.N_CORNERS, sz)
    g = torch.Generator(device="cuda").manual_seed(wl["seed"])
    src = torch.rand((wl["frames"], sz[1], sz[0]), dtype=torch.float32, device="cuda", generator=g)
    out = cc.warp(c, 0, src, ratio, axs).reshape(-1)
    idx = np.sort(np.random.default_rng(0).integers(0, out.numel(), bench.DUMP_MAX_ELEMS))
    ref = out[torch.from_numpy(idx).cuda()].cpu().numpy()
    assert np.array_equal(dumps[0][0], np.where(np.isnan(ref), np.float32(0), ref))
    assert np.array_equal(dumps[0][1], np.isnan(ref).astype(np.float32))
    assert 0 < dumps[0][1].mean() < 0.1                  # the bench view: a few fill pixels, mostly in bounds
