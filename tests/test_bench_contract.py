"""The bench.py contract: the reference arm (CPU oracle) prints ONE JSON line with the keys a consumer of the result reads,
the GPU arm refuses to run without a CUDA device (no CPU fallback), and --dump-outputs writes the frame of the last timed
step (checked on the CPU through the reference arm, and on a GPU through the single-GPU arm)."""
import json
import os
import subprocess
import sys

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _run(*argv, env=None):
    return subprocess.run([sys.executable, os.path.join(ROOT, "bench.py")] + list(argv), capture_output=True, text=True,
                          timeout=600, env=dict(os.environ, **(env or {})))


def test_reference_arm_prints_one_json_line():
    p = _run("--impl", "reference", "--workload", "cfg1", "--steps", "2", "--warmup", "1")
    assert p.returncode == 0, p.stderr[-2000:]
    lines = [ln for ln in p.stdout.splitlines() if ln.strip()]
    assert len(lines) == 1
    d = json.loads(lines[0])
    assert d["impl"] == "reference" and d["metric"] == "frames/sec" and d["unit"] == "frames/s" and d["higher_is_better"] is True
    assert d["steps"] == 2 and d["warmup"] == 1 and d["config"]["steps_requested"] == 2 and d["value"] > 0 and abs(d["ms_per_step"] * d["value"] - 1000.0) < 1.0
    assert d["cpu_baseline"]["kind"] == "port" and d["cpu_baseline"]["cores"] >= 1 and d["cpu_baseline"]["value"] == d["value"]
    assert d["e2e"] == {"value": d["value"], "unit": "frames/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}
    assert d["config"]["workload"].startswith("cfg1: 100000 synthetic Gaussians")
    assert d["gpu_launches"] == 0


def test_reference_arm_under_torchrun_only_rank0_works():
    p = _run("--impl", "reference", "--workload", "cfg1", "--steps", "1", "--warmup", "0", env={"RANK": "3", "WORLD_SIZE": "4"})
    assert p.returncode == 0 and p.stdout.strip() == ""


def test_gpu_arm_fails_loudly_without_a_gpu():
    try:
        import torch
        if torch.cuda.is_available():
            import pytest
            pytest.skip("a GPU is present")
    except ImportError:
        pass
    p = _run("--workload", "cfg1", "--steps", "1")
    assert p.returncode != 0 and "no CUDA device" in (p.stderr + p.stdout)


def test_reference_arm_sets_its_own_thread_count():
    """torchrun exports OMP_NUM_THREADS=1 to every rank; the reference arm (and the GPU arm's cpu_baseline) must not inherit
    it -- round 1's N >= 2 reference lines ran on one core (VERDICT r01, weak 10)."""
    p = _run("--impl", "reference", "--workload", "cfg1", "--steps", "1", "--warmup", "0", env={"OMP_NUM_THREADS": "1", "RANK": "0", "WORLD_SIZE": "2"})
    assert p.returncode == 0, p.stderr[-2000:]
    d = json.loads(p.stdout.strip().splitlines()[-1])
    try:
        want = len(os.sched_getaffinity(0))
    except AttributeError:
        want = os.cpu_count()
    assert d["cpu_baseline"]["cores"] == want


def test_frame_crc_is_a_full_frame_hash():
    """the parity evidence carried by the bench lines: every byte of the downloaded frame enters the checksum"""
    import numpy as np
    sys.path.insert(0, ROOT)
    import bench
    a = np.zeros((64, 48, 4), np.float16)
    c0 = bench.frame_crc(a)
    for y, x, ch in ((0, 0, 0), (63, 47, 3), (31, 7, 2)):
        b = a.copy(); b[y, x, ch] = np.float16(6.1e-5)
        assert bench.frame_crc(b) != c0
    assert bench.frame_crc(a.copy()) == c0 and len(c0) == 8


def test_reference_arm_dumps_the_frame_of_its_last_step(tmp_path):
    """--dump-outputs: the image the timed path computed, as float32 (cfg1 has one view, so every step renders it)"""
    import numpy as np
    sys.path.insert(0, ROOT)
    import bench
    import websplat_b200 as ws
    from oracle import oracle as orc
    p = _run("--impl", "reference", "--workload", "cfg1", "--steps", "2", "--warmup", "0", "--dump-outputs", str(tmp_path))
    assert p.returncode == 0, p.stderr[-2000:]
    assert sorted(os.listdir(tmp_path)) == ["image.npy"]
    img = np.load(tmp_path / "image.npy")
    cloud, W, H, views = bench.make_workload("cfg1")
    fovx, fovy = ws.synth.fov_for_viewport(W, H)
    want = orc.render_frame(cloud, views[0][0], views[0][1], W, H, fovx, fovy)["image"]
    assert img.dtype == np.float32 and np.array_equal(img, want)


def test_dump_outputs_samples_a_large_frame(tmp_path):
    """a frame above DUMP_PIXELS pixels is written as a fixed seeded pixel sample plus its indices, within 64 MB"""
    import numpy as np
    sys.path.insert(0, ROOT)
    import bench
    H, W = 2160, 3840
    frame = np.random.default_rng(3).random((H, W, 4)).astype(np.float16)
    bench.dump_outputs(str(tmp_path / "a"), frame)
    bench.dump_outputs(str(tmp_path / "b"), frame[::-1].copy())
    img, idx = np.load(tmp_path / "a" / "image.npy"), np.load(tmp_path / "a" / "image_pixel_index.npy")
    assert img.dtype == np.float32 and idx.dtype == np.float64 and img.shape == (bench.DUMP_PIXELS, 4) and idx.shape == (bench.DUMP_PIXELS,)
    assert np.array_equal(img, frame.reshape(-1, 4)[idx.astype(np.int64)].astype(np.float32))
    assert np.array_equal(idx, np.load(tmp_path / "b" / "image_pixel_index.npy"))      # the sample does not depend on the frame
    assert sum(f.stat().st_size for f in (tmp_path / "a").iterdir()) <= 64e6


@pytest.mark.gpu
def test_gpu_arm_dumps_the_frame_of_its_last_step(ctx, tmp_path):
    """--dump-outputs of the single-GPU arm: the RGBA16F frame of the last timed step, as float32, equal to the same view
    rendered through the API (cfg1 has one view, so every step renders it)"""
    import numpy as np
    import torch
    sys.path.insert(0, ROOT)
    import bench
    import websplat_b200 as ws
    p = _run("--workload", "cfg1", "--steps", "5", "--warmup", "2", "--no-cpu-baseline", "--no-extra", "--dump-outputs", str(tmp_path))
    assert p.returncode == 0, p.stderr[-2000:]
    assert json.loads(p.stdout.strip().splitlines()[-1])["steps"] == 5
    img = np.load(tmp_path / "image.npy")
    cloud, W, H, views = bench.make_workload("cfg1")
    pc = ws.PointCloud.new(ctx, ws.GenericGaussianPointCloud(cloud["gaussians"], cloud["sh_coefs"], cloud["sh_deg"], cloud["num_points"],
                                                              ws.Aabb(cloud["aabb_min"], cloud["aabb_max"]), cloud["center"]))
    r = ws.GaussianRenderer.new(ctx, ws.FORMAT_RGBA16_FLOAT, cloud["sh_deg"], False)
    r.prepare(None, pc, bench.frame_args(ws, cloud, views[0], W, H))
    target = torch.empty((H, W, 4), dtype=torch.float16, device="cuda")
    r.render(target, pc)
    torch.cuda.synchronize()
    assert img.dtype == np.float32 and np.array_equal(img, target.cpu().numpy().astype(np.float32))
