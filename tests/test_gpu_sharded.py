"""GPU tests of the sharded path.  world == 1 exercises the whole begin/exchange/finish/band sequence
on one GPU (the exchange then stores into local memory); the multi-GPU test runs on a machine with
2, 4 or 8 GPUs and checks that the sharded frame is BIT-IDENTICAL to the 1-GPU frame (it skips where fewer GPUs exist)."""
import os
import subprocess
import sys

import numpy as np
import pytest

from helpers import make_args, make_generic

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_sharded_world1_equals_plain(ws, orc, ctx):
    import torch
    cloud = ws.synth.make_cloud(50000, 31)
    W, H = 640, 360
    pos, rot = ws.synth.orbit_camera(110.0)
    fovx, fovy = ws.synth.fov_for_viewport(W, H)
    args = make_args(ws, cloud, pos, rot, W, H, fovx, fovy)
    pc = ws.PointCloud.new(ctx, make_generic(ws, cloud))
    plain = ws.GaussianRenderer.new(ctx, ws.FORMAT_RGBA32_FLOAT, 3, False)
    plain.set_occlusion_split(False)                     # num_pairs is compared below; sharded frames never split
    plain.prepare(None, pc, args)
    t = torch.empty((H, W, 4), dtype=torch.float32, device="cuda")
    plain.render(t, pc)
    torch.cuda.synchronize()
    sh = ws.ShardedRenderer(ws, ctx, ws.FORMAT_RGBA32_FLOAT, 3, False, pc, cloud["num_points"], (W, H))
    for _ in range(2):                                   # twice: buffers are reused frame to frame
        img = sh.frame(args)
        torch.cuda.synchronize()
        assert torch.equal(img, t)
    host = torch.zeros((H, W, 4), dtype=torch.float32).pin_memory()
    sh.frame_to_root(args, host=host)
    torch.cuda.synchronize()
    assert torch.equal(host, t.cpu())
    for _ in range(3):                                   # host-collective-free variant, epochs advance
        host.zero_()
        sh.frame_peer(args, host=host)
        torch.cuda.synchronize()
        assert torch.equal(host, t.cpu())
    # occlusion split inside the band (automatic from 2 M points per rank; forced here): same pixels from fewer pairs
    full_pairs = sh.stats()["num_pairs"]
    sh.r.set_occlusion_split(True)
    for _ in range(2):
        host.zero_()
        sh.frame_peer(args, host=host)
        torch.cuda.synchronize()
        assert torch.equal(host, t.cpu())
    assert sh.stats()["num_pairs"] <= full_pairs
    sh.r.set_occlusion_split(False)
    sh.frame_peer(args, host=host)
    torch.cuda.synchronize()
    st = sh.stats()
    # only splats that touch at least one tile are routed, so the received count can be below V
    assert st["num_visible"] <= plain.stats()["num_visible"] and st["num_pairs"] == plain.stats()["num_pairs"]
    # timing off: the frame runs as a CUDA graph, one per frame-buffer parity (two captures, then a replay)
    sh.r.set_timing(False)
    for _ in range(3):
        host.zero_()
        sh.frame_peer(args, host=host)
        torch.cuda.synchronize()
        assert torch.equal(host, t.cpu())
    # two frames in flight through the gated path (world 1: the gates wait on this rank's own flags)
    pipe = ws.ShardedPipeline(ws, ctx, ws.FORMAT_RGBA32_FLOAT, 3, False, pc, cloud["num_points"], (W, H), depth=2)
    hosts = [torch.zeros((H, W, 4), dtype=torch.float32).pin_memory() for _ in range(4)]
    for h in hosts:
        pipe.frame_peer(args, host=h)
    pipe.synchronize()
    torch.cuda.synchronize()
    for h in hosts:
        assert torch.equal(h, t.cpu())
    assert pipe.rebalance() == [0, (H + 15) // 16]


def _gpu_count():
    try:
        import torch
        return torch.cuda.device_count()
    except Exception:
        return 0


@pytest.mark.parametrize("world", [2, 4, 8])
def test_sharded_frames_bit_identical_to_one_gpu(world):
    """SURVEY.md 8(e): G in {1, 2, 4, 8} images bit-identical.  tests/sharded_worker.py renders the same frames on `world`
    GPUs (all three exchange variants, two frames in flight over re-cut bands, a cfg5-style cloud whose shards are
    generated per rank) and on one GPU and requires torch.equal.  Needs `world` GPUs; the log of the
    8-GPU run is committed under profiles/."""
    if _gpu_count() < world:
        pytest.skip("needs %d GPUs, this machine has %d" % (world, _gpu_count()))
    env = dict(os.environ, PYTHONPATH=ROOT)
    cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node=%d" % world, "--master-addr", "127.0.0.1",
           "--master-port", str(29517 + world), os.path.join(ROOT, "tests", "sharded_worker.py")]
    p = subprocess.run(cmd, env=env, capture_output=True, text=True, timeout=900)
    log = os.environ.get("WS_SHARDED_LOG_DIR")
    if log:
        with open(os.path.join(log, "sharded_worker_world%d.log" % world), "w") as f:
            f.write(p.stdout[-20000:] + "\n--- stderr tail ---\n" + p.stderr[-3000:])
    assert p.returncode == 0, p.stdout[-3000:] + p.stderr[-3000:]
    assert "SHARDED_OK" in p.stdout
