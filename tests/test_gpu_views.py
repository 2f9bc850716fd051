"""Batches of views (ws_renderer_prepare_views / render_views): every view of a batch must be bit-identical to the same
view rendered alone through prepare + render, whatever the format, viewport, occlusion split or CUDA-graph setting."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest

from helpers import make_args, make_generic

pytestmark = pytest.mark.gpu

FMT_TORCH = {0: "uint8", 1: "float16", 2: "float32"}


@pytest.fixture(scope="module")
def cloud(ws):
    return ws.synth.make_cloud(60000, 31)


@pytest.fixture(scope="module")
def pc(ws, ctx, cloud):
    return ws.PointCloud.new(ctx, make_generic(ws, cloud))


def _views(ws, cloud, K, W, H, **kw):
    fovx, fovy = ws.synth.fov_for_viewport(W, H)
    out = []
    for v in range(K):
        pos, rot = ws.synth.orbit_camera(360.0 * v / max(K, 1) + 11.0, radius=2.6 + 0.15 * v)
        out.append(make_args(ws, cloud, pos, rot, W, H, fovx, fovy, **kw))
    return out


def _renderer(ws, ctx, fmt, compressed=False, split=None, graphs=True):
    r = ws.GaussianRenderer.new(ctx, fmt, 3, compressed)
    r.set_occlusion_split(split)
    if graphs:
        r.set_timing(False)                 # graphs are captured only with timing off
    else:
        r.set_cuda_graphs(False)
    return r


def _single(ws, r, pc, args, fmt, clear=(0.1, 0.2, 0.3, 0.4)):
    import torch
    W, H = args.viewport
    t = torch.full((H, W, 4), 7, dtype=getattr(torch, FMT_TORCH[fmt]), device="cuda")
    r.prepare(None, pc, args)
    r.render(t, pc, clear=clear)
    n = r.num_visible_points()
    return t.view(torch.uint8).clone(), n


def _batch(ws, r, pc, args, fmt, clear=(0.1, 0.2, 0.3, 0.4)):
    import torch
    W, H = args[0].viewport
    t = torch.full((len(args), H, W, 4), 7, dtype=getattr(torch, FMT_TORCH[fmt]), device="cuda")
    r.prepare_views(None, pc, args)
    r.render_views(t, pc, clear=clear)
    torch.cuda.synchronize()
    return t.view(torch.uint8).clone()


def _check_batch(ws, ctx, pc, args, fmt, compressed=False, split=None, graphs=True, repeat=False):
    import torch
    rb = _renderer(ws, ctx, fmt, compressed, split, graphs)
    rs = _renderer(ws, ctx, fmt, compressed, split, graphs)
    out = _batch(ws, rb, pc, args, fmt)
    counts = rb.views_num_visible_points()
    st = rb.stats()
    W, H = args[0].viewport
    T = ((W + 15) // 16) * ((H + 15) // 16)
    assert st["num_tiles"] == len(args) * T and (st["width"], st["height"]) == (W, H)
    assert st["num_visible"] == sum(counts)
    for v, a in enumerate(args):
        ref, n = _single(ws, rs, pc, a, fmt)
        assert counts[v] == n, "view %d: %d visible in the batch, %d alone" % (v, counts[v], n)
        assert torch.equal(out[v], ref), "view %d of %d differs from the view rendered alone" % (v, len(args))
    if repeat:
        again = _batch(ws, rb, pc, args, fmt)
        assert torch.equal(again, out)
    return counts


@pytest.mark.parametrize("K", [1, 2, 3, 8])
@pytest.mark.parametrize("viewport", [(1200, 799), (33, 17)])
def test_batch_views_equal_single_views(ws, ctx, cloud, pc, K, viewport):
    W, H = viewport
    args = _views(ws, cloud, K, W, H)
    for fmt in (ws.FORMAT_RGBA8_UNORM, ws.FORMAT_RGBA16_FLOAT, ws.FORMAT_RGBA32_FLOAT):
        for split in (False, True, None):
            for graphs in (True, False):
                counts = _check_batch(ws, ctx, pc, args, fmt, split=split, graphs=graphs, repeat=(fmt == ws.FORMAT_RGBA32_FLOAT))
    if W > 100:
        assert min(counts) > 1000        # the orbit views see the cloud


def test_batch_views_with_different_settings(ws, ctx, cloud, pc):
    W, H = 640, 360
    fovx, fovy = ws.synth.fov_for_viewport(W, H)
    box = ws.Aabb([-0.5, -0.6, -0.4], [0.4, 0.5, 0.6])
    kws = [dict(), dict(clipping_box=box), dict(max_sh_deg=0), dict(max_sh_deg=1, mip_splatting=True, kernel_size=0.5),
           dict(max_sh_deg=2, gaussian_scaling=0.6, walltime=0.3), dict(mip_splatting=False, kernel_size=0.1, gaussian_scaling=1.4)]
    args = []
    for v, kw in enumerate(kws):
        pos, rot = ws.synth.orbit_camera(40.0 * v)
        args.append(make_args(ws, cloud, pos, rot, W, H, fovx, fovy, **kw))
    for graphs in (True, False):
        _check_batch(ws, ctx, pc, args, ws.FORMAT_RGBA32_FLOAT, graphs=graphs)


def test_batch_views_compressed(ws, ctx):
    cc = ws.synth.make_cloud_compressed(80000, 33)
    pcc = ws.PointCloud.new(ctx, make_generic(ws, cc))
    args = _views(ws, cc, 3, 800, 600)
    args[1].max_sh_deg = 1
    for split in (False, True):
        _check_batch(ws, ctx, pcc, args, ws.FORMAT_RGBA16_FLOAT, compressed=True, split=split)


def test_batch_edge_views(ws, ctx, cloud, pc):
    """A camera that sees nothing, two identical cameras and a normal view in one batch."""
    W, H = 320, 200
    fovx, fovy = ws.synth.fov_for_viewport(W, H)
    pos, rot = ws.synth.orbit_camera(30.0)
    away = make_args(ws, cloud, ws.synth.orbit_camera(30.0, radius=50.0)[0], ws.synth.orbit_camera(210.0)[1], W, H, fovx, fovy)
    same = make_args(ws, cloud, pos, rot, W, H, fovx, fovy)
    other = make_args(ws, cloud, *ws.synth.orbit_camera(100.0), W, H, fovx, fovy)
    for graphs in (True, False):
        counts = _check_batch(ws, ctx, pc, [away, same, same, other], ws.FORMAT_RGBA8_UNORM, graphs=graphs)
        assert counts[0] == 0 and counts[1] == counts[2] > 0


def test_batch_three_tile_passes(ws, ctx):
    """2048 x 2048 with K = 5: 81 920 tiles, above the 65 536 of two tile-id passes."""
    c = ws.synth.make_cloud(40000, 35)
    p = ws.PointCloud.new(ctx, make_generic(ws, c))
    _check_batch(ws, ctx, p, _views(ws, c, 5, 2048, 2048), ws.FORMAT_RGBA8_UNORM, split=False)


@pytest.mark.parametrize("name,K", [("cfg3", 4), ("cfg4", 3)])
def test_batch_full_size(ws, ctx, name, K):
    n, W, H, seed, compressed = ws.synth.CONFIGS[name]
    c = ws.synth.make_cloud_compressed(n, seed) if compressed else ws.synth.make_cloud(n, seed)
    p = ws.PointCloud.new(ctx, make_generic(ws, c))
    views = ws.synth.orbit_views(36)
    fovx, fovy = ws.synth.fov_for_viewport(W, H)
    args = [make_args(ws, c, *views[9 * v], W, H, fovx, fovy) for v in range(K)]
    _check_batch(ws, ctx, p, args, ws.FORMAT_RGBA16_FLOAT, compressed=compressed)


def test_batch_to_host_matches_device(ws, ctx, cloud, pc):
    import torch
    args = _views(ws, cloud, 3, 200, 120)
    r = _renderer(ws, ctx, ws.FORMAT_RGBA16_FLOAT)
    dev = _batch(ws, r, pc, args, ws.FORMAT_RGBA16_FLOAT)
    host = torch.empty((3, 120, 200, 4), dtype=torch.float16).pin_memory()
    r.prepare_views(None, pc, args)
    r.render_views_to_host(host, pc, clear=(0.1, 0.2, 0.3, 0.4))
    torch.cuda.synchronize()
    assert torch.equal(host.view(torch.uint8), dev.cpu())
    # a padded layout: rows of 256 pixels, views 130 rows apart
    pad = torch.zeros((3, 130, 256, 4), dtype=torch.float16, device="cuda")
    r.prepare_views(None, pc, args)
    r.render_views(pad, pc, clear=(0.1, 0.2, 0.3, 0.4), row_pitch=256 * 8, view_stride=130 * 256 * 8)
    torch.cuda.synchronize()
    assert torch.equal(pad[:, :120, :200].contiguous().view(torch.uint8), dev)
    assert not pad[:, 120:].any() and not pad[:, :, 200:].any()


def test_batch_errors(ws, ctx, cloud, pc):
    import torch
    W, H = 96, 64
    args = _views(ws, cloud, 3, W, H)
    r = _renderer(ws, ctx, ws.FORMAT_RGBA32_FLOAT)
    t = torch.empty((3, H, W, 4), dtype=torch.float32, device="cuda")

    def status(fn):
        with pytest.raises(ws.WsError) as e:
            fn()
        return e.value.status

    assert status(lambda: r.prepare_views(None, pc, [])) == ws.WS_ERR_INVALID_ARGUMENT
    assert status(lambda: r.prepare_views(None, pc, _views(ws, cloud, ws.MAX_VIEWS + 1, W, H))) == ws.WS_ERR_INVALID_ARGUMENT
    assert status(lambda: r.prepare_views(None, pc, args[:2] + _views(ws, cloud, 1, W, H + 1))) == ws.WS_ERR_INVALID_ARGUMENT
    bad = _views(ws, cloud, 2, W, H)
    bad[1].max_sh_deg = 4                                    # each view goes through the single-frame checks
    assert status(lambda: r.prepare_views(None, pc, bad)) == ws.WS_ERR_INVALID_ARGUMENT
    r.prepare_views(None, pc, args)
    assert status(lambda: r.render_views(t, pc, view_stride=H * W * 16 - 16)) == ws.WS_ERR_INVALID_ARGUMENT
    assert status(lambda: r.render(t, pc)) == ws.WS_ERR_INVALID_ARGUMENT
    assert status(lambda: r.render_to_host(np.empty((H, W, 4), np.float32), pc)) == ws.WS_ERR_INVALID_ARGUMENT
    assert status(lambda: r.read_buffer(ws.BUF_SPLATS_2D)) == ws.WS_ERR_UNSUPPORTED
    assert status(lambda: r.camera_uniform()) == ws.WS_ERR_UNSUPPORTED
    assert status(lambda: r.settings_uniform()) == ws.WS_ERR_UNSUPPORTED
    r.render_views(t, pc)
    r.prepare(None, pc, args[0])
    assert status(lambda: r.render_views(t, pc)) == ws.WS_ERR_INVALID_ARGUMENT
    assert status(lambda: r.views_num_visible_points()) == ws.WS_ERR_INVALID_ARGUMENT
    r.render(t[0], pc)
    torch.cuda.synchronize()
    # a sharded renderer takes no batches
    rsh = ws.GaussianRenderer.new(ctx, ws.FORMAT_RGBA32_FLOAT, 3, False)
    _status = ws.lib().ws_renderer_shard_configure(rsh._h, 0, 1, pc.num_points(), pc.num_points(), W, H)
    assert _status == ws.WS_OK
    assert status(lambda: rsh.prepare_views(None, pc, args)) == ws.WS_ERR_INVALID_ARGUMENT
    # pair capacity exceeded: reported by the next call, through the deferred frame status
    r.set_pair_capacity(100)
    r.prepare_views(None, pc, args); r.render_views(t, pc)
    torch.cuda.synchronize()
    assert status(lambda: r.prepare_views(None, pc, args)) == ws.WS_ERR_PAIR_OVERFLOW
    r.set_pair_capacity(0)
    r.prepare_views(None, pc, args); r.render_views(t, pc)
    assert r.stats()["num_pairs"] > 100
    # K x N >= 2^30: the look-back words carry 30-bit counts.  An all-zero compressed cloud of 2^27 points is enough.
    n = 1 << 27
    big = ws.GenericGaussianPointCloud(np.zeros(n * 24, np.uint8), np.zeros(48, np.uint8), 3, n,
                                       ws.Aabb([-1, -1, -1], [1, 1, 1]), [0, 0, 0], compressed=True, covars=np.zeros(12, np.uint8))
    pbig = ws.PointCloud.new(ctx, big)
    rbig = ws.GaussianRenderer.new(ctx, ws.FORMAT_RGBA8_UNORM, 3, True)
    assert status(lambda: rbig.prepare_views(None, pbig, _views(ws, cloud, 8, W, H))) == ws.WS_ERR_UNSUPPORTED
    rbig.close(); pbig.close()


def test_render_scene_batch_writes_the_same_pngs(ws, tmp_path):
    n, W, H = 20000, 320, 200
    ply = tmp_path / "cloud.ply"
    ply.write_bytes(ws.synth.ply_bytes(ws.synth.ply_vertices(n, 8, 3), 3))
    fovx, fovy = ws.synth.fov_for_viewport(W, H)
    entries = []
    for i in range(11):
        pos, rot = ws.synth.orbit_camera(360.0 * i / 11, radius=3.0 + 0.1 * i)
        cam = ws.PerspectiveCamera(pos, rot, ws.PerspectiveProjection(fovx, fovy, 0.01, 100.0))
        size = (W, H) if i != 5 else (W + 32, H)              # one camera of another size splits a batch
        entries.append(ws.SceneCamera.from_perspective(ws, cam, "img_%03d" % i, i, size).to_json())
    cams = tmp_path / "cameras.json"
    cams.write_text(json.dumps(entries))
    root = os.path.join(os.path.dirname(os.path.abspath(__file__)), "..")
    outs = {}
    for batch in (1, 4):
        out = tmp_path / ("out%d" % batch)
        p = subprocess.run([sys.executable, os.path.join(root, "scripts", "render_scene.py"), str(ply), str(cams), str(out),
                            "--batch", str(batch)], capture_output=True, text=True, timeout=300)
        assert p.returncode == 0, p.stdout + p.stderr
        outs[batch] = {os.path.join(s, f): (out / s / f).read_bytes() for s in ("test", "train") for f in sorted(os.listdir(out / s))}
    assert len(outs[1]) == 11 and outs[1] == outs[4]
