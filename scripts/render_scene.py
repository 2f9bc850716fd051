"""Offline dataset renderer: `python scripts/render_scene.py <input.ply|.npz> <cameras.json> <img_out> [--max-sh-deg N] [--batch K]`.
The B200 counterpart of the reference's `render` binary (bin/render.rs:14-180): renders the test split, then the
train split, of a 3DGS cameras.json to PNG files."""
import argparse
import os
import sys
import time

sys.path.insert(0, os.path.join(os.path.dirname(os.path.abspath(__file__)), ".."))
import websplat_b200 as ws   # noqa: E402


def main():
    ap = argparse.ArgumentParser(description="Dataset offline renderer. Renders to PNG files")
    ap.add_argument("input"); ap.add_argument("scene"); ap.add_argument("img_out")
    ap.add_argument("--max-sh-deg", type=int, default=3)
    ap.add_argument("--batch", type=int, default=1,
                    help="render up to this many consecutive cameras of equal resolution together (1..%d)" % ws.MAX_VIEWS)
    opt = ap.parse_args()
    if not 1 <= opt.batch <= ws.MAX_VIEWS:
        ap.error("--batch must be in [1, %d]" % ws.MAX_VIEWS)
    print("reading scene file '%s'" % opt.scene)
    scene = ws.Scene.from_json(opt.scene)
    ctx = ws.Context(0)
    print("reading point cloud file '%s'" % opt.input)
    pc = ws.scene.load_pointcloud(ws, ctx, opt.input)
    renderer = ws.GaussianRenderer.new(ctx, ws.FORMAT_RGBA16_FLOAT, pc.sh_deg(), pc.compressed())
    for split in (ws.scene.TEST, ws.scene.TRAIN):
        cams = scene.cameras(split)
        t0 = time.perf_counter()
        ws.scene.render_views(ws, ctx, renderer, pc, cams, opt.img_out, split, batch=opt.batch)
        print("rendering %s: %d views in %.2f s -> '%s'" % (split, len(cams), time.perf_counter() - t0, os.path.join(opt.img_out, split)))
    print("done!")


if __name__ == "__main__":
    main()
