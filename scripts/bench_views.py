"""Batches of views against single frames: `python scripts/bench_views.py [--workloads cfg1,cfg2,cfg3,cfg4] [--seconds 1.0]`.

For every workload of bench.py (same clouds, viewports and pair capacity) and K in {1, 2, 4, 8} orbit views of the cloud,
measures views/s of
  * batch:  ws_renderer_prepare_views + render_views of the K views, one renderer, one stream;
  * single: the same K views as K single frames with two frames in flight (two renderers, two streams: bench.py's default).
Both paths run in one process and alternate in windows of about seconds / 4 of GPU time, timed with CUDA events, after a
warm-up.  Prints one JSON line per workload with the CRC-32 of every view from both paths (they must match), the
per-stage times of one batch (a separate renderer with timing on) and the device name, power limit and SM clock limit.
Writes nothing but stdout."""
import argparse
import json
import os
import subprocess
import sys

ROOT = os.path.join(os.path.dirname(os.path.abspath(__file__)), "..")
sys.path.insert(0, ROOT)
import bench                 # noqa: E402  (make_workload / frame_args / frame_crc: the bench.py workloads)
import websplat_b200 as ws   # noqa: E402

KS = (1, 2, 4, 8)
DEPTH = 2                    # single frames in flight


def device_info():
    p = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True)
    line = p.stdout.strip().splitlines()[0] if p.returncode == 0 and p.stdout.strip() else ""
    f = [x.strip() for x in line.split(",")] if line else []
    return {"name": f[0] if f else None, "power_limit": f[1] if len(f) > 1 else None, "sm_clock_max": f[2] if len(f) > 2 else None}


def run_workload(name, seconds):
    import torch
    ctx = ws.Context(0)
    cloud, W, H, _ = bench.make_workload(name)
    orbit = ws.synth.orbit_views(36)                  # orbit views for every workload (bench.py's cfg1 uses one fixed camera)
    gen = ws.GenericGaussianPointCloud(cloud["gaussians"], cloud["sh_coefs"], cloud["sh_deg"], cloud["num_points"],
                                       ws.Aabb(cloud["aabb_min"], cloud["aabb_max"]), cloud["center"],
                                       compressed=cloud["compressed"], covars=cloud.get("covars"), quantization=cloud.get("quantization"))
    pc = ws.PointCloud.new(ctx, gen)
    n = cloud["num_points"]
    fmt = ws.FORMAT_RGBA16_FLOAT

    def renderer(pair_cap, timing=False):
        r = ws.GaussianRenderer.new(ctx, fmt, cloud["sh_deg"], cloud["compressed"])
        r.set_pair_capacity(pair_cap)
        r.set_timing(timing)
        return r

    single_cap = min(max(8 * n, 1 << 22), (1 << 30) - 1)           # bench.py's pair capacity
    singles = [renderer(single_cap) for _ in range(DEPTH)]
    streams = [torch.cuda.Stream() for _ in range(DEPTH)]
    s_targets = [torch.empty((H, W, 4), dtype=torch.float16, device="cuda") for _ in range(DEPTH)]
    out = {"workload": name, "num_points": n, "width": W, "height": H, "format": "RGBA16F",
           "single_frames_in_flight": DEPTH, "per_k": []}
    for K in KS:
        args = [bench.frame_args(ws, cloud, orbit[(36 * j) // K], W, H) for j in range(K)]
        rb = renderer(0)                                             # automatic: K x max(8 N, 4 Mi)
        bstream = torch.cuda.Stream()
        b_target = torch.empty((K, H, W, 4), dtype=torch.float16, device="cuda")

        def batch():
            rb.prepare_views(bstream, pc, args)
            rb.render_views(b_target, pc, stream=bstream)

        def single(i):
            k = i % DEPTH
            singles[k].prepare(streams[k], pc, args[i % K])
            singles[k].render(s_targets[k], pc, stream=streams[k])

        # CRCs of every view from both paths
        batch(); torch.cuda.synchronize()
        crc_b = [bench.frame_crc(b_target[v].cpu().numpy()) for v in range(K)]
        crc_s = []
        for v in range(K):
            singles[0].prepare(streams[0], pc, args[v]); singles[0].render(s_targets[0], pc, stream=streams[0])
            torch.cuda.synchronize()
            crc_s.append(bench.frame_crc(s_targets[0].cpu().numpy()))
        # per-stage times of one batch
        rt = renderer(0, timing=True)
        rt.prepare_views(None, pc, args); rt.render_views(b_target, pc); torch.cuda.synchronize()
        rt.prepare_views(None, pc, args); rt.render_views(b_target, pc)
        st = rt.stats()
        stages = {k: round(st[k], 4) for k in ("ms_preprocess", "ms_depth_sort", "ms_binning", "ms_tile_sort", "ms_blend")}
        counts = rt.views_num_visible_points()
        rt.close()

        cur = torch.cuda.current_stream()

        def timed(fn, iters, streams_used):
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            torch.cuda.synchronize()
            e0.record(cur)
            for s_ in streams_used:
                s_.wait_event(e0)
            for i in range(iters):
                fn(i)
            for s_ in streams_used:
                cur.wait_stream(s_)
            e1.record(cur)
            e1.synchronize()
            return e0.elapsed_time(e1) / 1e3

        run_b = lambda i: batch()                                    # noqa: E731
        # warm-up, then size the windows: 4 alternating windows per path, about `seconds` of GPU time per path
        timed(run_b, 5, [bstream]); timed(single, 5 * K, streams)
        tb = timed(run_b, 10, [bstream]) / 10
        ts = timed(single, 10 * K, streams) / (10 * K)
        ib = max(3, int(seconds / 4 / tb))
        i_s = max(3 * K, int(seconds / 4 / ts))
        sec_b = sec_s = 0.0
        views_b = views_s = 0
        for _ in range(4):
            sec_s += timed(single, i_s, streams); views_s += i_s
            sec_b += timed(run_b, ib, [bstream]); views_b += ib * K
        out["per_k"].append({
            "K": K, "views_per_s_batch": round(views_b / sec_b, 1), "views_per_s_single": round(views_s / sec_s, 1),
            "speedup": round((views_b / sec_b) / (views_s / sec_s), 3), "gpu_s_batch": round(sec_b, 3), "gpu_s_single": round(sec_s, 3),
            "crc_batch": crc_b, "crc_single": crc_s, "crc_match": crc_b == crc_s,
            "visible_per_view": counts, "occlusion_split": K * n >= 2_000_000,
            "num_pairs": st["num_pairs"], "batch_stage_ms": stages})
        rb.close()
        del b_target
    return out


def main():
    ap = argparse.ArgumentParser(description=__doc__.splitlines()[0])
    ap.add_argument("--workloads", default="cfg1,cfg2,cfg3,cfg4")
    ap.add_argument("--seconds", type=float, default=1.0, help="GPU time per path and K, in 4 alternating windows")
    opt = ap.parse_args()
    import torch
    if not torch.cuda.is_available():
        raise SystemExit("bench_views.py: no CUDA device -- the product path has no CPU fallback")
    dev = device_info()
    for name in opt.workloads.split(","):
        line = run_workload(name, opt.seconds)
        line["device"] = dev
        print(json.dumps(line), flush=True)


if __name__ == "__main__":
    main()
