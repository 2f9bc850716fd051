#!/usr/bin/env python
"""bench.py -- frames/s of the splat render hot path (preprocess | sort | blend).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--workload cfg3] [--dump-outputs DIR]

A "step" is one frame: GaussianRenderer.prepare + render of one camera of the 36-view orbit
(BASELINE.md section 3) over a synthetic cloud that is already resident in HBM (PointCloud::new is
load-time in the reference too, pointcloud.rs:99).  Default workload = cfg3, the configuration
BASELINE.json's metric and target are quoted on: 6M Gaussians, 1920x1080, SH degree 3, 1xB200.

  value  frames/s over exactly K frames, CUDA events on the launching stream, frame written to a
         device target (inputs resident; the 744 MB cloud is ~6x the 126 MB L2, so nothing
         survives in L2 between frames)
  e2e    the same K frames through the public API with HOST buffers: per frame the camera/settings
         uniforms go host->device and the finished RGBA16F frame comes back into pinned host memory
  roofline / kernels   per-kernel CUDA-event times of the same frames vs algorithmic HBM bytes
  cpu_baseline         the CPU oracle (port of the reference algorithm; the reference itself is
                       Rust+WGSL on wgpu/Vulkan and cannot run here) timed on one frame

--impl reference runs that CPU oracle as the reference arm (oracle/_ref cannot be built).

--dump-outputs DIR writes, after the timed steps, the frame of the last timed step (single-GPU arm or reference arm)
as DIR/image.npy, float32 [H, W, 4].  A frame larger than DUMP_PIXELS pixels is written as a fixed, seeded sample
of DUMP_PIXELS pixels, image.npy [DUMP_PIXELS, 4], with their row-major pixel indices in DIR/image_pixel_index.npy
(float64).  The inputs are seeded, so two builds run with the same arguments can be compared output for output.
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

import numpy as np  # noqa: E402

METRIC = "frames/sec"
REFERENCE_BUDGET_S = 120.0                  # host seconds the reference arm may spend on timed frames
KERNELS_STAGE1 = 3                          # count, scan, preprocess
KERNELS_BINNING = 3                         # count, scan, expand (per slab; the tile ranges are fused into the last onesweep pass)
DUMP_PIXELS = 1 << 21                       # --dump-outputs: a 1920x1080 frame (33 MB as f32) is written whole, larger
                                            # frames as this many sampled pixels (32 MB + 16 MB of indices)


# the HBM bandwidth every roofline fraction is priced at: device-to-device copy bandwidth, median of 7 runs of 20 copies
# of 4 GiB (torch copy_, CUDA events) on an NVIDIA B200 at a 1000 W power limit, 1965 MHz max SM clock.  Part of the
# source so that every checkout prices alike (the round-1/2 numbers in DESIGN.md and profiles/ used 6570.9 GB/s, an
# earlier per-machine measurement).
HBM_PEAK_GBS = 6655.0
SM_MAX_MHZ = 1965.0


def measured_peaks():
    return HBM_PEAK_GBS, "measured D2D copy bandwidth, NVIDIA B200 at 1000 W (bench.py HBM_PEAK_GBS)", SM_MAX_MHZ


class ClockSampler(threading.Thread):
    """SM clock + throttle reasons during the timed region (B200_PROFILING.md recipe), sampled through
    NVML every 10 ms (the nvidia-smi CLI takes ~100 ms per query, longer than a whole timed region)."""

    def __init__(self, index):
        super().__init__(daemon=True)
        self.index, self.rows, self._halt = index, [], threading.Event()
        self.nv = None
        try:
            import pynvml
            pynvml.nvmlInit()
            self.nv = pynvml
            self.h = pynvml.nvmlDeviceGetHandleByIndex(index)
            self.maxclk = pynvml.nvmlDeviceGetMaxClockInfo(self.h, pynvml.NVML_CLOCK_SM)
        except Exception:
            self.nv = None

    def run(self):
        nv = self.nv
        while not self._halt.is_set():
            try:
                if nv is not None:
                    clk = nv.nvmlDeviceGetClockInfo(self.h, nv.NVML_CLOCK_SM)
                    try:
                        rs = nv.nvmlDeviceGetCurrentClocksEventReasons(self.h)
                    except Exception:
                        rs = nv.nvmlDeviceGetCurrentClocksThrottleReasons(self.h)
                    util = nv.nvmlDeviceGetUtilizationRates(self.h).gpu
                    self.rows.append((float(clk), int(rs), int(util)))
                else:
                    out = subprocess.run(["nvidia-smi", "-i", str(self.index), "--query-gpu=clocks.sm,clocks.max.sm",
                                          "--format=csv,noheader,nounits"], capture_output=True, text=True, timeout=5).stdout
                    c = [float(x) for x in out.strip().split(",")]
                    self.maxclk = c[1]
                    self.rows.append((c[0], 0, 100))
            except Exception:
                pass
            self._halt.wait(0.01)

    def reset(self):
        """forget the samples taken so far (the sampler is started BEFORE the barrier in front of a timed region -- its NVML
        initialisation costs milliseconds on the one rank that runs it, which every other rank of a multi-GPU run would
        otherwise spend waiting inside ITS timed region -- and reset right at the region's start)"""
        self.rows = []

    def finish(self):
        self._halt.set()
        self.join(timeout=6)
        bits = {"hw_slowdown": 0x8, "sw_power_cap": 0x4, "sw_thermal_slowdown": 0x20, "hw_thermal_slowdown": 0x40,
                "hw_power_brake_slowdown": 0x80}
        sm = [r[0] for r in self.rows]
        reasons = sorted(k for k, b in bits.items() if any(r[1] & b for r in self.rows))
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": float(getattr(self, "maxclk", 0) or 0) or None,
                "reasons": reasons, "samples": len(sm)}


def frame_crc(host):
    """CRC-32 of EVERY byte of a downloaded frame (pinned host tensor or numpy array): the parity evidence the bench
    lines carry -- the same view must give the same value at 1, 2, 4 and 8 GPUs and with the occlusion split on or off."""
    import zlib
    a = host if isinstance(host, np.ndarray) else host.view(__import__("torch").uint8).numpy()
    return "%08x" % (zlib.crc32(a.tobytes()) & 0xffffffff)


def dump_outputs(path, image):
    """--dump-outputs: the frame as float32 [H, W, 4], or a fixed seeded sample of DUMP_PIXELS of its pixels"""
    img = np.asarray(image, dtype=np.float32)
    H, W, C = img.shape
    os.makedirs(path, exist_ok=True)
    if H * W > DUMP_PIXELS:
        idx = np.sort(np.random.default_rng(0).choice(H * W, size=DUMP_PIXELS, replace=False))
        img = img.reshape(H * W, C)[idx]
        np.save(os.path.join(path, "image_pixel_index.npy"), idx.astype(np.float64))
    np.save(os.path.join(path, "image.npy"), img)


CHECKSUM_VIEW = 0                           # index into the workload's camera list


def host_threads():
    """host cores this process may use (affinity / cgroup aware); the oracle legs set their OpenMP count from it --
    torchrun exports OMP_NUM_THREADS=1 to every rank, which would otherwise shrink the reference arm to one core"""
    try:
        return len(os.sched_getaffinity(0))
    except Exception:
        return os.cpu_count() or 1


def make_workload(name):
    import hashlib
    import tempfile
    import websplat_b200 as ws
    n, W, H, seed, compressed = ws.synth.CONFIGS[name]
    # generating cfg3 takes ~15 s of host time, so the cloud is cached in the temporary directory; the file name carries a
    # hash of the generator, so a cloud made by another version of synth.py is never picked up
    with open(ws.synth.__file__, "rb") as f:
        gen_hash = hashlib.sha1(f.read()).hexdigest()[:12]
    cache = os.path.join(tempfile.gettempdir(), "ws_cloud_%s_%s.npz" % (name, gen_hash))
    cloud = None
    if os.path.exists(cache):
        try:
            z = np.load(cache)
            cloud = {k: z[k] for k in z.files}
            cloud["gaussians"] = cloud["gaussians"].view(ws.synth.GAUSSIAN_COMPRESSED_DTYPE if compressed else ws.synth.GAUSSIAN_DTYPE).reshape(-1)
            for k in ("num_points", "sh_deg"):
                cloud[k] = int(cloud[k])
            cloud["compressed"] = bool(cloud["compressed"])
        except Exception:
            cloud = None
    if cloud is None:
        cloud = ws.synth.make_cloud_compressed(n, seed) if compressed else ws.synth.make_cloud(n, seed)
        if not compressed:
            try:
                np.savez(cache, **{k: (v.view(np.uint8) if k == "gaussians" else v) for k, v in cloud.items()})
            except Exception:
                pass
    views = [ws.synth.fixed_camera()] if name == "cfg1" else ws.synth.orbit_views(36)
    return cloud, W, H, views


def frame_args(ws, cloud, view, W, H):
    pos, rot = view
    fovx, fovy = ws.synth.fov_for_viewport(W, H)
    cam = ws.PerspectiveCamera(pos, rot, ws.PerspectiveProjection(fovx, fovy, 0.1, 100.0))
    cam.fit_near_far(ws.Aabb(cloud["aabb_min"], cloud["aabb_max"]))
    return ws.SplattingArgs(cam, (W, H))          # bin/render.rs:92-104: scaling 1, sh 3, transparent bg


def oracle_frame_seconds(cloud, view, W, H, repeats=1):
    """One full frame of the CPU oracle (stage 1 -> stable u32 sort -> back-to-front composite): (seconds, threads, image)."""
    import websplat_b200 as ws
    from oracle import oracle as orc
    orc.set_num_threads(host_threads())
    fovx, fovy = ws.synth.fov_for_viewport(W, H)
    best = None
    for _ in range(repeats):
        t0 = time.perf_counter()
        image = orc.render_frame(cloud, view[0], view[1], W, H, fovx, fovy)["image"]
        dt = time.perf_counter() - t0
        best = dt if best is None else min(best, dt)
    return best, orc.num_threads(), image


def run_reference(args):
    """Reference arm: the reference's algorithm on the host cores (CPU oracle port)."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return 0
    cloud, W, H, views = make_workload(args.workload)
    from oracle import oracle as orc
    orc.build()
    orc.set_num_threads(host_threads())
    # The driver launches this arm with the GPU arm's --steps / --warmup (hundreds of steps); a CPU frame of cfg3 takes
    # seconds.  The sample is therefore bounded: at most 3 warm-up frames, then as many FULL frames of the orbit as fit
    # REFERENCE_BUDGET_S (never fewer than 1, never more than --steps); `steps` reports the frames actually timed.
    t_frame = None
    for i in range(min(args.warmup, 3)):
        t1 = time.perf_counter()
        oracle_frame_seconds(cloud, views[i % len(views)], W, H)
        t_frame = time.perf_counter() - t1
    if t_frame is None:
        t1 = time.perf_counter()
        oracle_frame_seconds(cloud, views[0], W, H)
        t_frame = time.perf_counter() - t1
    timed = max(1, min(args.steps, int(REFERENCE_BUDGET_S / max(t_frame, 1e-6))))
    requested = args.steps
    args.steps = timed
    t0 = time.perf_counter()
    for i in range(args.steps):
        _, _, image = oracle_frame_seconds(cloud, views[i % len(views)], W, H)
    dt = time.perf_counter() - t0
    if args.dump_outputs:
        dump_outputs(args.dump_outputs, image)
    fps = args.steps / dt
    cores = orc.num_threads()
    line = {
        "impl": "reference", "metric": METRIC, "value": fps, "unit": "frames/s", "n_gpus": args.gpus,
        "steps": args.steps, "warmup": max(1, min(args.warmup, 3)), "ms_per_step": 1e3 * dt / args.steps, "higher_is_better": True,
        "scaling": "strong", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": {"workload": workload_name(args.workload, cloud, W, H), "views": len(views),
                   "steps_requested": requested, "warmup_requested": args.warmup},
        "cpu_baseline": {"value": fps, "unit": "frames/s", "cores": cores, "kind": "port",
                         "sample": "%d full frames of the same workload on the CPU oracle (OpenMP, %d threads; %d steps were requested, "
                                   "the sample is bounded to ~%d s of host time); the reference itself (Rust+WGSL on wgpu/Vulkan) "
                                   "cannot be built or run on this box" % (args.steps, cores, requested, int(REFERENCE_BUDGET_S))},
        "e2e": {"value": fps, "unit": "frames/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(line))
    return 0


def workload_name(name, cloud, W, H):
    return "%s: %d synthetic Gaussians (%s layout, SH deg %d), %dx%d, 36-view orbit" % (
        name, cloud["num_points"], "npz-compressed" if cloud["compressed"] else "raw f16", cloud["sh_deg"], W, H)


def run_ours(args):
    import torch
    import websplat_b200 as ws
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if world > 1:
        import bench_multi          # multi-GPU path lives next to this file
        return bench_multi.run(args)
    if args.gpus > 1:               # launched without torchrun: start one process per GPU ourselves
        cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node", str(args.gpus),
               "--master-addr", "127.0.0.1", "--master-port", "29533", os.path.abspath(__file__)] + sys.argv[1:]
        return subprocess.call(cmd)
    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device -- the product path has no CPU fallback")
    torch.cuda.set_device(local)
    ctx = ws.Context(local)
    cloud, W, H, views = make_workload(args.workload)
    fmt = ws.FORMAT_RGBA16_FLOAT
    gen = ws.GenericGaussianPointCloud(cloud["gaussians"], cloud["sh_coefs"], cloud["sh_deg"], cloud["num_points"],
                                       ws.Aabb(cloud["aabb_min"], cloud["aabb_max"]), cloud["center"],
                                       compressed=cloud["compressed"], covars=cloud.get("covars"),
                                       quantization=cloud.get("quantization"))
    pc = ws.PointCloud.new(ctx, gen)
    # `depth` frames in flight: one renderer (own scratch) + one stream + one target per frame slot, all reading the
    # same resident cloud; frame i runs in slot i % depth.  At the small configurations one frame's kernels are
    # latency-bound and a second frame fills the idle SMs (cfg1 +36 %, cfg2 +22 %, cfg3 +2 %: profiles/r01o_*).
    depth = int(args.frames_in_flight) if args.frames_in_flight > 0 else 2
    split_req = False if args.no_occlusion_split else None        # None = the library's automatic choice (on from 2 M points)
    split = (not args.no_occlusion_split) and cloud["num_points"] >= 2_000_000
    pair_cap = min(max(8 * cloud["num_points"], 1 << 22), (1 << 30) - 1)
    rs = []
    for _ in range(depth):
        r_ = ws.GaussianRenderer.new(ctx, fmt, cloud["sh_deg"], cloud["compressed"])
        r_.set_pair_capacity(pair_cap)
        r_.set_timing(False)
        r_.set_occlusion_split(split_req)
        rs.append(r_)
    r = rs[0]                                  # slot 0 also serves the per-stage breakdown below
    fargs = [frame_args(ws, cloud, v, W, H) for v in views]
    streams = [torch.cuda.Stream() for _ in range(depth)]
    stream = streams[0]
    targets = [torch.empty((H, W, 4), dtype=torch.float16, device="cuda") for _ in range(2 * depth)]
    target = targets[0]
    host = [torch.empty((H, W, 4), dtype=torch.float16).pin_memory() for _ in range(2 * depth)]
    K, Wu = args.steps, max(args.warmup, 3)

    def frame(i, to_host=None):
        k = i % depth
        rs[k].prepare(streams[k], pc, fargs[i % len(fargs)])
        if to_host is None:
            rs[k].render(targets[k], pc, stream=streams[k])
        else:
            rs[k].render_to_host(to_host, pc, stream=streams[k])

    # ---- kernel-only: inputs resident, frame stays on the device --------------------------------
    for i in range(depth * ((Wu + depth - 1) // depth)):
        frame(i)
    torch.cuda.synchronize()
    st0 = r.stats()
    sampler = ClockSampler(local); sampler.start()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    torch.cuda.synchronize()
    cur = torch.cuda.current_stream()
    e0.record(cur)
    for st_ in streams:
        st_.wait_event(e0)
    for i in range(K):
        frame(Wu + i)
    for st_ in streams:
        cur.wait_stream(st_)
    e1.record(cur)
    torch.cuda.synchronize()
    ms_total = e0.elapsed_time(e1)
    clocks = sampler.finish()
    fps = K / (ms_total * 1e-3)
    # the frame of the last timed step, taken before the e2e section below reuses the targets
    last_frame = targets[(Wu + K - 1) % depth].cpu().numpy() if args.dump_outputs else None

    # ---- e2e: host buffers, uniforms H2D + frame D2H inside the timed region ----------------------
    # The public API is asynchronous on the caller's stream, so a caller that wants throughput keeps
    # two device targets per frame slot and downloads frame i on a copy stream while later frames are being
    # rendered (bin/measure.rs also submits all frames and waits once, measure.rs:98-147).  Every frame
    # still lands in pinned host memory inside the timed region.
    copy_stream = torch.cuda.Stream()
    nb = 2 * depth
    rendered = [torch.cuda.Event() for _ in range(nb)]
    copied = [torch.cuda.Event() for _ in range(nb)]

    def frame_e2e(i):
        k, b = i % depth, i % nb                            # slot, buffer (two buffers per slot)
        streams[k].wait_event(copied[b])                   # target b is free again (its download finished)
        rs[k].prepare(streams[k], pc, fargs[i % len(fargs)])
        rs[k].render(targets[b], pc, stream=streams[k])
        rendered[b].record(streams[k])
        copy_stream.wait_event(rendered[b])
        with torch.cuda.stream(copy_stream):
            host[b].copy_(targets[b], non_blocking=True)
            copied[b].record(copy_stream)

    for b in range(nb):
        copied[b].record(copy_stream)
    for i in range(nb * ((Wu + nb - 1) // nb)):
        frame_e2e(i)
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    for i in range(K):
        frame_e2e(Wu + i)
    torch.cuda.synchronize()
    e2e_s = time.perf_counter() - t0
    e2e_fps = K / e2e_s

    # ---- parity evidence in the line: CRC-32 of the full downloaded frame of one fixed view, rendered through the
    #      product default (occlusion split automatic) and through a renderer with the split off; the multi-GPU arm
    #      prints the CRC of the same view, so identical values across the N = 1, 2, 4, 8 lines mean identical frames
    cview = fargs[CHECKSUM_VIEW % len(fargs)]
    rs[0].prepare(streams[0], pc, cview)
    rs[0].render_to_host(host[0], pc, stream=streams[0])
    torch.cuda.synchronize()
    checksum = frame_crc(host[0])
    r_off = ws.GaussianRenderer.new(ctx, fmt, cloud["sh_deg"], cloud["compressed"])
    r_off.set_pair_capacity(pair_cap)
    r_off.set_timing(False)
    r_off.set_occlusion_split(False)
    r_off.prepare(streams[0], pc, cview)
    r_off.render_to_host(host[1], pc, stream=streams[0])
    torch.cuda.synchronize()
    checksum_off = frame_crc(host[1])
    # the complete pair list (what a one-pass frame sorts and stages) over the timed views: prices `frac_full_pairs`
    p_full = []
    for i in range(min(K, len(fargs))):
        r_off.prepare(streams[0], pc, fargs[(Wu + i) % len(fargs)])
        p_full.append(r_off.stats()["num_pairs"])
    P_full = float(np.mean(p_full))
    del r_off

    # ---- per-stage CUDA-event breakdown over the same views (timing on: 8 event records per frame)
    r.set_timing(True)
    acc = {}
    counts = {"V": [], "P": []}
    for i in range(K):
        r.prepare(stream, pc, fargs[(Wu + i) % len(fargs)])
        r.render(target, pc, stream=stream)
        s = r.stats()
        for k_ in ("ms_preprocess", "ms_sort", "ms_blend", "ms_depth_sort", "ms_binning", "ms_tile_sort", "ms_ranges",
                   "bytes_preprocess", "bytes_sort", "bytes_blend"):
            acc[k_] = acc.get(k_, 0.0) + float(s[k_])
        counts["V"].append(s["num_visible"]); counts["P"].append(s["num_pairs"])
    for k_ in acc:
        acc[k_] /= K
    V, P = float(np.mean(counts["V"])), float(np.mean(counts["P"]))
    N = cloud["num_points"]
    T = ((W + 15) // 16) * ((H + 15) // 16)
    depth_passes = 4
    tile_passes = 3 if T > 65536 else (2 if T > 256 else 1)
    peak, peak_src, sm_max = measured_peaks()

    def gbs(nbytes, ms):
        return nbytes / (ms * 1e-3) / 1e9 if ms > 0 else 0.0

    bpp = 8                                            # rgba16float
    # algorithmic bytes per SURVEY.md 8(d), nothing else: in particular NOT the occlusion split's own state round trip
    # (W*H*32 B) nor the far slab's second sweep over slots + rectangles -- those are costs of this design, not work
    # the path requires.  P = pairs actually emitted; `frac_full_pairs` prices the same time at the complete pair list.
    kernels = {
        "preprocess": {"ms": acc["ms_preprocess"], "bytes": acc["bytes_preprocess"]},
        "depth_sort_pass": {"ms": acc["ms_depth_sort"] / depth_passes, "bytes": V * 16, "launches": depth_passes},
        "binning": {"ms": acc["ms_binning"], "bytes": V * 12 + P * 8, "bytes_full_pairs": V * 12 + P_full * 8},
        "tile_sort_pass": {"ms": acc["ms_tile_sort"] / tile_passes, "bytes": P * 16, "bytes_full_pairs": P_full * 16, "launches": tile_passes},
        "composite": {"ms": acc["ms_blend"], "bytes": P * 24 + T * 8 + W * H * bpp, "bytes_full_pairs": P_full * 24 + T * 8 + W * H * bpp},
    }
    for kv in kernels.values():
        kv["gbs"] = gbs(kv["bytes"], kv["ms"]); kv["frac"] = kv["gbs"] / peak
        if "bytes_full_pairs" in kv:
            kv["frac_full_pairs"] = gbs(kv["bytes_full_pairs"], kv["ms"]) / peak
    sb_bytes = depth_passes * V * 16 + V * 12 + P * 8 + tile_passes * P * 16 + T * 8 + P * 24 + T * 8 + W * H * bpp
    sb_bytes_full = depth_passes * V * 16 + V * 12 + P_full * 8 + tile_passes * P_full * 16 + T * 8 + P_full * 24 + T * 8 + W * H * bpp
    dom = max(kernels, key=lambda k_: kernels[k_]["ms"] * kernels[k_].get("launches", 1))
    # DRAM traffic of the dominant kernel (same unit of work as its `bytes`) from the committed ncu --set full captures (cfg3 only)
    traffic, traffic_src = None, None
    try:
        if args.workload == "cfg3" and split:
            tj = json.load(open(os.path.join(ROOT, "profiles", "kernel_traffic_cfg3_split.json")))
            traffic = tj["per_stage"][dom]["dram_bytes"]
            traffic_src = "profiles/kernel_traffic_cfg3_split.json (%s; %s)" % (tj.get("source", "ncu --set full"), tj["per_stage"][dom]["launches"])
        elif args.workload == "cfg3":
            tj = json.load(open(os.path.join(ROOT, "profiles", "kernel_traffic_cfg3.json")))
            key = {"composite": "composite_kernel<1>", "preprocess": "preprocess_kernel<0>", "binning": "bin_expand_kernel",
                   "tile_sort_pass": "onesweep_pass_kernel<1>", "depth_sort_pass": "onesweep_pass_kernel<0>"}[dom]
            traffic = tj[key]["dram_bytes_per_launch"]
            traffic_src = "profiles/kernel_traffic_cfg3.json (ncu --set full, r01m, one-pass frame)"
    except Exception:
        traffic = None
    # measured issue / pipe utilisation of the compositor (ncu capture committed under profiles/; None until one exists)
    pipes, pipes_src = None, None
    try:
        pj = json.load(open(os.path.join(ROOT, "profiles", "composite_pipes_%s.json" % args.workload)))
        pipes, pipes_src = pj.get("metrics"), pj.get("source")
    except Exception:
        pass
    sb_ms = acc["ms_sort"] + acc["ms_blend"]
    roofline = {
        "kernel": dom, "bound": "hbm", "achieved": kernels[dom]["gbs"], "peak": peak, "unit": "GB/s",
        "frac": kernels[dom]["frac"], "frac_full_pairs": kernels[dom].get("frac_full_pairs"),
        "traffic": traffic, "traffic_source": traffic_src, "peak_source": peak_src,
        "bytes_formula": "SURVEY.md 8(d): blend = P*(4+20) + T*8 + W*H*B_fmt with P = pairs emitted; no state round trip",
        "note": "stage 3 is FP32/MUFU-issue bound, not HBM bound (SURVEY 8(d)); its HBM fraction is reported because "
                "the north star asks for it; 'composite_pipes' holds the measured issue / pipe utilisation (ncu). `frac` prices the "
                "pairs actually EMITTED (%.1f M of the %.1f M of the complete list: the occlusion split drops the rest before they "
                "are sorted), so it falls when the split removes bytes faster than time; `frac_full_pairs` prices the same time at "
                "the complete pair list" % (P / 1e6, P_full / 1e6),
        "sort_plus_blend": {"bytes": sb_bytes, "ms": sb_ms, "gbs": gbs(sb_bytes, sb_ms), "frac": gbs(sb_bytes, sb_ms) / peak,
                            "frac_full_pairs": gbs(sb_bytes_full, sb_ms) / peak},
        "composite_pipes": pipes, "composite_pipes_source": pipes_src,
    }

    # ---- extra lines (not the headline): the reference's `measure` protocol and the CUB yard-stick ---------------
    extra = {}
    if not args.no_extra:
        # bin/measure.rs:34,98,147-153,184: 2048 x 2048, Rgba8Unorm, ONE renderer, 10 samples per camera submitted back
        # to back, one wait at the end, wall clock (the reference's timer also includes its lazy-init frame; here it does not)
        try:
            MW = MH = 2048
            rm = ws.GaussianRenderer.new(ctx, ws.FORMAT_RGBA8_UNORM, cloud["sh_deg"], cloud["compressed"])
            rm.set_pair_capacity(pair_cap); rm.set_timing(False)
            margs = [frame_args(ws, cloud, v, MW, MH) for v in views]
            mt = torch.empty((MH, MW, 4), dtype=torch.uint8, device="cuda")
            for a_ in margs[:3]:
                rm.prepare(stream, pc, a_); rm.render(mt, pc, stream=stream)
            torch.cuda.synchronize()
            samples = 10 if K >= 100 else 1
            tm = time.perf_counter()
            for a_ in margs:
                for _ in range(samples):
                    rm.prepare(stream, pc, a_); rm.render(mt, pc, stream=stream)
            torch.cuda.synchronize()
            dtm = time.perf_counter() - tm
            extra["measure_equivalent"] = {"frames_per_s": len(margs) * samples / dtm, "viewport": [MW, MH], "target_format": "rgba8unorm",
                                           "cameras": len(margs), "samples_per_camera": samples, "frames_in_flight": 1,
                                           "protocol": "bin/measure.rs:34,98,147-153,184 (wall clock, one final wait)"}
            del rm, mt
        except Exception as e:                         # never lose the headline to an extra
            extra["measure_equivalent"] = {"error": str(e)[:200]}
        try:
            extra["sort_vs_cub"] = json.load(open(os.path.join(ROOT, "profiles", "r02_sort_vs_cub.json")))
        except Exception:
            pass

    # ---- CPU baseline: one frame of the same workload on the host cores -------------------------
    cpu = None
    if not args.no_cpu_baseline:
        secs, cores, _ = oracle_frame_seconds(cloud, views[0], W, H)
        cpu = {"value": 1.0 / secs, "unit": "frames/s", "cores": cores, "kind": "port",
               "sample": "1 full frame (view 0) of the same workload on the CPU oracle: %.2f s" % secs}

    line = {
        "metric": METRIC, "value": fps, "unit": "frames/s", "n_gpus": 1, "steps": K, "warmup": Wu,
        "ms_per_step": ms_total / K, "higher_is_better": True, "scaling": "strong", "vs_baseline": None,
        "dtype": "f32", "data": "synthetic",
        "config": {"workload": workload_name(args.workload, cloud, W, H), "target_format": "rgba16float",
                   "l2": "inputs (%.0f MB cloud) larger than the 126 MB L2; no flush needed" % ((cloud["gaussians"].nbytes + cloud["sh_coefs"].nbytes) / 1e6),
                   "frames_in_flight": depth,
                   "occlusion_split": ("two depth slabs, the far one culled against the tiles the near one saturated: P_mean counts "
                                       "the pairs actually emitted; the image is bit-identical to the one-pass frame") if split else "off",
                   "N": N, "V_mean": V, "P_mean": P, "tiles": T},
        "ms_per_frame": {"note": "one frame at a time on one stream (CUDA events between the stages)", "preprocess": acc["ms_preprocess"], "sort": acc["ms_sort"], "blend": acc["ms_blend"],
                         "depth_sort": acc["ms_depth_sort"], "binning": acc["ms_binning"],
                         "tile_sort": acc["ms_tile_sort"]},
        "roofline": roofline, "kernels": kernels, "cpu_baseline": cpu,
        "e2e": {"value": e2e_fps, "unit": "frames/s", "h2d_bytes_per_step": 480, "d2h_bytes_per_step": W * H * 8,
                "checksum": checksum, "checksum_what": "CRC-32 of the full RGBA16F frame of view %d" % CHECKSUM_VIEW,
                "checksum_split_off": checksum_off, "checksum_split_identical": checksum == checksum_off},
        "extra": extra,
        # stage 1 + depth passes + per slab (binning + tile passes + compositor); two slabs with the occlusion split
        "gpu_launches": K * (KERNELS_STAGE1 + depth_passes + (2 if split else 1) * (KERNELS_BINNING + tile_passes + 1)),
        "clocks": clocks,
    }
    if args.dump_outputs:
        dump_outputs(args.dump_outputs, last_frame)
    if rank == 0:
        print(json.dumps(line))
    return 0


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=None)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--workload", default="cfg3", choices=["cfg1", "cfg2", "cfg3", "cfg4", "cfg5"])
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-extra", action="store_true", help="skip the `measure`-equivalent line (2048^2, RGBA8) under `extra`")
    ap.add_argument("--frames-in-flight", type=int, default=0,
                    help="frames in flight per GPU (one renderer + stream per frame slot); 0 = auto: 2 on one GPU, 3 on 2-4 GPUs, 4 on 8 GPUs "
                         "(the smaller the per-GPU share, the more latency-bound a single frame is)")
    ap.add_argument("--no-occlusion-split", action="store_true", help="single-GPU arm: bin / tile-sort / composite all pairs in one pass")
    ap.add_argument("--equal-bands", action="store_true", help="multi-GPU arm: keep the equal tile-row split instead of cost-balanced bands")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="after the timed steps, write the frame of the last one as DIR/image.npy (float32; see the module docstring)")
    args = ap.parse_args()
    if args.steps is not None and args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.gpus > 1 and args.impl == "ours":
        ap.error("--dump-outputs is implemented for the single-GPU and reference arms")
    if args.steps is None:
        args.steps = 360 if args.impl == "ours" else 10    # 10 orbits (~1 s of GPU time) / ~2-5 s per CPU frame
    if args.impl == "reference":
        return run_reference(args)
    return run_ours(args)


if __name__ == "__main__":
    sys.exit(main())
