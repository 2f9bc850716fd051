"""Dataset cameras and image output: the callers either side of the render path (SURVEY.md section 8(f) N3).

Mirrors, in the host language of this build:
  SceneCamera / Split / Scene          scene.rs:11-205   (cameras.json as written by the 3DGS trainer)
  focal2fov / fov2focal                camera.rs:236-242
  download_texture's f16 -> u8 pixel conversion and the PNG write     bin/render.rs:187-246
  render_views (the offline dataset renderer's loop)                   bin/render.rs:33-127
"""
import json
import math
import os
import struct
import zlib

import numpy as np


def focal2fov(focal, pixels):
    """camera.rs:236-238 (f32 arithmetic)."""
    return float(np.float32(2.0) * np.arctan(np.float32(pixels) / (np.float32(2.0) * np.float32(focal)), dtype=np.float32))


def fov2focal(fov, pixels):
    """camera.rs:240-242."""
    return float(np.float32(pixels) / (np.float32(2.0) * np.tan(np.float32(fov) * np.float32(0.5), dtype=np.float32)))


TRAIN, TEST = "train", "test"


def _quat_from_cgmath_matrix(M):
    """cgmath 0.18 `Quaternion::from(Matrix3)` in f32; M is the math matrix M[row][col] (cgmath mat[c][r] = M[r][c])."""
    f = np.float32
    m = np.asarray(M, dtype=np.float32)
    trace = f(m[0, 0] + m[1, 1]) + m[2, 2]
    half = f(0.5)
    if trace >= 0:
        s = np.sqrt(f(1.0) + trace, dtype=np.float32)
        w = half * s
        s = half / s
        x, y, z = (m[2, 1] - m[1, 2]) * s, (m[0, 2] - m[2, 0]) * s, (m[1, 0] - m[0, 1]) * s
    elif m[0, 0] > m[1, 1] and m[0, 0] > m[2, 2]:
        s = np.sqrt(f(m[0, 0] - m[1, 1]) - m[2, 2] + f(1.0), dtype=np.float32)
        x = half * s
        s = half / s
        y, z, w = (m[0, 1] + m[1, 0]) * s, (m[2, 0] + m[0, 2]) * s, (m[2, 1] - m[1, 2]) * s
    elif m[1, 1] > m[2, 2]:
        s = np.sqrt(f(m[1, 1] - m[0, 0]) - m[2, 2] + f(1.0), dtype=np.float32)
        y = half * s
        s = half / s
        z, x, w = (m[1, 2] + m[2, 1]) * s, (m[0, 1] + m[1, 0]) * s, (m[0, 2] - m[2, 0]) * s
    else:
        s = np.sqrt(f(m[2, 2] - m[0, 0]) - m[1, 1] + f(1.0), dtype=np.float32)
        z = half * s
        s = half / s
        x, y, w = (m[2, 0] + m[0, 2]) * s, (m[1, 2] + m[2, 1]) * s, (m[1, 0] - m[0, 1]) * s
    return np.array([w, x, y, z], dtype=np.float32)


def _cgmath_matrix_from_quat(q):
    """Matrix3::from(Quaternion), math layout M[row][col]."""
    w, x, y, z = [np.float32(v) for v in q]
    x2, y2, z2 = x + x, y + y, z + z
    xx2, xy2, xz2, yy2, yz2, zz2 = x2 * x, x2 * y, x2 * z, y2 * y, y2 * z, z2 * z
    sy2, sz2, sx2 = y2 * w, z2 * w, x2 * w
    one = np.float32(1.0)
    cols = [[one - yy2 - zz2, xy2 + sz2, xz2 - sy2], [xy2 - sz2, one - xx2 - zz2, yz2 + sx2], [xz2 + sy2, yz2 - sx2, one - xx2 - yy2]]
    return np.array(cols, dtype=np.float32).T


class SceneCamera:
    """scene.rs:11-24.  `rotation` keeps the file's nested lists: each inner list is one cgmath column."""

    def __init__(self, id, img_name, width, height, position, rotation, fx, fy, split=TRAIN):
        self.id, self.img_name, self.width, self.height = int(id), str(img_name), int(width), int(height)
        self.position = np.asarray(position, dtype=np.float32).reshape(3)
        self.rotation = np.asarray(rotation, dtype=np.float32).reshape(3, 3)
        self.fx, self.fy, self.split = float(np.float32(fx)), float(np.float32(fy)), split

    @classmethod
    def from_perspective(cls, ws, cam, name, id, viewport, split=TRAIN):
        """scene.rs:40-61."""
        fx = fov2focal(cam.projection.fovx, viewport[0])
        fy = fov2focal(cam.projection.fovy, viewport[1])
        M = _cgmath_matrix_from_quat(cam.rotation)
        return cls(id, name, viewport[0], viewport[1], cam.position, M.T, fx, fy, split)       # rot.into(): column arrays

    def to_perspective(self, ws):
        """`impl Into<PerspectiveCamera> for SceneCamera`, scene.rs:84-108."""
        fovx = focal2fov(self.fx, self.width)
        fovy = focal2fov(self.fy, self.height)
        M = self.rotation.T.copy()                       # Matrix3::from([[f32;3];3]): inner arrays are columns
        if np.linalg.det(M.astype(np.float64)) < 0:
            M[1, :] = -M[1, :]                           # rot.x[1], rot.y[1], rot.z[1]: row 1 of every column
        vr = np.float32(self.width) / np.float32(self.height)
        fr = np.float32(fovx) / np.float32(fovy)
        proj = ws.PerspectiveProjection(fovx, fovy, 0.01, 100.0, fov2view_ratio=float(vr / fr))     # camera.rs:115-131
        return ws.PerspectiveCamera(self.position, _quat_from_cgmath_matrix(M), proj)

    def to_json(self):
        return dict(id=self.id, img_name=self.img_name, width=self.width, height=self.height,
                    position=[float(v) for v in self.position], rotation=[[float(v) for v in r] for r in self.rotation],
                    fx=self.fx, fy=self.fy)


def _max_distance(points):
    """scene.rs:196-205: the largest pairwise distance (O(n^2) in the reference; same value here)."""
    p = np.asarray(points, dtype=np.float32).reshape(-1, 3)
    best = np.float32(0.0)
    for i in range(len(p) - 1):
        d = p[i + 1:] - p[i]
        best = max(best, np.max(np.sum(d * d, axis=1, dtype=np.float32)))
    return float(np.sqrt(best, dtype=np.float32))


class Scene:
    """scene.rs:110-192."""

    def __init__(self, cameras):
        self._extend = _max_distance([c.position for c in cameras]) if cameras else 0.0
        self._cameras = {}
        for c in cameras:                                 # HashMap::insert: a later duplicate id replaces the earlier one
            self._cameras[c.id] = c

    from_cameras = classmethod(lambda cls, cameras: cls(list(cameras)))

    @classmethod
    def from_json(cls, file):
        """scene.rs:136-150: `file` is a path, a file object or a JSON string; every 8th camera is the test split."""
        if hasattr(file, "read"):
            entries = json.load(file)
        elif isinstance(file, (str, os.PathLike)) and os.path.exists(file):
            with open(file) as f:
                entries = json.load(f)
        else:
            entries = json.loads(file)
        cams = []
        for i, e in enumerate(entries):
            cams.append(SceneCamera(e["id"], e["img_name"], e["width"], e["height"], e["position"], e["rotation"], e["fx"], e["fy"],
                                    TEST if i % 8 == 0 else TRAIN))
        return cls(cams)

    def camera(self, i):
        return self._cameras.get(i)

    def num_cameras(self):
        return len(self._cameras)

    def cameras(self, split=None):
        return sorted((c for c in self._cameras.values() if split is None or c.split == split), key=lambda c: c.id)

    def extend(self):
        return self._extend

    def nearest_camera(self, pos, split=None):
        """scene.rs:180-191: key = (distance^2 * 1e6) as u32 (saturating), first minimum."""
        best, best_key = None, None
        p = np.asarray(pos, dtype=np.float32)
        for c in self._cameras.values():
            if split is not None and c.split != split:
                continue
            d = c.position - p
            key = min(int(np.float32(np.sum(d * d, dtype=np.float32)) * np.float32(1e6)), 0xFFFFFFFF)
            if best_key is None or key < best_key:
                best, best_key = c.id, key
        return best


# ---- image output -------------------------------------------------------------------------------
def frame_to_rgba8(frame_f16):
    """download_texture's conversion (bin/render.rs:234-240): clamp(f16 -> f32, 0, 1) * 255, truncated to u8."""
    f = np.asarray(frame_f16, dtype=np.float16).astype(np.float32)
    f = np.where(np.isnan(f), np.float32(0.0), f)                      # `NaN as u8` is 0 in Rust
    return (np.clip(f, 0.0, 1.0) * np.float32(255.0)).astype(np.uint8)


def png_bytes(rgba8):
    """Minimal RGBA8 PNG encoder (what `image::ImageBuffer::save` produces, up to compression choices)."""
    a = np.ascontiguousarray(rgba8, dtype=np.uint8)
    h, w, ch = a.shape
    assert ch == 4

    def chunk(tag, data):
        return struct.pack(">I", len(data)) + tag + data + struct.pack(">I", zlib.crc32(tag + data) & 0xFFFFFFFF)

    raw = np.concatenate([np.zeros((h, 1), np.uint8), a.reshape(h, w * 4)], axis=1).tobytes()      # filter type 0 per scanline
    return (b"\x89PNG\r\n\x1a\n" + chunk(b"IHDR", struct.pack(">IIBBBBB", w, h, 8, 6, 0, 0, 0))
            + chunk(b"IDAT", zlib.compress(raw, 3)) + chunk(b"IEND", b""))


def decode_png(data):
    """Decoder for the files png_bytes writes (filter 0, RGBA8) -- used by the tests."""
    assert data[:8] == b"\x89PNG\r\n\x1a\n"
    pos, idat, w, h = 8, b"", 0, 0
    while pos < len(data):
        n, tag = struct.unpack(">I4s", data[pos:pos + 8])
        body = data[pos + 8:pos + 8 + n]
        assert struct.unpack(">I", data[pos + 8 + n:pos + 12 + n])[0] == zlib.crc32(tag + body) & 0xFFFFFFFF
        if tag == b"IHDR":
            w, h, depth, ctype = struct.unpack(">IIBB", body[:10])
            assert depth == 8 and ctype == 6
        elif tag == b"IDAT":
            idat += body
        pos += 12 + n
    rows = np.frombuffer(zlib.decompress(idat), np.uint8).reshape(h, 1 + w * 4)
    assert not rows[:, 0].any()
    return rows[:, 1:].reshape(h, w, 4).copy()


def render_resolution(width, height):
    """bin/render.rs:57-63: views wider than 1600 px are scaled down to 1600."""
    if width > 1600:
        s = np.float32(width) / np.float32(1600.0)
        return 1600, int(np.float32(height) / s)
    return int(width), int(height)


def _batches(cameras, batch):
    """Consecutive cameras of equal render resolution, in groups of at most `batch`: [(first index, [cameras])]."""
    groups = []
    for i, s in enumerate(cameras):
        res = render_resolution(s.width, s.height)
        if groups and len(groups[-1][2]) < batch and groups[-1][1] == res:
            groups[-1][2].append(s)
        else:
            groups.append((i, res, [s]))
    return [(i0, cams) for i0, _, cams in groups]


def render_views(ws, ctx, renderer, pc, cameras, img_out, split, on_frame=None, batch=1):
    """bin/render.rs:33-127: renders every camera of one split to `<img_out>/<split>/<index:05>.png`.
    The next view's prepare+render is enqueued while the previous frame is being encoded to PNG.
    batch > 1 renders consecutive cameras of equal resolution together, up to `batch` (<= ws.MAX_VIEWS) per
    prepare_views / render_views; the images are bit-identical to batch = 1."""
    import torch
    out_dir = os.path.join(img_out, split)
    os.makedirs(out_dir, exist_ok=True)
    bbox = pc.bbox()
    paths = []
    if batch > 1:
        for i0, cams in _batches(cameras, batch):
            W, H = render_resolution(cams[0].width, cams[0].height)
            args = []
            for s in cams:
                cam = s.to_perspective(ws)
                cam.fit_near_far(bbox)
                args.append(ws.SplattingArgs(cam, (W, H), gaussian_scaling=1.0, max_sh_deg=pc.sh_deg(), walltime=100.0))
            renderer.prepare_views(None, pc, args)
            host = torch.empty((len(cams), H, W, 4), dtype=torch.float16).pin_memory()
            renderer.render_views_to_host(host, pc, clear=(0.0, 0.0, 0.0, 0.0))
            torch.cuda.synchronize()
            frames = host.numpy()
            for j, s in enumerate(cams):
                if on_frame is not None:
                    on_frame(i0 + j, s, frames[j])
                path = os.path.join(out_dir, "%05d.png" % (i0 + j))
                with open(path, "wb") as f:
                    f.write(png_bytes(frame_to_rgba8(frames[j])))
                paths.append(path)
        return paths
    for i, s in enumerate(cameras):
        W, H = render_resolution(s.width, s.height)
        cam = s.to_perspective(ws)
        cam.fit_near_far(bbox)
        args = ws.SplattingArgs(cam, (W, H), gaussian_scaling=1.0, max_sh_deg=pc.sh_deg(), walltime=100.0)
        renderer.prepare(None, pc, args)
        host = torch.empty((H, W, 4), dtype=torch.float16).pin_memory()
        renderer.render_to_host(host, pc, clear=(0.0, 0.0, 0.0, 0.0))
        torch.cuda.synchronize()
        frame = host.numpy()
        if on_frame is not None:
            on_frame(i, s, frame)
        path = os.path.join(out_dir, "%05d.png" % i)
        with open(path, "wb") as f:
            f.write(png_bytes(frame_to_rgba8(frame)))
        paths.append(path)
    return paths


def load_pointcloud(ws, ctx, path):
    """GenericGaussianPointCloud::load (io/mod.rs:44-61): dispatch on the file's magic bytes."""
    with open(path, "rb") as f:
        data = f.read()
    if data[:3] == b"ply":
        return ws.PointCloud.from_ply(ctx, data)
    if data[:4] == b"PK\x03\x04":
        return ws.PointCloud.from_npz(ctx, data)
    raise ws.WsError(-1, "websplat_b200: invalid argument (status -1): Unknown file format")
