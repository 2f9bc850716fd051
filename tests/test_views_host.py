"""Batches of views, the parts that need no GPU: the C++ mirror of the batch API compiles cleanly, and the dataset
renderer groups cameras into batches the way it documents."""
import os
import subprocess

ROOT = os.path.join(os.path.dirname(os.path.abspath(__file__)), "..")


def test_cpp_batch_methods_compile(tmp_path):
    inc = os.path.join(ROOT, "include")
    cpp = tmp_path / "t.cpp"
    cpp.write_text('''#include "websplat_b200.hpp"
static_assert(WS_MAX_VIEWS == 8, "views per batch");
void frame(ws::GaussianRenderer &r, const ws::PointCloud &pc, void *stream, void *dev, void *host)
{
    std::vector<ws::SplattingArgs> views(3);
    r.prepare_views(stream, pc, views);
    const size_t pitch = 64 * 16, stride = 48 * pitch;
    r.render_views(stream, pc, dev, pitch, stride, {0.0, 0.0, 0.0, 1.0});
    r.render_views_to_host(stream, pc, host, pitch, stride, {0.0, 0.0, 0.0, 1.0});
    std::vector<uint32_t> v = r.views_num_visible_points();
    (void)v;
}
int main() { return 0; }
''')
    gxx = "/usr/bin/g++" if os.path.exists("/usr/bin/g++") else "g++"
    p = subprocess.run([gxx, "-std=c++17", "-Wall", "-Wextra", "-Werror", "-fsyntax-only", "-I", inc, str(cpp)], capture_output=True, text=True)
    assert p.returncode == 0, p.stderr


def test_scene_batches_group_consecutive_cameras_of_one_resolution(ws):
    def cam(i, w, h):
        return ws.SceneCamera(i, "c%d" % i, w, h, [0, 0, 0], [[1, 0, 0], [0, 1, 0], [0, 0, 1]], 500.0, 500.0)
    # 1920 wide renders at 1600 x 899, as does 3200 x 1798: both land in one group
    cams = [cam(0, 320, 200), cam(1, 320, 200), cam(2, 320, 200), cam(3, 640, 400), cam(4, 320, 200),
            cam(5, 1920, 1080), cam(6, 3200, 1798), cam(7, 320, 200)]
    got = [(i0, [c.id for c in cs]) for i0, cs in ws.scene._batches(cams, 2)]
    assert got == [(0, [0, 1]), (2, [2]), (3, [3]), (4, [4]), (5, [5, 6]), (7, [7])]
    assert [len(cs) for _, cs in ws.scene._batches(cams, 8)] == [3, 1, 1, 2, 1]
    assert [len(cs) for _, cs in ws.scene._batches(cams, 1)] == [1] * 8
