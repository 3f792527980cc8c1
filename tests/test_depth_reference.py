"""The numpy restatement of the depth-image contract (tests/depth_reference.py) against a verbatim
C++ transcription of depth_image_proc's convert<T> plus voxblox's finite filter, known answers,
the cg_depth_camera layout and the synthetic depth renderer.  No GPU needed."""
import ctypes as C
import os
import subprocess
import tempfile

import numpy as np
import pytest

from tests import depth_reference as ref

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


@pytest.fixture(scope="module")
def convert_bin():
    with tempfile.TemporaryDirectory() as d:
        src, exe = os.path.join(d, "convert.cc"), os.path.join(d, "convert")
        with open(src, "w") as f:
            f.write(ref.CONVERT_CC)
        subprocess.check_call(["g++", "-std=c++17", "-O2", "-ffp-contract=off", "-fno-fast-math",
                               src, "-o", exe])
        yield exe, d


def _transcription(convert_bin, depth, color, cam):
    exe, d = convert_bin
    (ro, go, bo), pix = ref.COLOR_LAYOUT[cam["color_encoding"]]
    H, W = depth.shape
    paths = [os.path.join(d, n) for n in ("depth.bin", "color.bin", "out.bin")]
    np.ascontiguousarray(depth).tofile(paths[0])
    np.ascontiguousarray(color, np.uint8).tofile(paths[1])
    args = [exe, str(ref.DEPTH_ENCODINGS.index(cam["depth_encoding"])), str(W), str(H)]
    args += [float(cam[k]).hex() for k in ("fx", "fy", "cx", "cy")]
    args += [str(pix), str(ro), str(go), str(bo)] + paths
    subprocess.check_call(args)
    raw = np.fromfile(paths[2], np.uint8)
    n = int(raw[:8].view(np.uint64)[0])
    rec = raw[8:].reshape(n, 16)
    return rec[:, :12].copy().view(np.float32).reshape(n, 3), rec[:, 12:].copy()


def _random_frame(rng, enc, color_encoding, W=53, H=37):
    """Images with zeros, NaN, +-inf and large values, and intrinsics from ordinary to extreme."""
    if enc == "16UC1":
        depth = rng.integers(0, 65536, (H, W)).astype(np.uint16)
        depth[rng.random((H, W)) < 0.2] = 0
        depth[rng.random((H, W)) < 0.05] = 65535
    else:
        depth = (rng.standard_normal((H, W)) * 3.0).astype(np.float32)
        r = rng.random((H, W))
        depth[r < 0.1] = 0.0
        depth[(r >= 0.1) & (r < 0.15)] = np.nan
        depth[(r >= 0.15) & (r < 0.2)] = np.inf
        depth[(r >= 0.2) & (r < 0.25)] = -np.inf
        depth[(r >= 0.25) & (r < 0.3)] = np.float32(3e38)
        depth[(r >= 0.3) & (r < 0.33)] = np.float32(-1e37)
    pix = ref.COLOR_LAYOUT[color_encoding][1]
    color = rng.integers(0, 256, (H, W, pix)).astype(np.uint8)
    return depth, color


CAMS = [dict(fx=611.16, fy=609.64, cx=323.45, cy=244.94), dict(fx=1.1e-4, fy=3.7e-3, cx=-7.3, cy=18.01),
        dict(fx=3.3e7, fy=0.71, cx=26.123456789, cy=1e6)]


@pytest.mark.parametrize("color_encoding", sorted(ref.COLOR_LAYOUT))
@pytest.mark.parametrize("enc", ref.DEPTH_ENCODINGS)
def test_restatement_matches_transcription(convert_bin, enc, color_encoding):
    rng = np.random.default_rng([ref.DEPTH_ENCODINGS.index(enc), sorted(ref.COLOR_LAYOUT).index(color_encoding)])
    for k, intr in enumerate(CAMS):
        cam = dict(intr, depth_encoding=enc, color_encoding=color_encoding)
        depth, color = _random_frame(rng, enc, color_encoding)
        got_p, got_c = ref.depth_cloud(depth, color, cam)
        exp_p, exp_c = _transcription(convert_bin, depth, color, cam)
        assert got_p.shape == exp_p.shape, (k, got_p.shape, exp_p.shape)
        assert np.array_equal(got_p.view(np.uint32), exp_p.view(np.uint32)), k
        assert np.array_equal(got_c, exp_c), k


@pytest.mark.parametrize("enc", ref.DEPTH_ENCODINGS)
def test_wrong_forms_are_told_apart(convert_bin, enc):
    """Keeping the invalid pixels as NaN points, or rounding x and y once, fails the comparison."""
    rng = np.random.default_rng(7)
    cam = dict(CAMS[0], depth_encoding=enc, color_encoding="rgb8")
    depth, color = _random_frame(rng, enc, "rgb8", W=160, H=120)
    exp_p, _ = _transcription(convert_bin, depth, color, cam)
    nan_p, _ = ref.depth_cloud(depth, color, cam, form="nan")
    assert nan_p.shape != exp_p.shape
    fma_p, _ = ref.depth_cloud(depth, color, cam, form="fma")
    assert fma_p.shape != exp_p.shape or not np.array_equal(fma_p.view(np.uint32),
                                                            exp_p.view(np.uint32))


def test_known_answers():
    W, H = 7, 5
    cam = dict(fx=500.0, fy=400.0, cx=3.0, cy=2.0, depth_encoding="16UC1", color_encoding="bgra8")
    depth = np.full((H, W), 1234, np.uint16)
    depth[0, :] = 0  # first row invalid
    depth[4, 6] = 0  # last pixel invalid
    color = np.arange(H * W * 4, dtype=np.uint8).reshape(H, W, 4)
    pts, cols = ref.depth_cloud(depth, color, cam)
    assert len(pts) == H * W - W - 1
    # row-major order: the first kept point is pixel (u=0, v=1)
    k = (2 - 1) * W + 3  # principal pixel (u=3, v=2)
    assert pts[k, 0] == 0.0 and pts[k, 1] == 0.0
    assert pts[k, 2].view(np.uint32) == (np.float32(1234) * np.float32(0.001)).view(np.uint32)
    assert np.array_equal(cols[0], [color[1, 0, 2], color[1, 0, 1], color[1, 0, 0], 255])
    assert (cols[:, 3] == 255).all()
    assert pts[0, 0] < 0 and pts[0, 1] < 0  # u < cx, v < cy
    xs = pts[:W, 0]
    assert (np.diff(xs) > 0).all()  # u ascending inside a row
    for enc_name, (offs, pix) in ref.COLOR_LAYOUT.items():
        c = np.arange(H * W * pix, dtype=np.uint8).reshape(H, W, pix)
        _, cc = ref.depth_cloud(depth, c, dict(cam, color_encoding=enc_name))
        assert np.array_equal(cc[0, :3], [c[1, 0, o] for o in offs]), enc_name
    # 32FC1: metres unchanged, 0 is a valid (finite) depth
    f = np.ones((H, W), np.float32) * np.float32(2.5)
    f[0, 0] = 0.0
    f[0, 1] = np.nan
    p32, _ = ref.depth_cloud(f, color, dict(cam, depth_encoding="32FC1"))
    assert len(p32) == H * W - 1 and p32[0, 2] == 0.0 and p32[-1, 2] == np.float32(2.5)


def test_depth_camera_layout_matches_the_header():
    from coxgraph_b200 import capi
    fields = [f[0] for f in capi.DepthCamera._fields_]
    expr = ",".join(f"offsetof(cg_depth_camera,{f})" for f in fields)
    src = ('#include <stdio.h>\n#include <stddef.h>\n#include "coxgraph_b200.h"\n'
           'int main(void){size_t v[]={sizeof(cg_depth_camera),' + expr + '};'
           'for(unsigned i=0;i<sizeof(v)/sizeof(v[0]);++i)printf("%zu ",v[i]);'
           'printf("%d %d %d %d %d %d %d\\n",CG_DEPTH_16UC1,CG_DEPTH_32FC1,CG_COLOR_RGB8,'
           'CG_COLOR_RGBA8,CG_COLOR_BGR8,CG_COLOR_BGRA8,CG_COLOR_MONO8);return 0;}')
    with tempfile.TemporaryDirectory() as d:
        with open(os.path.join(d, "s.c"), "w") as f:
            f.write(src)
        subprocess.check_call(["gcc", "-std=c99", "-I", os.path.join(ROOT, "include"),
                               os.path.join(d, "s.c"), "-o", os.path.join(d, "s")])
        vals = [int(x) for x in subprocess.check_output([os.path.join(d, "s")]).split()]
    n = len(fields)
    assert vals[0] == C.sizeof(capi.DepthCamera) == 48
    assert vals[1:1 + n] == [getattr(capi.DepthCamera, f).offset for f in fields]
    assert vals[1 + n:] == [capi.DEPTH_16UC1, capi.DEPTH_32FC1, capi.COLOR_RGB8, capi.COLOR_RGBA8,
                            capi.COLOR_BGR8, capi.COLOR_BGRA8, capi.COLOR_MONO8]


@pytest.mark.parametrize("enc", ref.DEPTH_ENCODINGS)
def test_render_depth_frame_is_deterministic(enc):
    from coxgraph_b200 import synth
    T = synth.trajectory(3)[2]
    a = synth.render_depth_frame(T, stride=8, depth_encoding=enc)
    b = synth.render_depth_frame(T, stride=8, depth_encoding=enc)
    assert a[0].shape == (60, 80) and a[1].shape == (60, 80, 3)
    assert a[0].dtype == (np.uint16 if enc == "16UC1" else np.float32)
    assert np.array_equal(a[0], b[0]) and np.array_equal(a[1], b[1]) and a[2] == b[2]
    assert a[2]["fx"] == synth.CAM_640x480["fx"] / 8 and a[2]["width"] == 80
    # the depth is the z of render_frame's points (rounded to mm for 16UC1)
    pts, cols = synth.render_frame(T, stride=8)
    z = pts[:, 2].numpy().reshape(60, 80)
    if enc == "16UC1":
        assert np.abs(a[0].astype(np.float64) / 1000.0 - z).max() <= 0.0005 + 1e-6
    else:
        assert np.array_equal(a[0], z)
    assert np.array_equal(a[1].reshape(-1, 3), cols[:, :3].numpy())
