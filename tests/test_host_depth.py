"""The C++ mirror of the depth-image entry points (TsdfIntegratorBase::integrateDepthImage /
integrateDepthImages, coxgraph_b200/host/coxgraph_b200.hpp): it compiles with plain g++ against the
C ABI, fails loudly without a GPU, and on the GPU box gives the layer of the Python path bit for
bit."""
import os
import struct
import subprocess

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
BIN = os.path.join(ROOT, "build", "depth_api_check")


def _binary():
    if not os.path.exists(BIN):
        subprocess.check_call(["make", "-C", ROOT, "-s", "build/depth_api_check"])
    return BIN


def test_depth_program_builds_and_fails_loudly_without_a_gpu():
    r = subprocess.run([_binary(), "nogpu"], capture_output=True, text=True)
    # 0: no device, context creation raised CG_ERR_CUDA; 3: a device is present (GPU box)
    assert r.returncode in (0, 3), r.stdout + r.stderr
    if r.returncode == 0:
        assert "no CPU fallback" in r.stdout


@pytest.mark.gpu
@pytest.mark.parametrize("enc", ["16UC1", "32FC1"])
def test_cpp_depth_matches_python(gpu_ctx, tmp_path, enc):
    from coxgraph_b200 import Layer, TsdfIntegrator, TsdfIntegratorConfig, VOXEL_DTYPE, capi, synth
    poses = synth.trajectory(3, robot=1).astype(np.float32)
    frames = [synth.render_depth_frame(T, stride=4, depth_encoding=enc) for T in poses]
    cam = dict(frames[0][2], color_encoding="bgr8")
    depth = np.stack([d for d, _, _ in frames])
    color = np.ascontiguousarray(np.stack([c for _, c, _ in frames])[..., ::-1])
    depth[1, ::5] = 0 if enc == "16UC1" else np.nan
    voxel, trunc = 0.05, 0.15
    with open(tmp_path / "in.bin", "wb") as f:
        f.write(struct.pack("<Iiiii", len(poses), cam["width"], cam["height"],
                            capi.DEPTH_ENCODINGS[enc], capi.COLOR_BGR8))
        f.write(struct.pack("<ddddff", cam["fx"], cam["fy"], cam["cx"], cam["cy"], voxel, trunc))
        for k in range(len(poses)):
            f.write(poses[k].tobytes() + depth[k].tobytes() + color[k].tobytes())
    r = subprocess.run([_binary(), "run", str(tmp_path / "in.bin"), str(tmp_path / "out.bin")],
                       capture_output=True, text=True)
    assert r.returncode == 0, r.stdout + r.stderr
    buf = open(tmp_path / "out.bin", "rb").read()
    (B,) = struct.unpack_from("<I", buf, 0)
    idx = np.frombuffer(buf, np.int32, 3 * B, 4).reshape(B, 3)
    vox = np.frombuffer(buf, VOXEL_DTYPE, 4096 * B, 4 + 12 * B).reshape(B, 4096)
    flags = np.frombuffer(buf, np.uint8, B, 4 + 12 * B + 4096 * 12 * B)
    L = Layer(gpu_ctx, voxel, max_blocks=4096)
    it = TsdfIntegrator(TsdfIntegratorConfig(default_truncation_distance=trunc), L)
    it.integrateDepthImage(poses[0], depth[0], color[0], cam)
    it.integrateDepthBatch(poses[1:], depth[1:], color[1:], cam)
    gi, gv, gf = L.download()
    assert np.array_equal(gi, idx) and np.array_equal(gf, flags)
    assert gv.tobytes() == vox.tobytes()
    L.close()
