"""The C++ mirror of the sharded mesh gather (gatherMeshSharded, coxgraph_b200/host/
coxgraph_b200.hpp): it compiles with plain g++ against the C ABI, fails loudly without a GPU, and on
the GPU box writes, through a one-rank communicator, the same PLY file as generateMesh +
getConnectedMesh + outputMeshAsPly of the same layer (tests/host/mesh_gather_check.cc).  The
library dlopens libnccl.so.2, so the driver runs with the NCCL the Python environment carries on
its library path."""
import os
import subprocess

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
BIN = os.path.join(ROOT, "build", "mesh_gather_check")


def _binary():
    if not os.path.exists(BIN):
        subprocess.check_call(["make", "-C", ROOT, "-s", "build/mesh_gather_check"])
    return BIN


def _env():
    """LD_LIBRARY_PATH with the nvidia/nccl/lib directory of the Python environment, if any."""
    import importlib.util
    env = dict(os.environ)
    spec = importlib.util.find_spec("nvidia.nccl")
    dirs = [os.path.join(p, "lib") for p in (spec.submodule_search_locations or [])] if spec else []
    dirs = [d for d in dirs if os.path.exists(os.path.join(d, "libnccl.so.2"))]
    if dirs:
        env["LD_LIBRARY_PATH"] = os.pathsep.join(dirs + [env.get("LD_LIBRARY_PATH", "")]).rstrip(os.pathsep)
    return env


def test_mesh_gather_program_builds_and_fails_loudly_without_a_gpu():
    r = subprocess.run([_binary(), "nogpu"], capture_output=True, text=True, env=_env())
    # 0: no device, context creation raised CG_ERR_CUDA; 3: a device is present (GPU box)
    assert r.returncode in (0, 3), r.stdout + r.stderr
    if r.returncode == 0:
        assert "no CPU fallback" in r.stdout


@pytest.mark.gpu
def test_cpp_gathered_ply_equals_single_gpu_ply(tmp_path):
    r = subprocess.run([_binary(), "run", str(tmp_path)], capture_output=True, text=True,
                       env=_env(), timeout=600)
    assert r.returncode == 0, r.stdout + r.stderr
    lines = r.stdout.splitlines()
    assert [l for l in lines if l.startswith("ok ")] == [
        "ok global totals", "ok gathered mesh == generateMesh", "ok PLY files identical",
        "ok second gather rejected"], r.stdout
    a, b = (tmp_path / "sharded.ply").read_bytes(), (tmp_path / "single.ply").read_bytes()
    assert a == b and a.count(b"\n3 ") > 100
