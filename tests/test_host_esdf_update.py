"""The C++ mirror of the incremental ESDF (EsdfIntegrator::updateFromTsdfLayer,
coxgraph_b200/host/coxgraph_b200.hpp): it compiles with plain g++ against the C ABI, fails loudly
without a GPU, and on the GPU box matches updateFromTsdfLayerBatch bit for bit over a chain of
layer edits (tests/host/esdf_update_check.cc)."""
import os
import subprocess

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
BIN = os.path.join(ROOT, "build", "esdf_update_check")


def _binary():
    if not os.path.exists(BIN):
        subprocess.check_call(["make", "-C", ROOT, "-s", "build/esdf_update_check"])
    return BIN


def test_esdf_update_program_builds_and_fails_loudly_without_a_gpu():
    r = subprocess.run([_binary(), "nogpu"], capture_output=True, text=True)
    # 0: no device, context creation raised CG_ERR_CUDA; 3: a device is present (GPU box)
    assert r.returncode in (0, 3), r.stdout + r.stderr
    if r.returncode == 0:
        assert "no CPU fallback" in r.stdout


@pytest.mark.gpu
def test_cpp_update_matches_batch():
    r = subprocess.run([_binary(), "run"], capture_output=True, text=True)
    assert r.returncode == 0, r.stdout + r.stderr
    lines = r.stdout.splitlines()
    assert len(lines) == 5 and all(l.startswith("ok ") for l in lines), r.stdout
    assert "removed 1 " in lines[2] and "full 0" in lines[4] and "region 0 " in lines[4]
