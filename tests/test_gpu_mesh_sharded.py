"""cg_layer_mesh_sharded (marching cubes over a sharded global map, the halo read from the peer
ranks) against cg_layer_mesh.  On one GPU a one-rank communicator must give cg_layer_mesh's bytes
exactly; with >= 2 GPUs scripts/multigpu_mesh_check.py compares the ranks' meshes with
cg_layer_mesh of the gathered map block by block."""
import os
import subprocess
import sys

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))

pytestmark = pytest.mark.gpu

ARGS = [dict(), dict(use_color=False), dict(min_weight=0.5), dict(min_weight=0.5, use_color=False)]


@pytest.fixture(scope="module")
def comm_ctx():
    import torch  # noqa: F401  (loads the libnccl.so.2 the library binds to)
    from coxgraph_b200.api import Context, commInit, commUniqueId
    ctx = Context(0)
    commInit(ctx, commUniqueId(), 0, 1)
    yield ctx
    ctx.close()


def _same(owned, what, **kw):
    from coxgraph_b200.api import generateMeshSharded
    got = generateMeshSharded(owned, **kw)
    ref = owned.generateMesh(**kw)
    for name, g, r in zip(("block order", "vertex ranges", "vertices", "normals", "colours"),
                          got, ref):
        assert g.dtype == r.dtype and np.array_equal(g.view(np.uint8), r.view(np.uint8)), \
            f"{what} {kw}: {name}"
    return got


def _fused_submap(ctx, robot, submap, frames=3, stride=2):
    import torch
    from coxgraph_b200 import Layer, TsdfIntegrator, TsdfIntegratorConfig, synth
    cfg = TsdfIntegratorConfig(use_const_weight=1, method=1, default_truncation_distance=0.16)
    L = Layer(ctx, 0.05, max_blocks=4096)
    integ = TsdfIntegrator(cfg, L)
    for (T, pts, cols) in synth.submap_frames(robot, submap, frames, device=torch.device("cuda", 0),
                                              stride=stride):
        integ.integratePointCloud(T, pts, cols)
    return L


def _reset_some_updated(layer, every=3):
    """Clear the `updated` flag of every `every`-th block (re-upload with the flag cleared)."""
    idx, vox, fl = layer.download()
    sel = np.arange(0, len(idx), every)
    layer.upload(idx[sel], vox[sel], fl[sel] & np.uint8(0xFD))
    return len(sel)


def _check_all(owned, what):
    for kw in ARGS:
        _same(owned, what, **kw)
    _same(owned, what, only_updated=True)
    assert _reset_some_updated(owned) > 0
    out = _same(owned, what + " after some flags were reset", only_updated=True)
    assert 0 < len(out[2]) < len(owned.generateMesh()[2])


def test_one_rank_fused_submap_equals_layer_mesh(comm_ctx):
    L = _fused_submap(comm_ctx, 0, 0)
    assert len(L.generateMesh()[2]) > 10000
    _check_all(L, "fused submap")
    L.close()


def test_one_rank_projected_c2_map_equals_layer_mesh(comm_ctx):
    """The C2 shape: submaps of two robots in one room, projected with cg_project_submaps_sharded
    (one rank: the owned layer is the whole global map)."""
    from coxgraph_b200 import Layer, getProjectedMap, synth
    from coxgraph_b200.api import getProjectedMapSharded
    subs = [_fused_submap(comm_ctx, k % 2, k, frames=2, stride=4) for k in range(4)]
    rng = np.random.default_rng(5)
    poses = np.stack([synth.perturb_pose(synth.robot_map_offset(k % 2), rng, sigma_t=0.2,
                                         sigma_yaw_deg=15.0) for k in range(4)])
    partial = Layer(comm_ctx, 0.05, max_blocks=16384)
    owned = Layer(comm_ctx, 0.05, max_blocks=16384)
    getProjectedMapSharded(subs, poses, partial, owned)
    # one rank owns the whole projected map
    single = Layer(comm_ctx, 0.05, max_blocks=16384)
    getProjectedMap(subs, poses, single)
    assert owned.num_blocks == single.num_blocks > 0
    assert np.array_equal(owned.block_indices()[np.lexsort(owned.block_indices().T)],
                          single.block_indices()[np.lexsort(single.block_indices().T)])
    single.close()
    _check_all(owned, "projected C2 map")
    # the count query leaves the mesh on the device for cg_mesh_fetch, as generateMesh does
    from coxgraph_b200.api import generateMeshSharded
    full = owned.generateMesh()
    assert generateMeshSharded(owned, fetch=False) == (len(full[0]), len(full[2]))
    for L in subs + [partial, owned]:
        L.close()


def test_one_rank_empty_layer(comm_ctx):
    from coxgraph_b200 import Layer
    from coxgraph_b200.api import generateMeshSharded
    E = Layer(comm_ctx, 0.05, max_blocks=64)
    idx, begin, v, n, c = generateMeshSharded(E)
    assert len(idx) == 0 and len(v) == 0 and list(begin) == [0]
    E.close()


def test_rejected_without_a_communicator(comm_ctx):
    from coxgraph_b200 import Context, Layer, capi
    from coxgraph_b200.api import generateMeshSharded
    other = Context(0)  # no commInit: the layer's context has no communicator
    L = Layer(other, 0.05, max_blocks=64)
    with pytest.raises(capi.CgError) as e:
        generateMeshSharded(L)
    assert e.value.status == capi.CG_ERR_INVALID_ARG and "cg_comm_init" in str(e.value)
    L.close()
    other.close()
    with pytest.raises(capi.CgError) as e:
        capi.check(capi.load().cg_layer_mesh_sharded(None, 1e-4, 1, 0, 0, 0, None, None, None, None,
                                                     None, None, None))
    assert e.value.status == capi.CG_ERR_INVALID_ARG


@pytest.mark.gpu
def test_sharded_mesh_over_nccl():
    import torch
    n = torch.cuda.device_count()
    if n < 2:
        pytest.skip("needs at least 2 GPUs")
    world = 4 if n >= 4 else 2
    r = subprocess.run([sys.executable, "-m", "torch.distributed.run", "--nnodes=1",
                        f"--nproc-per-node={world}", "--master-addr", "127.0.0.1",
                        "--master-port", "29523",
                        os.path.join(ROOT, "scripts", "multigpu_mesh_check.py")],
                       capture_output=True, text=True, timeout=900)
    assert r.returncode == 0 and "multigpu_mesh_check ok" in r.stdout, \
        r.stdout[-3000:] + r.stderr[-3000:]
