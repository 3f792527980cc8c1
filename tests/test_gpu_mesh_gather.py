"""cg_mesh_gather_sharded (the ranks' block meshes gathered onto one root) against cg_layer_mesh.
On one GPU a one-rank communicator must leave, after cg_layer_mesh_sharded and the gather, exactly
what cg_layer_mesh leaves: cg_mesh_fetch and cg_mesh_connect give the same bytes.  With >= 2 GPUs
scripts/multigpu_mesh_gather_check.py compares the root's mesh with cg_layer_mesh of the union of
the owned layers built on one GPU."""
import ctypes as C
import os
import subprocess
import sys

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))

pytestmark = pytest.mark.gpu

ARGS = [dict(), dict(use_color=False), dict(min_weight=0.5), dict(min_weight=0.5, use_color=False)]
NAMES = ("block order", "vertex ranges", "vertices", "normals", "colours")
CONNECTED = ("connected vertices", "connected normals", "connected colours", "indices")


@pytest.fixture(scope="module")
def comm_ctx():
    import torch  # noqa: F401  (loads the libnccl.so.2 the library binds to)
    from coxgraph_b200.api import Context, commInit, commUniqueId
    ctx = Context(0)
    commInit(ctx, commUniqueId(), 0, 1)
    yield ctx
    ctx.close()


def _bytes_equal(got, ref, names, what):
    assert len(got) == len(ref)
    for name, g, r in zip(names, got, ref):
        assert g.dtype == r.dtype and g.shape == r.shape and \
            np.array_equal(g.view(np.uint8), r.view(np.uint8)), f"{what}: {name}"


def _gather_same(layer, what, **kw):
    """cg_layer_mesh_sharded + gather to root 0 == cg_layer_mesh: fetched and connected bytes."""
    from coxgraph_b200.api import gatherMeshSharded, generateMeshSharded
    ref = layer.generateMesh(**kw)
    ref_connected = layer.getConnectedMesh()
    generateMeshSharded(layer, fetch=False, **kw)
    got = gatherMeshSharded(layer.ctx, 0)
    _bytes_equal(got, ref, NAMES, f"{what} {kw}")
    _bytes_equal(layer.getConnectedMesh(), ref_connected, CONNECTED, f"{what} {kw}")
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


def _check_all(layer, what):
    for kw in ARGS:
        _gather_same(layer, what, **kw)
    _gather_same(layer, what, only_updated=True)
    idx, vox, fl = layer.download()
    sel = np.arange(0, len(idx), 3)
    layer.upload(idx[sel], vox[sel], fl[sel] & np.uint8(0xFD))  # clear every third `updated` flag
    out = _gather_same(layer, what + " after some flags were reset", only_updated=True)
    assert 0 < len(out[2]) < len(layer.generateMesh()[2])


def test_fused_submap_gathers_to_layer_mesh(comm_ctx):
    L = _fused_submap(comm_ctx, 0, 0)
    assert len(L.generateMesh()[2]) > 10000
    _check_all(L, "fused submap")
    L.close()


def test_projected_c2_map_gathers_to_layer_mesh(comm_ctx):
    """The C2 shape: submaps of two robots in one room, projected with cg_project_submaps_sharded
    (one rank: the owned layer is the whole global map)."""
    from coxgraph_b200 import Layer, synth
    from coxgraph_b200.api import gatherMeshSharded, generateMeshSharded, getProjectedMapSharded
    subs = [_fused_submap(comm_ctx, k % 2, k, frames=2, stride=4) for k in range(4)]
    rng = np.random.default_rng(5)
    poses = np.stack([synth.perturb_pose(synth.robot_map_offset(k % 2), rng, sigma_t=0.2,
                                         sigma_yaw_deg=15.0) for k in range(4)])
    partial = Layer(comm_ctx, 0.05, max_blocks=16384)
    owned = Layer(comm_ctx, 0.05, max_blocks=16384)
    getProjectedMapSharded(subs, poses, partial, owned)
    assert owned.num_blocks > 0
    _check_all(owned, "projected C2 map")
    # fetch=False: the global counts, the mesh stays retained for cg_mesh_fetch
    full = owned.generateMesh()
    generateMeshSharded(owned, fetch=False)
    assert gatherMeshSharded(comm_ctx, 0, fetch=False) == (len(full[0]), len(full[2]))
    from coxgraph_b200.api import _fetch_mesh
    _bytes_equal(_fetch_mesh(comm_ctx, len(full[0]), len(full[2])), full, NAMES, "fetch after count")
    for L in subs + [partial, owned]:
        L.close()


def test_empty_layer(comm_ctx):
    from coxgraph_b200 import Layer
    from coxgraph_b200.api import gatherMeshSharded, generateMeshSharded
    E = Layer(comm_ctx, 0.05, max_blocks=64)
    generateMeshSharded(E, fetch=False)
    assert gatherMeshSharded(comm_ctx, 0, fetch=False) == (0, 0)
    generateMeshSharded(E, fetch=False)
    idx, begin, v, n, c = gatherMeshSharded(comm_ctx, 0)
    assert len(idx) == 0 and len(v) == 0 and list(begin) == [0]
    cv, cn, cc, ci = E.getConnectedMesh()
    assert len(cv) == len(cn) == len(cc) == len(ci) == 0
    E.close()


def _expect_invalid(fn, needle):
    from coxgraph_b200 import capi
    with pytest.raises(capi.CgError) as e:
        fn()
    assert e.value.status == capi.CG_ERR_INVALID_ARG and needle in str(e.value), str(e.value)


def test_rejections_each_followed_by_a_good_gather(comm_ctx):
    from coxgraph_b200 import Context, capi
    from coxgraph_b200.api import _fetch_mesh, commInit, commUniqueId, gatherMeshSharded, generateMeshSharded
    L = _fused_submap(comm_ctx, 1, 2, frames=2, stride=4)
    lib = capi.load()
    nb, nv = C.c_size_t(7), C.c_size_t(7)

    def good():
        _gather_same(L, "after a rejection")

    # a NULL context
    generateMeshSharded(L, fetch=False)
    _expect_invalid(lambda: capi.check(lib.cg_mesh_gather_sharded(None, 0, C.byref(nb), C.byref(nv))),
                    "null context")
    assert (nb.value, nv.value) == (0, 0)
    good()
    # no communicator; then a communicator but no mesh retained
    other = Context(0)
    _expect_invalid(lambda: gatherMeshSharded(other, 0), "cg_comm_init")
    good()
    commInit(other, commUniqueId(), 0, 1)
    _expect_invalid(lambda: gatherMeshSharded(other, 0), "does not exist")
    other.close()
    good()
    # roots outside [0, 1); the retained mesh is left alone
    for root in (1, -1):
        B, V = generateMeshSharded(L, fetch=False)
        _expect_invalid(lambda: gatherMeshSharded(comm_ctx, root), f"root {root}")
        _bytes_equal(_fetch_mesh(comm_ctx, B, V), L.generateMesh(), NAMES, f"root {root}: retained")
        good()
    # a plain cg_layer_mesh since the sharded one
    generateMeshSharded(L, fetch=False)
    L.generateMesh(fetch=False)
    _expect_invalid(lambda: gatherMeshSharded(comm_ctx, 0), "cg_layer_mesh, not cg_layer_mesh_sharded")
    good()
    # cg_esdf_free_points reuses the mesh buffers
    L.updateEsdfBatch(fetch=False)
    generateMeshSharded(L, fetch=False)
    assert len(L.esdfFreePoints(0.1)) > 0
    _expect_invalid(lambda: gatherMeshSharded(comm_ctx, 0), "cg_esdf_free_points")
    good()
    # a second gather without meshing again
    generateMeshSharded(L, fetch=False)
    gatherMeshSharded(comm_ctx, 0, fetch=False)
    _expect_invalid(lambda: gatherMeshSharded(comm_ctx, 0), "gathered already")
    good()
    L.close()


def test_gather_over_nccl():
    import torch
    n = torch.cuda.device_count()
    if n < 2:
        pytest.skip("needs at least 2 GPUs")
    world = 4 if n >= 4 else 2
    r = subprocess.run([sys.executable, "-m", "torch.distributed.run", "--nnodes=1",
                        f"--nproc-per-node={world}", "--master-addr", "127.0.0.1",
                        "--master-port", "29541",
                        os.path.join(ROOT, "scripts", "multigpu_mesh_gather_check.py")],
                       capture_output=True, text=True, timeout=900)
    assert r.returncode == 0 and "multigpu_mesh_gather_check ok" in r.stdout, \
        r.stdout[-3000:] + r.stderr[-3000:]
