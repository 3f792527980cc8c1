"""GPU parity: cg_merge_layer_into_layer / cg_project_submaps against the CPU oracle.  Both sides
merge the same input layers, so the results must be bit-identical (distance, weight, colour and
block flags); only test_integrate_then_merge_end_to_end, whose inputs are fused separately, is
held to the tolerance.
Reference call sites: coxgraph/src/client/map_server.cpp:59-73,
coxgraph/src/server/visualizer/server_visualizer.cpp:123-126."""
import numpy as np
import pytest

from coxgraph_b200 import synth
from tests import util

pytestmark = pytest.mark.gpu


def _submap(orc, ocfg, robot, submap, frames=2, stride=8, voxel_size=0.05):
    ol = orc.Layer(voxel_size)
    for (T, p, c) in util.small_frames(frames, stride=stride, robot=robot, submap=submap):
        ol.integrate(ocfg, T, p, c)
    return ol


def _to_gpu(gpu_ctx, ol, max_blocks=4096):
    from coxgraph_b200 import Layer
    gl = Layer(gpu_ctx, ol.voxel_size, max_blocks=max_blocks)
    idx, vox, fl = ol.download()
    gl.upload(idx, vox, np.ones_like(fl))
    return gl


POSES = [
    np.array([1, 0, 0, 0, 0, 0, 0], np.float32),                       # identity
    np.array([1, 0, 0, 0, 0.8, -1.6, 0.8], np.float32),                 # whole-block shift
    np.array([np.cos(0.3), 0, 0, np.sin(0.3), 0.37, -0.21, 0.05], np.float32),
    synth.robot_map_offset(1),
    np.array([0.9238795, 0.2209424, 0.2209424, 0.2209424, -1.3, 0.4, 0.2], np.float32),
]


@pytest.mark.parametrize("pose_id", range(len(POSES)))
def test_merge_matches_oracle(gpu_ctx, pose_id):
    from coxgraph_b200 import Layer, mergeLayerAintoLayerB
    from oracle import oracle_py as orc
    ocfg, _ = util.make_cfgs()
    T = POSES[pose_id].copy()
    T[:4] /= np.linalg.norm(T[:4])
    oa = _submap(orc, ocfg, 0, 0)
    ga = _to_gpu(gpu_ctx, oa)
    ob = orc.Layer(0.05)
    gb = Layer(gpu_ctx, 0.05, max_blocks=4096)
    for rep in range(2):  # second pass merges into existing blocks
        ob.merge_from(oa, T)
        st = mergeLayerAintoLayerB(ga, T, gb)
        assert st.blocks_out == ob.last_blocks_out
        assert st.blocks_in == oa.num_blocks
        util.compare_layers(gb.download(), ob.download(), f"merge pose {pose_id} rep {rep}",
                            exact=True, check_flags=True)
    ga.close()
    gb.close()


@pytest.mark.parametrize("src_voxel,dst_voxel", [(0.05, 0.10), (0.10, 0.05), (0.05, 0.04)])
def test_merge_between_different_voxel_sizes(gpu_ctx, src_voxel, dst_voxel):
    """mergeLayerAintoLayerB resamples, so the two layers need not share a grid: coarser and finer
    destinations, single merge and batched projection (the slot table of the gather covers 4^3
    source blocks; a coarser destination reaches beyond it and takes the hash path)."""
    from coxgraph_b200 import Layer, getProjectedMap, mergeLayerAintoLayerB
    from oracle import oracle_py as orc
    ocfg, _ = util.make_cfgs()
    subs_o = [_submap(orc, ocfg, k % 2, k, voxel_size=src_voxel) for k in range(3)]
    subs_g = [_to_gpu(gpu_ctx, o) for o in subs_o]
    poses = [POSES[2] / np.linalg.norm(POSES[2][:4]).astype(np.float32), POSES[3], POSES[4].copy()]
    poses[2][:4] /= np.linalg.norm(poses[2][:4])
    poses = [np.asarray(p, np.float32) for p in poses]
    ob, gb = orc.Layer(dst_voxel), Layer(gpu_ctx, dst_voxel, max_blocks=16384)
    ob.merge_from(subs_o[0], poses[0])
    st = mergeLayerAintoLayerB(subs_g[0], poses[0], gb)
    assert st.blocks_out == ob.last_blocks_out
    util.compare_layers(gb.download(), ob.download(), "single merge", exact=True, check_flags=True)
    og, gg = orc.Layer(dst_voxel), Layer(gpu_ctx, dst_voxel, max_blocks=16384)
    for o, T in zip(subs_o, poses):
        og.merge_from(o, T)
    getProjectedMap(subs_g, np.stack(poses), gg)
    util.compare_layers(gg.download(), og.download(), "projection", exact=True, check_flags=True)
    for L in subs_g + [gb, gg]:
        L.close()


def test_dense_submaps_project_matches_oracle(gpu_ctx):
    """Submaps fused from full 640x480 frames (dense truncation bands, ~100 blocks each) projected
    into one global layer under oblique poses, batched on the device, against the oracle's
    sequential mergeLayerAintoLayerB."""
    from coxgraph_b200 import Layer, getProjectedMap
    from oracle import oracle_py as orc
    ocfg, _ = util.make_cfgs(default_truncation_distance=0.16)
    subs_o = [_submap(orc, ocfg, r, s, frames=2, stride=1) for (r, s) in ((0, 0), (1, 3), (0, 5))]
    subs_g = [_to_gpu(gpu_ctx, ol) for ol in subs_o]
    poses = [POSES[2].copy(), synth.robot_map_offset(1), POSES[4].copy()]
    for T in poses:
        T[:4] /= np.linalg.norm(T[:4])
    og = orc.Layer(0.05)
    for ol, T in zip(subs_o, poses):
        og.merge_from(ol, T, threads=8)
    gg = Layer(gpu_ctx, 0.05, max_blocks=8192)
    st = getProjectedMap(subs_g, np.stack(poses), gg, want_stats=True)
    assert st.blocks_in == sum(ol.num_blocks for ol in subs_o)
    util.compare_layers(gg.download(), og.download(), "dense projection", exact=True,
                        check_flags=True)
    for g in subs_g + [gg]:
        g.close()


def test_project_submaps_matches_sequential_oracle(gpu_ctx):
    from coxgraph_b200 import Layer, getProjectedMap
    from oracle import oracle_py as orc
    ocfg, _ = util.make_cfgs(default_truncation_distance=0.16)
    subs, poses = [], []
    for robot in (0, 1):
        for sm in range(2):
            subs.append(_submap(orc, ocfg, robot, sm))
            poses.append(synth.robot_map_offset(robot))
    og = orc.Layer(0.05)
    for s, T in zip(subs, poses):
        og.merge_from(s, T)
    gsubs = [_to_gpu(gpu_ctx, s) for s in subs]
    gg = Layer(gpu_ctx, 0.05, max_blocks=8192)
    st = getProjectedMap(gsubs, np.stack(poses), gg, want_stats=True)
    assert st.blocks_in == sum(s.num_blocks for s in subs)
    util.compare_layers(gg.download(), og.download(), "projected map", exact=True, check_flags=True)
    # re-projection after a pose update (config 5): fresh global layer, perturbed poses
    rng = np.random.default_rng(synth.SEED)
    poses2 = [synth.perturb_pose(T, rng) for T in poses]
    gg.removeAllBlocks()
    og.clear()
    for s, T in zip(subs, poses2):
        og.merge_from(s, T)
    getProjectedMap(gsubs, np.stack(poses2), gg)
    util.compare_layers(gg.download(), og.download(), "re-projected map", exact=True,
                        check_flags=True)
    for g in gsubs + [gg]:
        g.close()


def test_merge_empty_and_errors(gpu_ctx):
    from coxgraph_b200 import Layer, capi, mergeLayerAintoLayerB
    a = Layer(gpu_ctx, 0.05, max_blocks=16)
    b = Layer(gpu_ctx, 0.05, max_blocks=16)
    st = mergeLayerAintoLayerB(a, POSES[0], b)
    assert st.blocks_out == 0 and b.num_blocks == 0
    with pytest.raises(capi.CgError):
        mergeLayerAintoLayerB(a, POSES[0], a)
    a.close()
    b.close()


def test_integrate_then_merge_end_to_end(gpu_ctx):
    """Fuse on the GPU, merge on the GPU, compare with the oracle doing the same."""
    from coxgraph_b200 import Layer, TsdfIntegrator, mergeLayerAintoLayerB
    from oracle import oracle_py as orc
    ocfg, gcfg = util.make_cfgs()
    frames = util.small_frames(3, stride=8, robot=1)
    oa, ga = orc.Layer(0.05), Layer(gpu_ctx, 0.05, max_blocks=2048)
    integ = TsdfIntegrator(gcfg, ga)
    for (T, p, c) in frames:
        oa.integrate(ocfg, T, p, c)
        integ.integratePointCloud(T, p, c)
    ob, gb = orc.Layer(0.05), Layer(gpu_ctx, 0.05, max_blocks=4096)
    T = synth.robot_map_offset(1)
    ob.merge_from(oa, T)
    mergeLayerAintoLayerB(ga, T, gb)
    util.compare_layers(gb.download(), ob.download(), "fuse+merge")
    ga.close()
    gb.close()
