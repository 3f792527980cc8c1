"""GPU parity: cg_integrate_* against the CPU oracle on identical seeded inputs (through the
C ABI).  Reference call site: coxgraph/include/coxgraph/map_comm/tsdf_recover.h:59-99."""
import numpy as np
import pytest

from tests import util

pytestmark = pytest.mark.gpu


def _run_both(gpu_ctx, frames, voxel_size=0.05, batch=False, max_blocks=2048, **over):
    from coxgraph_b200 import Layer, TsdfIntegrator
    from oracle import oracle_py as orc
    ocfg, gcfg = util.make_cfgs(**over)
    ol = orc.Layer(voxel_size)
    gl = Layer(gpu_ctx, voxel_size, max_blocks=max_blocks)
    integ = TsdfIntegrator(gcfg, gl)
    touched = []
    for (T, p, c) in frames:
        ol.integrate(ocfg, T, p, c)
        touched.append(ol.last_blocks_touched)
    if batch:
        offs = np.cumsum([0] + [len(p) for (_, p, _) in frames]).astype(np.uint64)
        integ.integrateBatch(np.stack([T for (T, _, _) in frames]),
                             np.concatenate([p for (_, p, _) in frames]),
                             np.concatenate([c for (_, _, c) in frames]), offs)
    else:
        for k, (T, p, c) in enumerate(frames):
            st = integ.integratePointCloud(T, p, c)
            assert st.blocks_touched == touched[k], "B_touched differs from the oracle"
            assert st.points_in == len(p)
    return gl.download(), ol.download(), gl


@pytest.mark.parametrize("method", [1, 0])
def test_single_frames_match_oracle(gpu_ctx, method):
    frames = util.small_frames(3, stride=8 if method == 1 else 16)
    got, ref, gl = _run_both(gpu_ctx, frames, method=method)
    util.compare_layers(got, ref, f"method {method}")
    # the voxel update composes clamped affine maps in a tree: not bit-identical to the
    # sequential oracle, but nearly every voxel is still within a couple of ulps
    assert util.exact_fraction(got, ref) > 0.5
    gl.close()


def test_batch_equals_sequential(gpu_ctx):
    frames = util.small_frames(5, stride=8)
    got, ref, gl = _run_both(gpu_ctx, frames, batch=True)
    util.compare_layers(got, ref, "batch")
    gl.close()


def test_batch_many_ragged_frames(gpu_ctx):
    """40 small frames of different sizes in ONE group, one of them empty, one with dropped (NaN /
    too close) points only at its end: the bundles of all frames interleave in the voxel-major
    sort and the ray ids must still come out in (frame, clearing, voxel) order — a wrong order
    shows up in every voxel that two frames update."""
    base = util.small_frames(8, stride=16)
    frames = []
    for k in range(40):
        T, p, c = base[k % len(base)]
        n = len(p) - 37 * (k % 5)              # ragged
        p, c = p[:n].copy(), c[:n].copy()
        if k == 7:
            p, c = p[:0], c[:0]                # an empty frame
        if k == 11:
            p[-200:] = np.nan                  # dropped points
            p[-400:-200] *= 0.001              # closer than min_ray_length
        frames.append((T, p, c))
    got, ref, gl = _run_both(gpu_ctx, frames, batch=True)
    util.compare_layers(got, ref, "40 ragged frames in one group")
    gl.close()


def test_batch_split_path(gpu_ctx, monkeypatch):
    monkeypatch.setenv("CG_MAX_PAIRS", "100000")
    frames = util.small_frames(4, stride=8)
    got, ref, gl = _run_both(gpu_ctx, frames, batch=True)
    util.compare_layers(got, ref, "batch split")
    gl.close()


def test_far_points_regroup_then_out_of_range(gpu_ctx):
    """The bundle keys cover the box of voxels (relative to the sensor) that earlier jobs measured;
    a point outside it makes the library redo the group with the measured extent instead of
    failing.  A stray return more than 8191 voxels from the sensor (410 m at 5 cm) is dropped and
    counted — the frame is integrated without it — where round 1 failed the whole frame."""
    from coxgraph_b200 import Layer, TsdfIntegrator
    from oracle import oracle_py as orc
    frames = util.small_frames(5, stride=8)
    T, p, c = frames[2]
    p = p.copy()
    p[7] = (0.5, -0.3, 150.0)          # 3000 voxels away: a clearing ray (beyond max_ray)
    frames[2] = (T, p, c)
    got, ref, gl = _run_both(gpu_ctx, frames, batch=True)
    util.compare_layers(got, ref, "far clearing point in a batch")
    gl.close()
    ocfg, gcfg = util.make_cfgs()
    gl = Layer(gpu_ctx, 0.05, max_blocks=2048)
    p2 = p.copy()
    # 20000 voxels: some axis is beyond 8191 whatever the pose.  The last point of the cloud: it
    # lies in the tail the "mixed" order visits in natural order, so removing it leaves the
    # visiting order of all the others as it is
    assert len(p2) % 1024 != 0 and (len(p2) - 1) // 1024 == len(p2) // 1024
    p2[-1] = (0.0, 0.0, 1000.0)
    st = TsdfIntegrator(gcfg, gl).integratePointCloud(T, p2, c)
    assert st.points_beyond_reach == 1 and st.points_in == len(p2)
    ol = orc.Layer(0.05)
    ol.integrate(ocfg, T, p2[:-1], c[:-1])   # the oracle without the dropped point
    util.compare_layers(gl.download(), ol.download(), "frame with one point beyond the key reach")
    gl.close()


def test_staged_double_buffer(gpu_ctx):
    """cg_stage_batch_async + cg_integrate_batch_staged: inputs of job k+1 are copied while job k
    is fused; results equal the plain calls."""
    import torch
    from coxgraph_b200 import Layer, TsdfIntegrator
    from oracle import oracle_py as orc
    ocfg, gcfg = util.make_cfgs()
    jobs = [util.small_frames(2, stride=8, submap=s) for s in range(3)]
    gl = Layer(gpu_ctx, 0.05, max_blocks=2048)
    integ = TsdfIntegrator(gcfg, gl)
    host = []
    for frames in jobs:
        p = torch.from_numpy(np.concatenate([p for (_, p, _) in frames])).pin_memory().numpy()
        c = torch.from_numpy(np.concatenate([c for (_, _, c) in frames])).pin_memory().numpy()
        offs = np.cumsum([0] + [len(p_) for (_, p_, _) in frames]).astype(np.uint64)
        host.append((np.stack([T for (T, _, _) in frames]), p, c, offs))
    integ.stageBatch(0, host[0][1], host[0][2])
    for k, (poses, p, c, offs) in enumerate(host):
        if k + 1 < len(host):
            integ.stageBatch((k + 1) % 2, host[k + 1][1], host[k + 1][2])
        gl.clear()
        integ.integrateStaged(k % 2, poses, offs)
        ol = orc.Layer(0.05)
        for (T, pp, cc) in jobs[k]:
            ol.integrate(ocfg, T, pp, cc)
        util.compare_layers(gl.download(), ol.download(), f"staged job {k}")
    with pytest.raises(Exception):
        integ.integrateStaged(0, host[0][0], host[0][3][:-1])
    gl.close()


def test_touch_scratch_growth(monkeypatch):
    """The per-call touch scratch starts too small, overflows, grows and the walks are redone."""
    from coxgraph_b200 import Context
    monkeypatch.setenv("CG_TOUCH_CAP", "8")
    ctx = Context(0)          # fresh context: its scratch starts at the tiny capacity
    frames = util.small_frames(2, stride=8)
    got, ref, gl = _run_both(ctx, frames)
    util.compare_layers(got, ref, "touch growth")
    gl.close()
    ctx.close()


@pytest.mark.parametrize("over", [
    dict(use_const_weight=0),
    dict(voxel_carving_enabled=0),
    dict(allow_clear=0),
    dict(use_weight_dropoff=0, use_sparsity_compensation_factor=1,
         sparsity_compensation_factor=20.0, max_weight=1000.0),
    dict(integration_order_mode=1),
    dict(default_truncation_distance=0.16),
    dict(enable_anti_grazing=1),
    dict(enable_anti_grazing=1, voxel_carving_enabled=0, use_const_weight=0),
])
def test_config_variants(gpu_ctx, over):
    frames = util.small_frames(2, stride=8, robot=1)
    got, ref, gl = _run_both(gpu_ctx, frames, **over)
    util.compare_layers(got, ref, str(over))
    gl.close()


def test_full_resolution_frames_match_oracle(gpu_ctx):
    """Dense 640x480 frames (bundles of up to ~1000 points, update lists of hundreds): the paths
    the sub-sampled cases never reach — warp-cooperative bundle fold, warp replay of long update
    lists, block tiles with many segments — against the oracle, voxel by voxel."""
    frames = util.small_frames(3, stride=1, robot=1, submap=2)
    assert len(frames[0][1]) == 640 * 480
    got, ref, gl = _run_both(gpu_ctx, frames, batch=True, max_blocks=4096,
                             default_truncation_distance=0.16)
    util.compare_layers(got, ref, "full resolution, batch of 3")
    gl.close()
    got, ref, gl = _run_both(gpu_ctx, frames[:2], max_blocks=4096, use_const_weight=0)
    util.compare_layers(got, ref, "full resolution, per frame, 1/z^2 weights")
    gl.close()
    # anti-grazing at full density: many voxels are skipped (the result must differ from the
    # plain one) and segments are split at every skipped voxel
    plain = got
    got, ref, gl = _run_both(gpu_ctx, frames[:2], batch=True, max_blocks=4096,
                             use_const_weight=0, enable_anti_grazing=1)
    util.compare_layers(got, ref, "full resolution, anti-grazing")
    assert got[0].shape != plain[0].shape or not np.array_equal(got[1]["weight"], plain[1]["weight"])
    gl.close()


def test_fine_voxels_720p(gpu_ctx):
    from coxgraph_b200 import synth
    frames = util.small_frames(2, stride=8, cam=synth.CAM_1280x720)
    got, ref, gl = _run_both(gpu_ctx, frames, voxel_size=0.02, max_blocks=8192,
                             default_truncation_distance=0.06, max_ray_length_m=3.0)
    util.compare_layers(got, ref, "2 cm")
    gl.close()


def test_freespace_and_edge_inputs(gpu_ctx):
    from coxgraph_b200 import Layer, TsdfIntegrator
    from oracle import oracle_py as orc
    ocfg, gcfg = util.make_cfgs()
    (T, p, c), = util.small_frames(1, stride=16)
    p = p.copy()
    p[5] = np.nan          # non-finite points are dropped
    p[6] = [0, 0, 0.01]    # closer than min_ray
    p[7] = [np.inf, 0, 1]
    ol = orc.Layer(0.05)
    gl = Layer(gpu_ctx, 0.05, max_blocks=1024)
    integ = TsdfIntegrator(gcfg, gl)
    ol.integrate(ocfg, T, p, c, freespace=True)
    integ.integratePointCloud(T, p, c, freespace_points=True)
    # empty cloud is a no-op
    integ.integratePointCloud(T, np.zeros((0, 3), np.float32), np.zeros((0, 4), np.uint8))
    util.compare_layers(gl.download(), ol.download(), "freespace")
    gl.removeAllBlocks()
    assert gl.num_blocks == 0 and len(gl.download()[0]) == 0
    # after a clear the pool is back in its default state
    integ.integratePointCloud(T, p, c)
    ol.clear()
    ol.integrate(ocfg, T, p, c)
    util.compare_layers(gl.download(), ol.download(), "after clear")
    gl.close()


def test_pool_exhaustion_and_unsupported(gpu_ctx):
    from coxgraph_b200 import Layer, TsdfIntegrator, capi
    _, gcfg = util.make_cfgs()
    (T, p, c), = util.small_frames(1, stride=16)
    gl = Layer(gpu_ctx, 0.05, max_blocks=8)
    with pytest.raises(capi.CgError) as e:
        TsdfIntegrator(gcfg, gl).integratePointCloud(T, p, c)
    assert e.value.status == capi.CG_ERR_POOL_FULL
    assert gl.num_blocks == 8
    gl.close()
    _, fast = util.make_cfgs(method=2)
    gl = Layer(gpu_ctx, 0.05, max_blocks=64)
    with pytest.raises(capi.CgError) as e:
        TsdfIntegrator(fast, gl).integratePointCloud(T, p, c)
    assert e.value.status == capi.CG_ERR_UNSUPPORTED
    gl.close()


def test_device_pointer_inputs(gpu_ctx):
    import torch
    from coxgraph_b200 import Layer, TsdfIntegrator
    _, gcfg = util.make_cfgs()
    (T, p, c), = util.small_frames(1, stride=8)
    a = Layer(gpu_ctx, 0.05, max_blocks=1024)
    b = Layer(gpu_ctx, 0.05, max_blocks=1024)
    TsdfIntegrator(gcfg, a).integratePointCloud(T, p, c)
    TsdfIntegrator(gcfg, b).integratePointCloud(T, torch.from_numpy(p).cuda(),
                                                torch.from_numpy(c).cuda())
    util.compare_layers(b.download(), a.download(), "device inputs", exact=True)
    a.close()
    b.close()


def test_upload_download_roundtrip(gpu_ctx):
    from coxgraph_b200 import Layer
    from oracle import oracle_py as orc
    ocfg, _ = util.make_cfgs()
    (T, p, c), = util.small_frames(1, stride=8)
    ol = orc.Layer(0.05)
    ol.integrate(ocfg, T, p, c)
    idx, vox, fl = ol.download()
    gl = Layer(gpu_ctx, 0.05, max_blocks=1024)
    perm = np.random.default_rng(0).permutation(len(idx))
    gl.upload(idx[perm], vox[perm], fl[perm])
    util.compare_layers(gl.download(), (idx, vox, fl), "roundtrip", exact=True, check_flags=True)
    assert np.array_equal(gl.block_indices(), idx)
    gl.close()


def test_prepared_jobs_equal_plain_calls(gpu_ctx):
    """cg_prepare_batch_device / cg_integrate_prepared: the first half of job k+1 is queued (second
    stream, own scratch set) before job k is completed.  Same layer, bit for bit, as the plain
    cg_integrate_batch_device calls; a job the fast path cannot take (a point outside the
    bundle-key box) silently goes the plain way."""
    _prepared_vs_plain(gpu_ctx)


@pytest.mark.parametrize("over", [{"method": 0}, {"enable_anti_grazing": 1}],
                         ids=["simple", "merged_anti_grazing"])
def test_prepared_jobs_equal_plain_calls_other_configs(gpu_ctx, over):
    """The same for the SIMPLE integrator and for the merged one with anti-grazing: the prepared
    path then queues a front half without bundles, or one that also builds the grazing set."""
    _prepared_vs_plain(gpu_ctx, **over)


@pytest.mark.parametrize("way", ["fast", "groups", "other_voxel_size"])
def test_prepared_staged_jobs_equal_plain_calls(gpu_ctx, monkeypatch, way):
    """cg_prepare_batch_staged: the inputs come from cg_stage_batch_async's copy stream.  "fast":
    the queued front half waits for the copy.  "groups" (CG_MAX_GROUP_POINTS below the job) and
    "other_voxel_size" (integrated through a second integrator whose layer has another voxel size,
    so the queued front half is dropped) run the job the plain way on the context's stream, which
    must wait for the copy too.  The slot first holds cloud X, which is integrated; then cloud Y
    (same point count: nothing is reallocated, so a read that does not wait sees X's points, which
    are valid points) — 25 full frames, long enough a copy for an unordered read to overtake it —
    is staged, prepared and integrated at once.  The layer must be a plain integrateBatch of Y."""
    _staged_vs_plain(gpu_ctx, monkeypatch, way)


def _staged_vs_plain(gpu_ctx, monkeypatch, way):
    import torch
    from coxgraph_b200 import Layer, TsdfIntegrator
    _, gcfg = util.make_cfgs()
    clouds = []
    for robot, submap in ((0, 0), (1, 2)):  # X, Y
        frames = util.small_frames(25, stride=1, robot=robot, submap=submap)
        poses = np.stack([T for (T, _, _) in frames]).astype(np.float32)
        p = torch.from_numpy(np.concatenate([p for (_, p, _) in frames])).pin_memory().numpy()
        c = torch.from_numpy(np.concatenate([c for (_, _, c) in frames])).pin_memory().numpy()
        offs = np.cumsum([0] + [len(p_) for (_, p_, _) in frames]).astype(np.uint64)
        clouds.append((poses, p, c, offs))
    (px, xp, xc, xo), (py, yp, yc, yo) = clouds
    assert len(xp) == len(yp)
    if way == "groups":
        monkeypatch.setenv("CG_MAX_GROUP_POINTS", str(int(yo[-1]) // 3))
    vs = 0.1 if way == "other_voxel_size" else 0.05
    scratch = Layer(gpu_ctx, 0.05, max_blocks=16384)
    ix = TsdfIntegrator(gcfg, scratch)
    ix.stageBatch(0, xp, xc)
    ix.integrateStaged(0, px, xo)
    target, ref = Layer(gpu_ctx, vs, max_blocks=16384), Layer(gpu_ctx, vs, max_blocks=16384)
    it = TsdfIntegrator(gcfg, target)
    prep = ix if way == "other_voxel_size" else it  # the slots belong to the context
    prep.stageBatch(0, yp, yc)
    prep.prepareStaged(1, 0, py, yo)
    st = it.integratePrepared(1)
    assert st.points_in == int(yo[-1]) and st.rays > 0
    TsdfIntegrator(gcfg, ref).integrateBatch(py, yp, yc, yo)
    util.compare_layers(target.download(), ref.download(), f"staged job ({way}) vs plain", exact=True)
    for L in (scratch, target, ref):
        L.close()


def _prepared_vs_plain(gpu_ctx, **over):
    import torch
    from coxgraph_b200 import Layer, TsdfIntegrator
    _, gcfg = util.make_cfgs(**over)
    dev = torch.device("cuda", 0)
    jobs = []
    for k in range(4):
        frames = util.small_frames(3, stride=4, robot=k % 2, submap=k)
        if k == 2:   # a stray far return: outside the key box measured so far
            T, p, c = frames[1]
            p = p.copy()
            p[5] = (0.4, 0.2, 90.0)
            frames[1] = (T, p, c)
        poses = np.stack([T for (T, _, _) in frames]).astype(np.float32)
        pts = torch.from_numpy(np.concatenate([p for (_, p, _) in frames])).to(dev)
        cols = torch.from_numpy(np.concatenate([c for (_, _, c) in frames])).to(dev)
        offs = np.cumsum([0] + [len(p) for (_, p, _) in frames]).astype(np.uint64)
        jobs.append((poses, pts, cols, offs))
    a, b = Layer(gpu_ctx, 0.05, max_blocks=4096), Layer(gpu_ctx, 0.05, max_blocks=4096)
    ia, ib = TsdfIntegrator(gcfg, a), TsdfIntegrator(gcfg, b)
    for (poses, pts, cols, offs) in jobs:
        ia.integrateBatch(poses, pts, cols, offs)
    ib.prepareBatch(0, *jobs[0])
    for k, job in enumerate(jobs):
        if k + 1 < len(jobs):
            ib.prepareBatch((k + 1) % 2, *jobs[k + 1])
        st = ib.integratePrepared(k % 2)
        assert st.points_in == int(job[3][-1]) and st.rays > 0
    util.compare_layers(a.download(), b.download(), "prepared vs plain jobs", exact=True)
    with pytest.raises(Exception):
        ib.integratePrepared(0)   # nothing prepared any more
    a.close()
    b.close()
