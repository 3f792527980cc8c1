"""Depth-image integration (cg_integrate_depth_*) against the cloud path: every depth job must leave
the layer bit-identical, flags and stats included, to cg_integrate_batch_device on the cloud
depth_image_proc + TsdfServer would build from the same images (tests/depth_reference.py)."""
import numpy as np
import pytest

from tests import depth_reference as ref
from tests import util

pytestmark = pytest.mark.gpu

STATS = ("points_in", "rays", "voxel_updates", "general_updates", "blocks_touched",
         "blocks_allocated", "points_beyond_reach")


def _images(F, enc="16UC1", stride=4, robot=0, submap=0, masks=None, seed=0):
    """F synthetic frames as registered images; masks[f] in {None, "random", "rows", "edge",
    "none_valid", "all_valid", "one_valid"} invalidates pixels (0 / NaN)."""
    from coxgraph_b200 import synth
    poses = synth.trajectory(F, robot=robot, submap=submap)
    rng = np.random.default_rng(seed)
    depth, rgb, cam = [], [], None
    for f in range(F):
        d, c, cam = synth.render_depth_frame(poses[f], stride=stride, depth_encoding=enc)
        m = (masks or [None] * F)[f]
        bad = np.zeros(d.shape, bool)
        if m == "random":
            bad = rng.random(d.shape) < 0.1
        elif m == "rows":
            bad[::7] = True
        elif m == "edge":
            bad[:, :5] = True
            bad[-3:, :] = True
        elif m == "none_valid":
            bad[:] = True
        elif m == "one_valid":
            bad[:] = True
            bad[d.shape[0] // 2, d.shape[1] // 3] = False
        d = d.copy()
        d[bad] = 0 if enc == "16UC1" else np.nan
        depth.append(d)
        rgb.append(c)
    return poses.astype(np.float32), np.stack(depth), np.stack(rgb), cam


def _encode_color(rgb, encoding):
    """rgb8 [F,H,W,3] -> the same colours in `encoding`."""
    if encoding == "rgb8":
        return rgb
    if encoding == "bgr8":
        return np.ascontiguousarray(rgb[..., ::-1])
    if encoding == "rgba8":
        return np.concatenate([rgb, np.full(rgb.shape[:-1] + (1,), 77, np.uint8)], -1)
    if encoding == "bgra8":
        return np.concatenate([rgb[..., ::-1], np.full(rgb.shape[:-1] + (1,), 77, np.uint8)], -1)
    return np.ascontiguousarray(rgb[..., 1:2])  # mono8


def _cloud_layer(ctx, gcfg, poses, pts, cols, offs, voxel_size=0.05):
    import torch
    from coxgraph_b200 import Layer, TsdfIntegrator
    L = Layer(ctx, voxel_size, max_blocks=16384)
    it = TsdfIntegrator(gcfg, L)
    dev = torch.device("cuda", 0)
    st = it.integrateBatch(poses, torch.from_numpy(pts).to(dev), torch.from_numpy(cols).to(dev), offs)
    return L, {k: getattr(st, k) for k in STATS}


def _depth_vs_cloud(ctx, poses, depth, color, cam, oracle=True, **over):
    from coxgraph_b200 import Layer, TsdfIntegrator
    ocfg, gcfg = util.make_cfgs(**over)
    pts, cols, offs = ref.depth_batch_cloud(depth, color, cam)
    cl, cst = _cloud_layer(ctx, gcfg, poses, pts, cols, offs)
    dl = Layer(ctx, 0.05, max_blocks=16384)
    st = TsdfIntegrator(gcfg, dl).integrateDepthBatch(poses, depth, color, cam)
    dst = {k: getattr(st, k) for k in STATS}
    got = dl.download()
    util.compare_layers(got, cl.download(), "depth vs cloud", exact=True, check_flags=True)
    assert dst == cst, (dst, cst)
    assert dst["points_in"] == int(offs[-1])
    if oracle:
        from oracle import oracle_py as orc
        ol = orc.Layer(0.05)
        for f in range(len(poses)):
            ol.integrate(ocfg, poses[f], pts[offs[f]:offs[f + 1]], cols[offs[f]:offs[f + 1]])
        util.compare_layers(got, ol.download(), "depth vs oracle")
    dl.close()
    cl.close()


@pytest.mark.parametrize("enc", ["16UC1", "32FC1"])
@pytest.mark.parametrize("order", [0, 1])
@pytest.mark.parametrize("method", [1, 0])
def test_depth_equals_cloud_path(gpu_ctx, method, order, enc):
    poses, depth, rgb, cam = _images(3, enc, masks=["random", "rows", "edge"], seed=method * 2 + order)
    _depth_vs_cloud(gpu_ctx, poses, depth, rgb, cam, method=method, integration_order_mode=order)


@pytest.mark.parametrize("encoding", ["rgb8", "rgba8", "bgr8", "bgra8", "mono8"])
def test_every_color_encoding(gpu_ctx, encoding):
    poses, depth, rgb, cam = _images(2, masks=["random", None], seed=3)
    cam = dict(cam, color_encoding=encoding)
    _depth_vs_cloud(gpu_ctx, poses, depth, _encode_color(rgb, encoding), cam, oracle=False)


def test_anti_grazing(gpu_ctx):
    poses, depth, rgb, cam = _images(2, "32FC1", masks=["random", "edge"], seed=4)
    _depth_vs_cloud(gpu_ctx, poses, depth, rgb, cam, enable_anti_grazing=1)


@pytest.mark.parametrize("method", [1, 0])
def test_ragged_frames_in_one_job(gpu_ctx, method):
    """A frame with no valid pixel, one with every pixel valid, one with a single valid pixel, and
    ragged masks, in one job."""
    masks = ["none_valid", "all_valid", "one_valid", "random", "rows", "edge", "none_valid"]
    poses, depth, rgb, cam = _images(len(masks), masks=masks, seed=5)
    _depth_vs_cloud(gpu_ctx, poses, depth, rgb, cam, method=method)


def test_guard_dropping_differs_from_nan_points(gpu_ctx):
    """On this scene the contract (invalid pixels dropped) and the NaN-keeping cloud give different
    layers through the cloud path, so the tests above would catch an implementation that keeps
    the invalid pixels as NaN points."""
    _, gcfg = util.make_cfgs()
    poses, depth, rgb, cam = _images(3, masks=["random", "rows", "edge"], seed=0)
    a = _cloud_layer(gpu_ctx, gcfg, poses, *ref.depth_batch_cloud(depth, rgb, cam))[0]
    b = _cloud_layer(gpu_ctx, gcfg, poses, *ref.depth_batch_cloud(depth, rgb, cam, form="nan"))[0]
    with pytest.raises(AssertionError):
        util.compare_layers(a.download(), b.download(), "guard", exact=True)
    a.close()
    b.close()


@pytest.mark.parametrize("path", ["groups", "pairs"])
def test_driver_paths(gpu_ctx, monkeypatch, path):
    poses, depth, rgb, cam = _images(5, masks=["random", "all_valid", "rows", "edge", "one_valid"],
                                     seed=6)
    if path == "groups":
        monkeypatch.setenv("CG_MAX_GROUP_POINTS", str(2 * cam["width"] * cam["height"]))
    else:
        monkeypatch.setenv("CG_MAX_PAIRS", "100000")
    _depth_vs_cloud(gpu_ctx, poses, depth, rgb, cam, oracle=False)


def test_key_box_retry(monkeypatch):
    """A far frame after a near job: the bundle-key box is exceeded and the group redone, on fresh
    contexts for both paths."""
    from coxgraph_b200 import Context, Layer, TsdfIntegrator
    monkeypatch.setenv("CG_KEY_MEASURE_PERIOD", "1")
    _, gcfg = util.make_cfgs()
    poses, depth, rgb, cam = _images(2, "32FC1", masks=["random", None], seed=8)
    near = depth * np.float32(0.3)
    far = depth.copy()
    far[1, 10, 10] = np.float32(60.0)
    layers = []
    for kind in ("depth", "cloud"):
        ctx = Context(0)
        L = Layer(ctx, 0.05, max_blocks=16384)
        it = TsdfIntegrator(gcfg, L)
        for d in (near, far):
            if kind == "depth":
                it.integrateDepthBatch(poses, d, rgb, cam)
            else:
                import torch
                p, c, o = ref.depth_batch_cloud(d, rgb, cam)
                it.integrateBatch(poses, torch.from_numpy(p).cuda(), torch.from_numpy(c).cuda(), o)
        layers.append((L.download(), L, ctx))
    util.compare_layers(layers[0][0], layers[1][0], "key-box retry", exact=True, check_flags=True)
    for _, L, ctx in layers:
        L.close()
        ctx.close()


def _reference(ctx, gcfg, poses, depth, rgb, cam, voxel_size=0.05):
    L, st = _cloud_layer(ctx, gcfg, poses, *ref.depth_batch_cloud(depth, rgb, cam),
                         voxel_size=voxel_size)
    out = L.download()
    L.close()
    return out, st


def test_every_entry_point_gives_the_same_bits(gpu_ctx):
    import torch
    from coxgraph_b200 import Layer, TsdfIntegrator
    _, gcfg = util.make_cfgs()
    dev = torch.device("cuda", 0)
    poses, depth, rgb, cam = _images(4, masks=["random", "rows", None, "edge"], seed=9)
    want, want_st = _reference(gpu_ctx, gcfg, poses, depth, rgb, cam)
    pin = lambda a: torch.from_numpy(np.ascontiguousarray(a)).pin_memory().numpy()  # noqa: E731
    ways = ["pageable", "pinned", "device", "staged", "prepared_device", "prepared_staged"]
    for way in ways:
        L = Layer(gpu_ctx, 0.05, max_blocks=16384)
        it = TsdfIntegrator(gcfg, L)
        if way == "pageable":
            st = it.integrateDepthBatch(poses, depth, rgb, cam)
        elif way == "pinned":
            st = it.integrateDepthBatch(poses, pin(depth), pin(rgb), cam)
        elif way == "device":
            st = it.integrateDepthBatch(poses, torch.from_numpy(depth.view(np.int16)).to(dev),
                                        torch.from_numpy(rgb).to(dev), cam)
        elif way == "staged":
            it.stageDepth(1, pin(depth), pin(rgb), cam)
            st = it.integrateDepthStaged(1, poses, cam)
        elif way == "prepared_device":
            it.prepareDepth(0, poses, torch.from_numpy(depth.view(np.int16)).to(dev),
                            torch.from_numpy(rgb).to(dev), cam)
            st = it.integratePrepared(0)
        else:
            it.stageDepth(0, pin(depth), pin(rgb), cam)
            it.prepareDepthStaged(1, 0, poses, cam)
            st = it.integratePrepared(1)
        util.compare_layers(L.download(), want, way, exact=True, check_flags=True)
        assert {k: getattr(st, k) for k in STATS} == want_st, way
        L.close()


def test_pipelined_loop(gpu_ctx):
    """Six jobs: prepare k + 1, then integratePrepared k; the same layer as six plain calls."""
    import torch
    from coxgraph_b200 import Layer, TsdfIntegrator
    _, gcfg = util.make_cfgs()
    dev = torch.device("cuda", 0)
    jobs = []
    for k in range(6):
        poses, depth, rgb, cam = _images(2, robot=k % 2, submap=k, masks=["random", "rows"], seed=k)
        jobs.append((poses, torch.from_numpy(depth.view(np.int16)).to(dev),
                     torch.from_numpy(rgb).to(dev), cam, depth, rgb))
    a, b = Layer(gpu_ctx, 0.05, max_blocks=16384), Layer(gpu_ctx, 0.05, max_blocks=16384)
    ia, ib = TsdfIntegrator(gcfg, a), TsdfIntegrator(gcfg, b)
    for (poses, _, _, cam, depth, rgb) in jobs:
        p, c, o = ref.depth_batch_cloud(depth, rgb, cam)
        ia.integrateBatch(poses, torch.from_numpy(p).to(dev), torch.from_numpy(c).to(dev), o)
    ib.prepareDepth(0, *jobs[0][:4])
    for k in range(len(jobs)):
        if k + 1 < len(jobs):
            ib.prepareDepth((k + 1) % 2, *jobs[k + 1][:4])
        st = ib.integratePrepared(k % 2)
        assert st.points_in == int(ref.depth_batch_cloud(jobs[k][4], jobs[k][5], jobs[k][3])[2][-1])
    util.compare_layers(b.download(), a.download(), "pipelined depth", exact=True, check_flags=True)
    a.close()
    b.close()


@pytest.mark.parametrize("way", ["other_voxel_size", "groups"])
def test_prepared_fallbacks(gpu_ctx, monkeypatch, way):
    """A prepared depth job the fast path cannot take runs the plain way from the points kept in
    the prepare slot."""
    import torch
    from coxgraph_b200 import Layer, TsdfIntegrator
    _, gcfg = util.make_cfgs()
    dev = torch.device("cuda", 0)
    poses, depth, rgb, cam = _images(3, masks=["random", "edge", None], seed=11)
    vs = 0.1 if way == "other_voxel_size" else 0.05
    if way == "groups":
        monkeypatch.setenv("CG_MAX_GROUP_POINTS", str(cam["width"] * cam["height"]))
    want, want_st = _reference(gpu_ctx, gcfg, poses, depth, rgb, cam, voxel_size=vs)
    scratch = Layer(gpu_ctx, 0.05, max_blocks=16384)
    target = Layer(gpu_ctx, vs, max_blocks=16384)
    it = TsdfIntegrator(gcfg, target)
    prep = TsdfIntegrator(gcfg, scratch) if way == "other_voxel_size" else it
    prep.prepareDepth(0, poses, torch.from_numpy(depth.view(np.int16)).to(dev),
                      torch.from_numpy(rgb).to(dev), cam)
    st = it.integratePrepared(0)
    util.compare_layers(target.download(), want, way, exact=True, check_flags=True)
    assert {k: getattr(st, k) for k in STATS} == want_st
    scratch.close()
    target.close()


def test_stage_slot_kinds(gpu_ctx):
    """A depth job staged into a slot that last held a cloud; a cloud call on a depth slot fails."""
    import torch
    from coxgraph_b200 import Layer, TsdfIntegrator, capi
    _, gcfg = util.make_cfgs()
    poses, depth, rgb, cam = _images(2, masks=["random", None], seed=12)
    pts, cols, offs = ref.depth_batch_cloud(depth, rgb, cam)
    pin = lambda a: torch.from_numpy(np.ascontiguousarray(a)).pin_memory().numpy()  # noqa: E731
    want, _ = _reference(gpu_ctx, gcfg, poses, depth, rgb, cam)
    L = Layer(gpu_ctx, 0.05, max_blocks=16384)
    it = TsdfIntegrator(gcfg, L)
    it.stageBatch(0, pin(pts), pin(cols))
    it.stageDepth(0, pin(depth), pin(rgb), cam)   # replaces the cloud
    with pytest.raises(capi.CgError) as e:
        it.integrateStaged(0, poses, offs)
    assert e.value.status == capi.CG_ERR_INVALID_ARG
    with pytest.raises(capi.CgError) as e:
        it.prepareStaged(0, 0, poses, offs)
    assert e.value.status == capi.CG_ERR_INVALID_ARG
    assert L.num_blocks == 0
    it.integrateDepthStaged(0, poses, cam)
    util.compare_layers(L.download(), want, "depth staged over a cloud slot", exact=True,
                        check_flags=True)
    it.stageBatch(0, pin(pts), pin(cols))       # and back: a depth call on a cloud slot fails
    with pytest.raises(capi.CgError) as e:
        it.integrateDepthStaged(0, poses, cam)
    assert e.value.status == capi.CG_ERR_INVALID_ARG
    L.close()


def test_launch_budget(gpu_ctx):
    import torch
    from coxgraph_b200 import Layer, TsdfIntegrator
    _, gcfg = util.make_cfgs()
    poses, depth, rgb, cam = _images(3, masks=["random", "rows", None], seed=13)
    pts, cols, offs = ref.depth_batch_cloud(depth, rgb, cam)
    dev = torch.device("cuda", 0)
    counts = []
    for kind in ("cloud", "depth", "cloud", "depth"):  # warm: the second of each pair is counted
        L = Layer(gpu_ctx, 0.05, max_blocks=16384)
        it = TsdfIntegrator(gcfg, L)
        before = gpu_ctx.kernel_launches
        if kind == "cloud":
            it.integrateBatch(poses, torch.from_numpy(pts).to(dev), torch.from_numpy(cols).to(dev), offs)
        else:
            it.integrateDepthBatch(poses, depth, rgb, cam)
        counts.append(gpu_ctx.kernel_launches - before)
        L.close()
    assert counts[3] <= counts[2] + 2, counts


def test_argument_errors(gpu_ctx):
    import ctypes as C
    from coxgraph_b200 import Layer, TsdfIntegrator, capi, depthCamera
    _, gcfg = util.make_cfgs()
    poses, depth, rgb, cam = _images(1, seed=14)
    lib = capi.load()
    L = Layer(gpu_ctx, 0.05, max_blocks=4096)
    it = TsdfIntegrator(gcfg, L)
    it.integrateDepthBatch(poses, depth, rgb, cam)
    before = L.download()
    d = np.ascontiguousarray(depth)
    c = np.ascontiguousarray(rgb)
    P = np.ascontiguousarray(poses)
    st = capi.IntegrateStats()

    def call(cam_over=None, F=1, dptr=True, cptr=True, pptr=True, camp=True):
        k = depthCamera(dict(cam, **(cam_over or {})))
        return lib.cg_integrate_depth_batch(
            L._h, C.byref(gcfg), F, P.ctypes.data if pptr else None, C.byref(k) if camp else None,
            d.ctypes.data if dptr else None, c.ctypes.data if cptr else None, C.byref(st))
    bad = [dict(dptr=False), dict(cptr=False), dict(pptr=False), dict(camp=False), dict(F=0),
           dict(cam_over=dict(width=0)), dict(cam_over=dict(height=-3)),
           dict(cam_over=dict(depth_encoding=7)), dict(cam_over=dict(color_encoding=5)),
           dict(cam_over=dict(color_encoding=-1)), dict(cam_over=dict(fx=0.0)),
           dict(cam_over=dict(fy=-1.0)), dict(cam_over=dict(fx=float("nan"))),
           dict(cam_over=dict(fy=float("inf"))), dict(cam_over=dict(cx=float("nan"))),
           dict(cam_over=dict(cy=float("-inf"))),
           dict(cam_over=dict(width=1 << 16, height=1 << 15)), dict(F=1 << 20)]
    for b in bad:
        assert call(**b) == capi.CG_ERR_INVALID_ARG, b
        assert lib.cg_last_error().decode()
    k = depthCamera(cam)
    assert lib.cg_integrate_depth_batch_device(L._h, C.byref(gcfg), 1, P.ctypes.data, C.byref(k),
                                               None, None, C.byref(st)) == capi.CG_ERR_INVALID_ARG
    assert lib.cg_stage_depth_async(gpu_ctx._h, 2, C.byref(k), 1, d.ctypes.data,
                                    c.ctypes.data) == capi.CG_ERR_INVALID_ARG
    assert lib.cg_prepare_depth_device(L._h, C.byref(gcfg), 1, P.ctypes.data, C.byref(k), None,
                                       None, 0) == capi.CG_ERR_INVALID_ARG
    after = L.download()
    util.compare_layers(after, before, "after rejected calls", exact=True, check_flags=True)
    L.close()
