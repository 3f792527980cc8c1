"""Edge-case parity of the CUDA integration path against the oracle on hand-built clouds (not
depth images): one giant bundle, thousands of updates on the same voxels (the long-list replay
and its closed form), points exactly on voxel faces, duplicates, non-finite and zero points,
rays along the axes, random poses.  Reference call site: tsdf_recover.h:75."""
import numpy as np
import pytest

from tests import util

pytestmark = pytest.mark.gpu


def _pose(rng=None):
    if rng is None:
        return np.array([1, 0, 0, 0, 0.01, 0.02, 0.03], np.float32)
    q = rng.standard_normal(4)
    q /= np.linalg.norm(q)
    return np.concatenate([q, rng.uniform(-2, 2, 3)]).astype(np.float32)


def _colors(n, rng):
    c = rng.integers(0, 256, (n, 4), dtype=np.uint8)
    c[:, 3] = 255
    return c


def _compare(gpu_ctx, frames, batch, max_blocks=4096, **cfg):
    from coxgraph_b200 import Layer, TsdfIntegrator
    from oracle import oracle_py as orc
    ocfg, gcfg = util.make_cfgs(**cfg)
    ol, gl = orc.Layer(0.05), Layer(gpu_ctx, 0.05, max_blocks=max_blocks)
    for (T, p, c) in frames:
        ol.integrate(ocfg, T, p, c)
    integ = TsdfIntegrator(gcfg, gl)
    if batch:
        offs = np.cumsum([0] + [len(p) for (_, p, _) in frames]).astype(np.uint64)
        st = integ.integrateBatch(np.stack([T for (T, _, _) in frames]),
                                  np.concatenate([p for (_, p, _) in frames]),
                                  np.concatenate([c for (_, _, c) in frames]), offs)
    else:
        for (T, p, c) in frames:
            st = integ.integratePointCloud(T, p, c)
    util.compare_layers(gl.download(), ol.download(), "edge case")
    gl.close()
    return st


def test_one_giant_bundle(gpu_ctx):
    """6000 points inside one voxel: a single sequential fold of 6000 steps."""
    rng = np.random.default_rng(3)
    p = (np.array([0.52, 0.27, 1.51]) + rng.uniform(0, 0.045, (6000, 3))).astype(np.float32)
    st = _compare(gpu_ctx, [(_pose(), p, _colors(len(p), rng))], batch=False, use_const_weight=0)
    assert st.rays <= 8


@pytest.mark.parametrize("carving", [1, 0])
def test_thousands_of_updates_per_voxel(gpu_ctx, carving):
    """300 frames of the same small cluster from the same pose, all in one job: the free-space
    voxels near the sensor get > 2048 updates (the fixed-point sum), the band ones up to about
    1400 (the warp replay).  Band lists of 2048 or more are in test_gpu_update_paths.py; the
    closed form of k_long_finish is never reached (DESIGN §4.2)."""
    rng = np.random.default_rng(5)
    base = np.array([0.3, -0.2, 1.4])
    frames = []
    for f in range(300):
        p = (base + rng.uniform(-0.08, 0.08, (40, 3))).astype(np.float32)
        frames.append((_pose(), p, _colors(len(p), rng)))
    st = _compare(gpu_ctx, frames, batch=True, voxel_carving_enabled=carving,
                  default_truncation_distance=0.16)
    assert st.voxel_updates > (100_000 if carving else 20_000)


def test_degenerate_points_and_exact_faces(gpu_ctx):
    rng = np.random.default_rng(7)
    grid = np.stack(np.meshgrid(np.arange(-6, 7), np.arange(-6, 7), [20, 30, 40]), -1).reshape(-1, 3)
    on_faces = (grid * 0.05).astype(np.float32)                  # coordinates exactly k * 0.05
    axis = np.array([[0, 0, 2.0], [0, 1.5, 0], [1.25, 0, 0], [0, 0, -1.0], [-0.75, 0, 0]], np.float32)
    dup = np.repeat(np.array([[0.4, 0.4, 2.2]], np.float32), 300, axis=0)
    junk = np.array([[np.nan, 0, 1], [0, np.inf, 1], [0, 0, 0], [0.01, 0.0, 0.02],
                     [0, 0, 7.5], [3, 4, 50.0], [1e-4, 0, 5.0001]], np.float32)
    p = np.concatenate([on_faces, axis, dup, junk, rng.normal(0, 1.2, (500, 3)).astype(np.float32)])
    c = _colors(len(p), rng)
    T = np.array([1, 0, 0, 0, 0, 0, 0], np.float32)              # origin exactly on a voxel corner
    for over in (dict(), dict(use_const_weight=0, allow_clear=0), dict(voxel_carving_enabled=0),
                 dict(method=0)):
        _compare(gpu_ctx, [(T, p, c)], batch=False, **over)


@pytest.mark.parametrize("seed", [11, 12, 13])
def test_random_clouds_random_poses(gpu_ctx, seed):
    rng = np.random.default_rng(seed)
    frames = []
    for f in range(4):
        n = int(rng.integers(200, 3000))
        d = rng.standard_normal((n, 3))
        d /= np.linalg.norm(d, axis=1, keepdims=True)
        p = (d * rng.uniform(0.05, 7.0, (n, 1))).astype(np.float32)   # below min_ray .. beyond max_ray
        frames.append((_pose(rng), p, _colors(n, rng)))
    _compare(gpu_ctx, frames, batch=bool(seed & 1), use_const_weight=int(seed % 3 == 0),
             max_weight=50.0 if seed == 13 else 10000.0)


def test_bundle_key_box_grows_and_shrinks(monkeypatch):
    """The bundle keys cover a per-axis box of voxels around the sensor that the context learns
    from its jobs: a fresh context, jobs whose extent grows step by step (every growth is a redo
    of the group with the measured extent), one far outlier, then enough ordinary jobs for the
    window over the last 8 measured jobs to shrink the box again.  Every result must match the
    oracle whatever box was in force."""
    from coxgraph_b200 import Context, Layer, TsdfIntegrator, synth
    from oracle import oracle_py as orc
    monkeypatch.setenv("CG_KEY_MEASURE_PERIOD", "1")   # measure on every job: the window fills fast
    ctx = Context(0)
    ocfg, gcfg = util.make_cfgs()
    rng = np.random.default_rng(5)
    T = synth.camera_pose((0.3, -0.2, 1.1), yaw=0.4)
    gl, ol = Layer(ctx, 0.05, max_blocks=8192), orc.Layer(0.05)
    integ = TsdfIntegrator(gcfg, gl)
    reach = [0.6, 1.0, 1.8, 3.0, 4.5, 4.5]            # metres: the cloud's extent per job
    reach += [60.0]                                   # one stray far return (a clearing ray)
    reach += [1.5] * 12                               # back to ordinary clouds: the box shrinks
    for k, r in enumerate(reach):
        n = 4000
        p = rng.uniform(-1, 1, (n, 3)).astype(np.float32) * np.float32(min(r, 4.5))
        p[:, 2] = np.abs(p[:, 2]) + 0.3
        if r > 10:
            p[17] = (0.2, -0.1, r)
        c = rng.integers(0, 256, (n, 4), dtype=np.uint8)
        for batch in (False, True):                   # single frame, then the same cloud in a batch
            if batch:
                integ.integrateBatch(np.stack([T, T]), np.concatenate([p, p]), np.concatenate([c, c]),
                                     np.array([0, n, 2 * n], np.uint64))
                ol.integrate(ocfg, T, p, c)
                ol.integrate(ocfg, T, p, c)
            else:
                integ.integratePointCloud(T, p, c)
                ol.integrate(ocfg, T, p, c)
        util.compare_layers(gl.download(), ol.download(), f"job {k} (reach {r} m)")
    gl.close()
    ctx.close()


def test_listed_blocks_download_and_hash_stats(gpu_ctx):
    """cg_layer_download_blocks returns exactly what cg_layer_download holds for the listed
    indices and flags the ones that are not allocated; cg_layer_hash_stats reports the occupancy
    of the block hash."""
    from coxgraph_b200 import Layer, TsdfIntegrator
    _, gcfg = util.make_cfgs()
    gl = Layer(gpu_ctx, 0.05, max_blocks=2048)
    integ = TsdfIntegrator(gcfg, gl)
    for (T, p, c) in util.small_frames(2, stride=8):
        integ.integratePointCloud(T, p, c)
    idx, vox, flags = gl.download()
    pick = idx[::3]
    missing = np.array([[1000, 1000, 1000], [-999, 5, 7]], np.int32)
    ask = np.concatenate([pick[:5], missing, pick[5:]])
    v, f, found = gl.download_blocks(ask)
    assert found.tolist() == [True] * 5 + [False, False] + [True] * (len(pick) - 5)
    got = np.concatenate([v[:5], v[7:]])
    ref = vox[::3]
    for name in ("distance", "weight"):
        assert np.array_equal(got[name].view(np.uint32), ref[name].view(np.uint32))
    assert np.array_equal(got["rgba"], ref["rgba"])
    assert np.array_equal(np.concatenate([f[:5], f[7:]]), flags[::3])
    st = gl.hash_stats()
    assert st.num_blocks == len(idx) and st.hash_capacity >= 2 * gl.max_blocks
    assert 0 < st.load_factor < 0.5 and 1.0 <= st.mean_probe_length < 2.0
    assert st.max_probe_length >= 1
    gl.close()
