"""cg_reproject_submaps_sharded against the sequence it stands for: cg_layer_clear(owned) +
cg_project_submaps_sharded under the effective poses.  Every check is an exact comparison of both
layers (block set, voxel bits, has_data and updated flags) with that sequence run into fresh layers
of a second context.  On one GPU the communicator has one rank; with >= 2 GPUs
scripts/multigpu_reproject_check.py compares every rank's layers the same way."""
import ctypes as C
import os
import subprocess
import sys

import numpy as np
import pytest

from tests import util

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))

pytestmark = pytest.mark.gpu

MAX_BLOCKS = 16384
EPS = dict(eps_translation=1e-3, eps_rotation=1e-4)


def _comm_context():
    from coxgraph_b200.api import Context, commInit, commUniqueId
    ctx = Context(0)
    commInit(ctx, commUniqueId(), 0, 1)
    return ctx


@pytest.fixture(scope="module")
def ctxs():
    import torch  # noqa: F401  (loads the libnccl.so.2 the library binds to)
    a, b = _comm_context(), _comm_context()
    yield a, b
    a.close()
    b.close()


@pytest.fixture(params=["block_by_block", "default"])
def mode(request, monkeypatch):
    if request.param == "block_by_block":
        monkeypatch.setenv("CG_REPROJECT_FULL_FRACTION", "2")
    return request.param


def _submaps(ctx, count):
    import torch
    from coxgraph_b200 import Layer, TsdfIntegrator, TsdfIntegratorConfig, synth
    cfg = TsdfIntegratorConfig(use_const_weight=1, method=1, default_truncation_distance=0.16)
    out = []
    for k in range(count):
        L = Layer(ctx, 0.05, max_blocks=2048)
        integ = TsdfIntegrator(cfg, L)
        for (T, pts, cols) in synth.submap_frames(k % 2, k, 2, device=torch.device("cuda", 0),
                                                  stride=4):
            integ.integratePointCloud(T, pts, cols)
        out.append(L)
    return out


def _copy(layer, ctx):
    from coxgraph_b200 import Layer
    L = Layer(ctx, 0.05, max_blocks=2048)
    L.upload(*layer.download())
    return L


class Scene:
    """The submaps in the context under test and a copy of them in the reference context."""

    def __init__(self, ctxs, count):
        from coxgraph_b200 import Layer
        self.ctx, self.ref_ctx = ctxs
        self.subs = _submaps(self.ctx, count)
        self.ref_subs = [_copy(L, self.ref_ctx) for L in self.subs]
        self.partial = Layer(self.ctx, 0.05, max_blocks=MAX_BLOCKS)
        self.owned = Layer(self.ctx, 0.05, max_blocks=MAX_BLOCKS)

    def project(self, ids, poses):
        from coxgraph_b200.api import getProjectedMapSharded
        self.owned.clear()
        getProjectedMapSharded([self.subs[i] for i in ids], poses, self.partial, self.owned)

    def reproject(self, ids, poses_old, poses_new, **kw):
        from coxgraph_b200.api import reprojectSubmapsSharded
        return reprojectSubmapsSharded([self.subs[i] for i in ids], poses_old, poses_new,
                                       self.partial, self.owned, **kw)

    def reference(self, ids, poses):
        from coxgraph_b200 import Layer
        from coxgraph_b200.api import getProjectedMapSharded
        P = Layer(self.ref_ctx, 0.05, max_blocks=MAX_BLOCKS)
        O = Layer(self.ref_ctx, 0.05, max_blocks=MAX_BLOCKS)
        getProjectedMapSharded([self.ref_subs[i] for i in ids], poses, P, O)
        out = P.download(), O.download()
        P.close()
        O.close()
        return out

    def check(self, ids, poses, what):
        want_p, want_o = self.reference(ids, poses)
        util.compare_layers(self.owned.download(), want_o, what + ": owned", exact=True,
                            check_flags=True)
        util.compare_layers(self.partial.download(), want_p, what + ": partial", exact=True,
                            check_flags=True)

    def close(self):
        for L in self.subs + self.ref_subs + [self.partial, self.owned]:
            L.close()


def _poses(rng, ids):
    from coxgraph_b200 import synth
    return np.stack([synth.perturb_pose(synth.robot_map_offset(i % 2), rng, sigma_t=0.4,
                                        sigma_yaw_deg=25.0) for i in ids])


def _same_bytes(a, b):
    return all(np.array_equal(x.view(np.uint8), y.view(np.uint8)) for x, y in zip(a, b))


def test_chained_moves_far_move_and_eps(ctxs, mode, monkeypatch):
    from coxgraph_b200 import synth
    sc = Scene(ctxs, 6)
    ids = [k % 6 for k in range(12)]
    rng = np.random.default_rng(7)
    cur = _poses(rng, ids)
    sc.project(ids, cur)
    # nothing moved and nothing added: both layers byte-identical, flags included
    before = sc.owned.download(), sc.partial.download()
    changed, st = sc.reproject(ids, cur, cur)
    assert not changed.any() and st.submaps_moved == st.submaps_added == st.blocks_dirty == 0
    util.compare_layers(sc.owned.download(), before[0], "unchanged: owned", exact=True, check_flags=True)
    util.compare_layers(sc.partial.download(), before[1], "unchanged: partial", exact=True,
                        check_flags=True)
    for step in range(3):
        new = cur.copy()
        moved = rng.choice(len(ids), 3, replace=False)
        for k in moved:
            new[k] = synth.perturb_pose(cur[k], rng, sigma_t=0.05, sigma_yaw_deg=1.0)
        still = int(np.setdiff1d(np.arange(len(ids)), moved)[0])
        new[still, 4] += 1e-4  # below eps_translation: not moved
        changed, st = sc.reproject(ids, cur, new, **EPS)
        assert np.array_equal(np.flatnonzero(changed), np.sort(moved)), f"step {step}"
        assert st.submaps_moved == 3 and st.submaps_added == 0 and st.blocks_dirty > 0
        if mode == "block_by_block":
            assert st.full_rebuild == 0 and st.blocks_folded > 0
        cur = np.where(changed[:, None], new, cur)
        sc.check(ids, cur, f"{mode} step {step}")
    # one submap moves far away from everything: its blocks leave both layers (the dirty set is
    # then about twice the map: a fraction above that keeps the block-by-block path)
    if mode == "block_by_block":
        monkeypatch.setenv("CG_REPROJECT_FULL_FRACTION", "1e9")
    only = np.array([[1, 0, 0, 0, 0, 0, 0]], np.float32)
    sc.project([0], only)
    n0 = sc.owned.num_blocks
    away = only.copy()
    away[0, 4:7] = (80.0, 80.0, 0.0)
    changed, st = sc.reproject([0], only, away)
    assert changed.all() and sc.owned.num_blocks > 0
    if mode == "block_by_block":
        assert st.full_rebuild == 0 and st.blocks_removed == n0
        assert st.blocks_folded == sc.owned.num_blocks
    sc.check([0], away, f"{mode} far move")
    sc.close()


def test_appended_submaps(ctxs, mode):
    from coxgraph_b200 import synth
    sc = Scene(ctxs, 6)
    rng = np.random.default_rng(11)
    ids = [0, 1, 2]
    cur = _poses(rng, ids)
    sc.project(ids, cur)
    # appended alone
    ids2 = ids + [3]
    new = np.concatenate([cur, _poses(rng, [3])])
    changed, st = sc.reproject(ids2, cur, new)
    assert list(changed) == [False, False, False, True]
    assert st.submaps_added == 1 and st.submaps_moved == 0 and st.blocks_dirty_local > 0
    sc.check(ids2, new, f"{mode} appended")
    cur = new
    # appended together with moved ones
    ids3 = ids2 + [4, 5]
    new = np.concatenate([cur, _poses(rng, [4, 5])])
    new[1] = synth.perturb_pose(cur[1], rng, sigma_t=0.1, sigma_yaw_deg=2.0)
    changed, st = sc.reproject(ids3, cur, new, **EPS)
    assert list(np.flatnonzero(changed)) == [1, 4, 5]
    assert st.submaps_added == 2 and st.submaps_moved == 1
    sc.check(ids3, new, f"{mode} appended and moved")
    sc.close()


def test_only_updated_after_reset(ctxs, mode):
    from coxgraph_b200 import synth
    from coxgraph_b200.api import generateMeshSharded
    sc = Scene(ctxs, 6)
    ids = [k % 6 for k in range(12)]
    rng = np.random.default_rng(3)
    cur = _poses(rng, ids)
    sc.project(ids, cur)
    sc.owned.resetUpdated()
    bi, bv, _ = sc.owned.download()
    new = cur.copy()
    new[5] = synth.perturb_pose(cur[5], rng, sigma_t=0.05, sigma_yaw_deg=1.0)
    changed, st = sc.reproject(ids, cur, new)
    ai, av, af = sc.owned.download()
    updated = (af & 2) != 0
    if mode == "block_by_block":
        assert st.full_rebuild == 0
        assert 0 < updated.sum() <= st.blocks_dirty < len(ai)
        # every block whose bits changed (or that is new) carries the flag
        old = {tuple(b): k for k, b in enumerate(bi)}
        for k, b in enumerate(ai):
            j = old.get(tuple(b))
            if j is None or not (np.array_equal(av[k]["distance"].view(np.uint32),
                                                bv[j]["distance"].view(np.uint32))
                                 and np.array_equal(av[k]["weight"].view(np.uint32),
                                                    bv[j]["weight"].view(np.uint32))
                                 and np.array_equal(av[k]["rgba"], bv[j]["rgba"])):
                assert updated[k], f"block {b} changed without the updated flag"
    else:
        assert updated.sum() > 0
    got = generateMeshSharded(sc.owned, only_updated=True)
    ref = sc.owned.generateMesh(only_updated=True)
    assert _same_bytes(got, ref)
    assert 0 < len(got[2])
    if mode == "block_by_block":
        assert len(got[2]) < len(sc.owned.generateMesh()[2])
    sc.close()


def _raw(sc, subs, n, num_known, po, pn, partial=None, owned=None):
    from coxgraph_b200 import capi
    arr = (C.c_void_p * max(len(subs), 1))(*[s._h if s is not None else None for s in subs])
    st = capi.ReprojectShardedStats()
    return capi.load().cg_reproject_submaps_sharded(
        arr, n, num_known, po, pn, 0.0, 0.0, (partial or sc.partial)._h, (owned or sc.owned)._h,
        None, C.byref(st))


def test_rejections_leave_the_layers_untouched(ctxs):
    from coxgraph_b200 import Context, Layer, capi, synth
    from coxgraph_b200.api import reprojectSubmapsSharded
    sc = Scene(ctxs, 3)
    ids = [0, 1]
    rng = np.random.default_rng(5)
    cur = _poses(rng, ids)
    sc.project(ids, cur)
    subs = [sc.subs[i] for i in ids]
    P = np.ascontiguousarray(cur, np.float32)
    p = P.ctypes.data_as(C.c_void_p)
    snapshot = sc.owned.download(), sc.partial.download()

    def untouched(what):
        util.compare_layers(sc.owned.download(), snapshot[0], what + ": owned", exact=True,
                            check_flags=True)
        util.compare_layers(sc.partial.download(), snapshot[1], what + ": partial", exact=True,
                            check_flags=True)

    step = [0]

    def then_succeeds(what):
        nonlocal cur, snapshot, P, p
        new = cur.copy()
        new[step[0] % 2] = synth.perturb_pose(cur[step[0] % 2], rng, sigma_t=0.05, sigma_yaw_deg=1.0)
        step[0] += 1
        changed, _ = sc.reproject(ids, cur, new)
        assert changed.any()
        cur = new
        sc.check(ids, cur, "after " + what)
        snapshot = sc.owned.download(), sc.partial.download()
        P = np.ascontiguousarray(cur, np.float32)
        p = P.ctypes.data_as(C.c_void_p)

    def rejected(rc, needle, what):
        assert rc == capi.CG_ERR_INVALID_ARG, f"{what}: status {rc}"
        msg = capi.load().cg_last_error().decode()
        assert needle in msg, f"{what}: {msg}"
        untouched(what)
        then_succeeds(what)

    rejected(_raw(sc, subs, 2, 3, p, p), "num_known", "num_known > n")
    rejected(_raw(sc, subs, 2, 2, None, p), "null", "null poses_old")
    rejected(_raw(sc, subs, 2, 2, p, None), "null", "null poses_new")
    rejected(_raw(sc, [subs[0], None], 2, 2, p, p), "submap 1", "null submap")
    rejected(_raw(sc, [subs[0], sc.partial], 2, 2, p, p), "submap 1", "submap is partial")
    rejected(_raw(sc, [sc.owned, subs[1]], 2, 2, p, p), "submap 0 is the owned", "submap is owned")
    foreign = _copy(subs[1], sc.ref_ctx)
    rejected(_raw(sc, [subs[0], foreign], 2, 2, p, p), "submap 1", "submap of another context")
    other = Layer(sc.ctx, 0.05, max_blocks=MAX_BLOCKS)
    rejected(_raw(sc, subs, 2, 2, p, p, partial=other), "partial layer of the last",
             "partial not bound")
    # no communicator
    lone = Context(0)
    A, B = Layer(lone, 0.05, max_blocks=64), Layer(lone, 0.05, max_blocks=64)
    with pytest.raises(capi.CgError) as e:
        reprojectSubmapsSharded([], np.zeros((0, 7)), np.zeros((0, 7)), A, B)
    assert e.value.status == capi.CG_ERR_INVALID_ARG and "cg_comm_init" in str(e.value)
    untouched("no communicator")
    then_succeeds("no communicator")
    for L in (A, B, other, foreign):
        L.close()
    lone.close()
    sc.close()


@pytest.mark.gpu
def test_sharded_reprojection_over_nccl():
    import torch
    n = torch.cuda.device_count()
    if n < 2:
        pytest.skip("needs at least 2 GPUs")
    world = 4 if n >= 4 else 2
    r = subprocess.run([sys.executable, "-m", "torch.distributed.run", "--nnodes=1",
                        f"--nproc-per-node={world}", "--master-addr", "127.0.0.1",
                        "--master-port", "29547",
                        os.path.join(ROOT, "scripts", "multigpu_reproject_check.py")],
                       capture_output=True, text=True, timeout=1500)
    assert r.returncode == 0 and "multigpu_reproject_check ok" in r.stdout, \
        r.stdout[-3000:] + r.stderr[-3000:]
