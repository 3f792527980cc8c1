"""GPU: cg_layer_esdf_update (EsdfIntegrator::updateFromTsdfLayer) against cg_layer_esdf_batch.

After every mutation the layer is copied into a second context, which runs the batch; the update
runs on the original context and must leave the same bits (block order, distances, packed words,
free points, whole-map totals).  The update's context is never re-based by a batch, so an error
would carry over the chain of mutations and be caught at a later step.  DESIGN §4.6 has the
argument that re-solving the blocks within R of a change is exact."""
import math

import numpy as np
import pytest

pytestmark = pytest.mark.gpu

VS = 0.05
FREE = 0.3


@pytest.fixture(scope="module")
def ref_ctx():
    from coxgraph_b200 import Context
    ctx = Context(0)
    yield ctx
    ctx.close()


def _cfg(**over):
    from coxgraph_b200 import esdfConfig
    over.setdefault("min_distance_m", 0.1)
    return esdfConfig(**over)


def _batch_of_copy(layer, ref_ctx, cfg):
    from coxgraph_b200 import Layer
    idx, vox, flags = layer.download()
    R = Layer(ref_ctx, layer.voxel_size, max_blocks=max(64, len(idx)))
    if len(idx):
        R.upload(idx, vox, flags)
    want = R.updateEsdfBatch(cfg)
    want["free"] = R.esdfFreePoints(FREE)
    R.close()
    return want


def _same(got, want, what):
    assert np.array_equal(got["idx"], want["idx"]), f"{what}: block list"
    d = got["distance"].view(np.uint32) != want["distance"].view(np.uint32)
    assert not d.any(), f"{what}: {d.sum()} distances differ"
    p = got["packed"] != want["packed"]
    assert not p.any(), f"{what}: {p.sum()} packed words differ"
    for k in ("blocks", "observed_voxels", "fixed_voxels"):
        assert getattr(got["stats"], k) == getattr(want["stats"], k), f"{what}: stats.{k}"


def _update(layer, ref_ctx, cfg, what):
    want = _batch_of_copy(layer, ref_ctx, cfg)
    got = layer.updateEsdf(cfg)
    _same(got, want, what)
    free = layer.esdfFreePoints(FREE)
    assert np.array_equal(free.view(np.uint32), want["free"].view(np.uint32)), f"{what}: free points"
    u = got["update"]
    assert u.blocks_region <= got["stats"].blocks and u.blocks_changed <= got["stats"].blocks
    if not u.full_rebuild:
        assert got["stats"].block_passes >= u.blocks_region
    return got


def _submaps(ctx, count, frames=2, stride=4):
    import torch
    from coxgraph_b200 import Layer, TsdfIntegrator, TsdfIntegratorConfig, synth
    cfg = TsdfIntegratorConfig(use_const_weight=1, method=1, default_truncation_distance=0.16)
    out = []
    for k in range(count):
        L = Layer(ctx, VS, max_blocks=4096)
        integ = TsdfIntegrator(cfg, L)
        for (T, pts, cols) in synth.submap_frames(k % 2, k + 1, frames, device=torch.device("cuda", 0),
                                                  stride=stride):
            integ.integratePointCloud(T, pts, cols)
        out.append(L)
    return out


VARIANTS = {
    "default": {},
    "narrow band": dict(min_distance_m=0.05),
    "everything fixed": dict(min_distance_m=0.2),
    "short reach": dict(max_distance_m=0.6, default_distance_m=0.6),
    "occupied crust": dict(add_occupied_crust=1),
    "higher min weight": dict(min_weight=1.5),
}


@pytest.mark.parametrize("variant", list(VARIANTS))
def test_session_chain_equals_batch(gpu_ctx, ref_ctx, variant):
    import torch
    from coxgraph_b200 import (Layer, TsdfIntegrator, TsdfIntegratorConfig, getProjectedMap,
                               mergeLayerAintoLayerB, reprojectSubmaps, synth)
    cfg = _cfg(**VARIANTS[variant])
    icfg = TsdfIntegratorConfig(use_const_weight=1, method=1, default_truncation_distance=0.16)
    G = Layer(gpu_ctx, VS, max_blocks=16384)
    integ = TsdfIntegrator(icfg, G)
    frames = synth.submap_frames(0, 0, 4, device=torch.device("cuda", 0), stride=4)
    for (T, pts, cols) in frames[:2]:
        integ.integratePointCloud(T, pts, cols)
    g = _update(G, ref_ctx, cfg, f"{variant}: fused")
    assert g["update"].full_rebuild == 1  # the context's ESDF belonged to another layer
    for (T, pts, cols) in frames[2:]:
        integ.integratePointCloud(T, pts, cols)
    g = _update(G, ref_ctx, cfg, f"{variant}: more frames")
    u = g["update"]
    assert u.full_rebuild == 0 and u.blocks_changed > 0 and u.blocks_region >= u.blocks_changed
    subs = _submaps(gpu_ctx, 3)
    rng = np.random.default_rng(7)
    poses = np.stack([synth.perturb_pose(synth.robot_map_offset(k % 2), rng, 0.2, 5.0) for k in range(3)])
    mergeLayerAintoLayerB(subs[0], poses[0], G)
    g = _update(G, ref_ctx, cfg, f"{variant}: merged submap")
    assert g["update"].full_rebuild == 0
    new = poses.copy()
    new[1, 4:7] += np.array([3.0, -2.0, 0.0], np.float32)
    reprojectSubmaps(subs, poses, new, G)
    g = _update(G, ref_ctx, cfg, f"{variant}: re-projected")
    assert g["update"].full_rebuild == 0
    idx = G.block_indices()
    drop = idx[np.random.default_rng(1).choice(len(idx), max(1, len(idx) // 10), replace=False)]
    G.removeBlocks(drop)
    g = _update(G, ref_ctx, cfg, f"{variant}: removed blocks")
    assert g["update"].blocks_removed == len(drop) and g["update"].full_rebuild == 0
    bi, bv, bf = G.download()
    k = len(bi) // 2
    bv = bv[k:k + 1].copy()
    bv["distance"] = -bv["distance"]
    bv["weight"] = 2.0
    G.upload(bi[k:k + 1], bv, bf[k:k + 1])
    g = _update(G, ref_ctx, cfg, f"{variant}: uploaded block")
    assert g["update"].blocks_changed == 1 and g["update"].full_rebuild == 0
    G.clear()
    getProjectedMap(subs, new, G)
    _update(G, ref_ctx, cfg, f"{variant}: projected")
    G.clear()
    getProjectedMap(subs, new, G)  # same content, slots assigned anew
    g = _update(G, ref_ctx, cfg, f"{variant}: projected again")
    u = g["update"]
    assert (u.blocks_changed, u.blocks_removed, u.blocks_region, u.full_rebuild) == (0, 0, 0, 0)
    h = _update(G, ref_ctx, cfg, f"{variant}: no mutation")
    u = h["update"]
    assert (u.blocks_changed, u.blocks_region, u.full_rebuild) == (0, 0, 0)
    assert h["stats"].sweeps == 0 and h["stats"].block_passes == 0
    assert np.array_equal(h["packed"], g["packed"])
    for L in subs + [G]:
        L.close()


def _row(n, weight=1.0):
    from oracle import oracle_py as orc
    idx = np.array([(x, 0, 0) for x in range(n)], np.int32)
    vox = np.zeros((n, 4096), orc.VOXEL_DTYPE)
    vox["distance"], vox["weight"] = 0.16, weight
    return idx, vox


@pytest.mark.parametrize("over", [{}, dict(default_distance_m=3.0)])
def test_reach_of_a_lowering_and_a_raising_wave(gpu_ctx, ref_ctx, over):
    """A row of observed, unfixed blocks; one fixed voxel of 1 mm at x = 15 of block 0 lowers its
    neighbours out to block R = 3 (x = 54, or 55 when default > max lets the hop at max be
    taken), and removing it raises them again."""
    from coxgraph_b200 import Layer
    cfg = _cfg(**over)
    R = math.ceil((math.ceil(2.0 / VS) + 3) / 16)
    assert R == 3
    idx, vox = _row(8)
    L = Layer(gpu_ctx, VS, max_blocks=64)
    L.upload(idx, vox)
    a = _update(L, ref_ctx, cfg, "row")
    v = 15 + 16 * (8 + 16 * 8)
    vox2 = vox.copy()
    vox2[0]["distance"][v] = np.float32(0.001)
    L.upload(idx[:1], vox2[:1])
    b = _update(L, ref_ctx, cfg, "lowering wave")
    assert (b["update"].blocks_changed, b["update"].blocks_region, b["update"].full_rebuild) == (1, R + 1, 0)
    diff = (a["distance"] != b["distance"]) | (a["packed"] != b["packed"])
    far = max(int(bi) * 16 + (int(li) & 15) for bi, li in zip(*np.nonzero(diff)))
    assert far // 16 == R and far - 15 == (40 if over else 39), far
    L.upload(idx[:1], vox[:1])
    c = _update(L, ref_ctx, cfg, "raising wave")
    assert c["update"].blocks_region == R + 1
    assert np.array_equal(c["packed"], a["packed"])
    assert np.array_equal(c["distance"].view(np.uint32), a["distance"].view(np.uint32))
    L.close()


def test_full_rebuild_when_there_is_nothing_to_start_from(ref_ctx):
    from coxgraph_b200 import Context, Layer
    ctx = Context(0)
    idx, vox = _row(5)
    vox[2]["distance"][100:200] = 0.02
    A = Layer(ctx, VS, max_blocks=64)
    A.upload(idx, vox)
    cfg = _cfg()
    assert _update(A, ref_ctx, cfg, "first call")["update"].full_rebuild == 1
    assert _update(A, ref_ctx, cfg, "again")["update"].full_rebuild == 0
    for what, c in (("max distance", _cfg(max_distance_m=1.0)), ("min distance", _cfg(min_distance_m=0.15)),
                    ("default distance", _cfg(default_distance_m=2.5)), ("min weight", _cfg(min_weight=0.5)),
                    ("crust", _cfg(add_occupied_crust=1))):
        assert _update(A, ref_ctx, c, f"config change: {what}")["update"].full_rebuild == 1, what
        assert _update(A, ref_ctx, c, f"after {what}")["update"].full_rebuild == 0, what
    # fields the result does not depend on do not force a rebuild
    c = _cfg(add_occupied_crust=1, min_diff_m=0.0, num_buckets=3)
    assert _update(A, ref_ctx, c, "ignored fields")["update"].full_rebuild == 0
    B = Layer(ctx, VS, max_blocks=64)
    B.upload(idx[:3], vox[:3])
    B.updateEsdfBatch(cfg)
    assert _update(A, ref_ctx, cfg, "batch of another layer between")["update"].full_rebuild == 1
    B.close()
    A.close()
    C_ = Layer(ctx, VS, max_blocks=64)  # may take A's address: identified by serial
    C_.upload(idx, vox)
    assert _update(C_, ref_ctx, cfg, "replaced layer")["update"].full_rebuild == 1
    C_.clear()
    e = _update(C_, ref_ctx, cfg, "emptied layer")
    assert e["update"].full_rebuild == 1 and e["stats"].blocks == 0 and len(e["idx"]) == 0
    C_.upload(idx, vox)
    assert _update(C_, ref_ctx, cfg, "refilled layer")["update"].full_rebuild == 1
    C_.close()
    ctx.close()


def test_rejected_calls_leave_the_retained_esdf(gpu_ctx, ref_ctx):
    from coxgraph_b200 import Layer, capi
    idx, vox = _row(4)
    vox[1]["distance"][:50] = 0.03
    L = Layer(gpu_ctx, VS, max_blocks=64)
    L.upload(idx, vox)
    before = _update(L, ref_ctx, _cfg(), "before")
    free = L.esdfFreePoints(FREE)
    for bad, status in ((_cfg(full_euclidean_distance=1), capi.CG_ERR_UNSUPPORTED),
                        (_cfg(default_distance_m=1.0), capi.CG_ERR_INVALID_ARG),
                        (_cfg(max_distance_m=0.0), capi.CG_ERR_INVALID_ARG),
                        (_cfg(min_distance_m=-1.0), capi.CG_ERR_INVALID_ARG)):
        with pytest.raises(capi.CgError) as ei:
            L.updateEsdf(bad)
        assert ei.value.status == status
    assert np.array_equal(L.esdfFreePoints(FREE).view(np.uint32), free.view(np.uint32))
    after = L.updateEsdf(_cfg())
    _same(after, before, "after rejected calls")
    assert (after["update"].full_rebuild, after["update"].blocks_region) == (0, 0)
    L.close()
