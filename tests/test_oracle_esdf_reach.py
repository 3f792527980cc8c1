"""CPU: the reach bound behind cg_layer_esdf_update (DESIGN §4.6), on the sequential oracle.

A voxel only feeds a neighbour while |d| < max_distance_m, and every hop adds at least one voxel
size, so the result of a voxel (distance and packed word: flags and parent) depends only on the
init states within L + 1 voxels (Chebyshev) of it, L = ceil(max_distance_m / voxel_size) + 1.
Random voxel and block edits are applied to small layers; the ESDF before and after (min_diff_m = 0,
the fixed point the device computes) may differ only within L + 1 of an edited voxel.  A
constructed case shows the change travelling L - 2 voxels: the bound is nearly tight."""
import math

import numpy as np
import pytest
from scipy import ndimage

from oracle import oracle_py as orc

VS = 0.05


def _dense(idx, values, lo, shape, fill):
    """[B,4096] per-block values -> dense [z, y, x] grid starting at block `lo`."""
    g = np.full(shape, fill, values.dtype)
    for b, (bx, by, bz) in enumerate(idx):
        x0, y0, z0 = (np.array([bx, by, bz]) - lo) * 16
        g[z0:z0 + 16, y0:y0 + 16, x0:x0 + 16] = values[b].reshape(16, 16, 16)
    return g


def _esdf_dense(layer, cfg, lo, shape):
    e = layer.esdf_batch(cfg)
    packed = (e["flags"].astype(np.uint32) |
              (e["parent"].view(np.uint8).astype(np.uint32) << np.array([24, 16, 8], np.uint32)).sum(-1))
    return (_dense(e["idx"], e["distance"].view(np.uint32), lo, shape, np.uint32(0xFFFFFFFF)),
            _dense(e["idx"], packed.astype(np.uint32), lo, shape, np.uint32(0xFFFFFFFF)))


def _changed_voxels(layer_a, layer_b, cfg, lo, shape):
    da, pa = _esdf_dense(layer_a, cfg, lo, shape)
    db, pb = _esdf_dense(layer_b, cfg, lo, shape)
    return (da != db) | (pa != pb)


def _reach(cfg):
    return math.ceil(np.float32(cfg.max_distance_m) / np.float32(VS)) + 1


def _layer(idx, vox):
    L = orc.Layer(VS)
    L.upload(np.ascontiguousarray(idx), np.ascontiguousarray(vox))
    return L


def _random_layer(rng, nb=(4, 3, 2)):
    idx = np.array([(x, y, z) for z in range(nb[2]) for y in range(nb[1]) for x in range(nb[0])], np.int32)
    vox = np.zeros((len(idx), 4096), orc.VOXEL_DTYPE)
    i = np.arange(4096)
    c = rng.uniform(0.5, 2.5, size=(3, 3))
    for b, (bx, by, bz) in enumerate(idx):
        p = np.stack([(bx * 16 + (i & 15) + 0.5) * VS, (by * 16 + ((i >> 4) & 15) + 0.5) * VS,
                      (bz * 16 + (i >> 8) + 0.5) * VS], -1)
        sdf = np.min(np.linalg.norm(p[:, None, :] - c[None], axis=-1), axis=1) - 0.3
        vox[b]["distance"] = np.clip(sdf, -0.16, 0.16).astype(np.float32)
        vox[b]["weight"] = np.where(rng.random(4096) < 0.05, 0.0, 1.0).astype(np.float32)
    return idx, vox


@pytest.mark.parametrize("seed", range(6))
@pytest.mark.parametrize("variant", [dict(max_distance_m=0.6, default_distance_m=0.6),
                                     dict(max_distance_m=0.45, default_distance_m=0.45,
                                          add_occupied_crust=1)])
def test_result_changes_only_within_reach_of_an_edit(seed, variant):
    rng = np.random.default_rng(seed)
    cfg = orc.default_esdf_config(min_diff_m=0.0, min_distance_m=0.1, **variant)
    idx, vox = _random_layer(rng)
    lo, shape = np.zeros(3, np.int64), (2 * 16, 3 * 16, 4 * 16)
    vox2 = vox.copy()
    edited = np.zeros(shape, bool)
    # voxel edits: fix, flip sign, unobserve, observe
    for _ in range(int(rng.integers(1, 5))):
        b, v = int(rng.integers(len(idx))), int(rng.integers(4096))
        kind = int(rng.integers(4))
        if kind == 0:
            vox2[b]["distance"][v] = np.float32(rng.uniform(-0.09, 0.09))
        elif kind == 1:
            vox2[b]["distance"][v] = -vox2[b]["distance"][v] if vox2[b]["distance"][v] else np.float32(0.15)
        vox2[b]["weight"][v] = np.float32(0.0 if kind == 2 else 1.0)
        x, y, z = idx[b] * 16 + np.array([v & 15, (v >> 4) & 15, v >> 8])
        edited[z, y, x] = True
    # block edits: remove one, and (seeds 3..5) keep only a part of the layer
    keep = np.ones(len(idx), bool)
    keep[int(rng.integers(len(idx)))] = False
    if seed >= 3:
        keep[int(rng.integers(len(idx)))] = False
    for b in np.flatnonzero(~keep):
        x0, y0, z0 = idx[b] * 16
        edited[z0:z0 + 16, y0:y0 + 16, x0:x0 + 16] = True
    before, after = _layer(idx, vox), _layer(idx[keep], vox2[keep])
    diff = _changed_voxels(before, after, cfg, lo, shape)
    assert diff.any()
    dist = ndimage.distance_transform_cdt(~edited, metric="chessboard")
    L = _reach(cfg)
    assert dist[diff].max() <= L + 1, (dist[diff].max(), L)


def test_a_change_travels_nearly_the_whole_reach():
    """A row of observed, unfixed blocks (all at +default) and one fixed voxel of distance 1 mm at
    x = 15 of block 0.  Hop k takes 0.001 + k * voxel_size and is lowered while that is below
    default = max = 2 m: the change travels 39 = L - 2 voxels, and the next voxel (hop L - 1) would
    need default_distance_m > max_distance_m, which the oracle does not model (the device reach test
    covers it)."""
    cfg = orc.default_esdf_config(min_diff_m=0.0, min_distance_m=0.1)
    idx = np.array([(x, 0, 0) for x in range(6)], np.int32)
    vox = np.zeros((len(idx), 4096), orc.VOXEL_DTYPE)
    vox["distance"], vox["weight"] = 0.16, 1.0
    vox2 = vox.copy()
    vox2[0]["distance"][15 + 16 * (8 + 16 * 8)] = np.float32(0.001)
    shape = (16, 16, 6 * 16)
    diff = _changed_voxels(_layer(idx, vox), _layer(idx, vox2), cfg, np.zeros(3, np.int64), shape)
    edited = np.zeros(shape, bool)
    edited[8, 8, 15] = True
    far = ndimage.distance_transform_cdt(~edited, metric="chessboard")[diff].max()
    L = _reach(cfg)
    assert far == L - 2, (far, L)
