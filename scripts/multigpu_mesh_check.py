#!/usr/bin/env python
"""Multi-GPU check of cg_layer_mesh_sharded, one process per GPU (torchrun, NCCL): the global map
is projected with cg_project_submaps_sharded, every rank meshes its owned layer where it lies, and
rank 0 compares the ranks' block meshes, merged by block index, byte for byte with cg_layer_mesh of
one layer U holding the union of the owned layers (voxels and flags).

  python -m torch.distributed.run --nnodes=1 --nproc-per-node N --master-addr 127.0.0.1 \\
      --master-port 29523 scripts/multigpu_mesh_check.py

Cases: the C2 shape (every rank's submaps cover the same room, so ownership interleaves block by
block) and a corridor shape (consecutive corridor submaps on different ranks), each for colour
on / off, default and raised min_weight, and only_updated after some flags were reset; a guard
that plain cg_layer_mesh of the owned layers differs (the halo is exercised); a rank with an empty
owned layer; a colour block held by a third rank; gather / mesh calls alternating without new peer
mappings; a key held by two ranks and mismatched voxel sizes rejected on every rank, each followed
by a successful call.  Prints "multigpu_mesh_check ok" when everything holds.
"""
import os
import sys

import numpy as np
import torch
import torch.distributed as dist

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

from coxgraph_b200 import (VOXEL_DTYPE, Context, Layer, TsdfIntegrator,  # noqa: E402
                           TsdfIntegratorConfig, capi, sharding, synth)
from coxgraph_b200.api import commPeerMappings, getProjectedMapSharded  # noqa: E402

CFG = dict(use_const_weight=1, method=1, default_truncation_distance=0.16)
ARGS = [dict(), dict(use_color=False), dict(min_weight=0.5), dict(min_weight=0.5, use_color=False),
        dict(only_updated=True)]
MAX_BLOCKS = 32768


def fuse(ctx, frames):
    L = Layer(ctx, 0.05, max_blocks=8192)
    integ = TsdfIntegrator(TsdfIntegratorConfig(**CFG), L)
    for (T, pts, cols) in frames:
        integ.integratePointCloud(T, pts, cols)
    return L


def shape_submaps(ctx, shape, rank, world, per_rank, frames, stride, robot_per_rank=False):
    """This rank's fused submaps and their poses.
    C2: submaps of two robots in one room (robot_map_offset), interleaved over the ranks.
    C3: corridor submaps.  robot_per_rank: rank r drives robot r's corridor (the benchmark's C3,
    robots 128 m apart); otherwise consecutive submaps of one corridor drive go to consecutive
    ranks, so the ranks meet wherever two submaps overlap."""
    dev = torch.device("cuda", torch.cuda.current_device())
    subs, poses = [], []
    for k in range(per_rank):
        if shape == "C2":
            sid = rank * per_rank + k
            robot = sid % 2
            fr = synth.submap_frames(robot, sid, frames, device=dev, stride=stride)
            pose = synth.robot_map_offset(robot)
        else:
            robot, sm = (rank, k) if robot_per_rank else (0, rank + world * k)
            fr = synth.corridor_frames(sm * frames, frames, robot=robot, advance=0.2,
                                       start_x=128.0 * robot, device=dev, stride=stride)
            pose = synth.robot_map_offset(0)
        subs.append(fuse(ctx, fr))
        poses.append(pose)
    return subs, np.stack(poses) if poses else np.zeros((0, 7), np.float32)


def merged(per_rank):
    """Block meshes of all ranks merged by block index in (z, y, x) order."""
    idx = np.concatenate([m[0] for m in per_rank])
    order = np.lexsort((idx[:, 0], idx[:, 1], idx[:, 2]))
    src = [(r, b) for r, m in enumerate(per_rank) for b in range(len(m[0]))]
    begin, v, n, c = [0], [], [], []
    for o in order:
        r, b = src[o]
        m = per_rank[r]
        lo, hi = int(m[1][b]), int(m[1][b + 1])
        v.append(m[2][lo:hi])
        n.append(m[3][lo:hi])
        c.append(m[4][lo:hi])
        begin.append(begin[-1] + hi - lo)
    cat = (lambda xs, shape, dt: np.concatenate(xs) if xs else np.zeros(shape, dt))
    return (idx[order], np.array(begin, np.uint32), cat(v, (0, 3), np.float32),
            cat(n, (0, 3), np.float32), cat(c, (0, 4), np.uint8))


def same_bytes(a, b):
    return all(x.shape == y.shape and np.array_equal(x.view(np.uint8), y.view(np.uint8))
               for x, y in zip(a, b))


def union_check(ctx, owned, rank, world, what, failures, reset_flags=True):
    """Every argument combination: the ranks' meshes merged == cg_layer_mesh(U).  Returns this
    rank's results of the default arguments."""
    results = [sharding.mesh_sharded(owned, **kw) for kw in ARGS[:-1]]
    if reset_flags:  # only_updated after clearing the flag of every third block
        idx, vox, fl = owned.download()
        sel = np.arange(0, len(idx), 3)
        if len(sel):
            owned.upload(idx[sel], vox[sel], fl[sel] & np.uint8(0xFD))
    results.append(sharding.mesh_sharded(owned, **ARGS[-1]))
    gathered = [None] * world
    dist.all_gather_object(gathered, (owned.download(), results))
    if rank == 0:
        gi = np.concatenate([g[0][0] for g in gathered])
        gv = np.concatenate([g[0][1] for g in gathered])
        gf = np.concatenate([g[0][2] for g in gathered])
        if len(np.unique(gi, axis=0)) != len(gi):
            failures.append(f"{what}: a block is held by two ranks")
        U = Layer(ctx, 0.05, max_blocks=max(len(gi), 1) * 2)
        if len(gi):
            U.upload(gi, gv, gf)
        for a, kw in enumerate(ARGS):
            ref = U.generateMesh(**kw)
            got = merged([g[1][a] for g in gathered])
            if not same_bytes(got, ref):
                failures.append(f"{what} {kw}: merged sharded meshes differ from cg_layer_mesh(U)")
        print(f"{what}: {len(gi)} blocks over {world} ranks "
              f"({[len(g[0][0]) for g in gathered]}), {len(U.generateMesh()[2])} vertices",
              flush=True)
        U.close()
    return results[0]


def expect_invalid(fn, needle, what, failures):
    try:
        fn()
    except capi.CgError as e:
        if e.status != capi.CG_ERR_INVALID_ARG or needle not in str(e):
            failures.append(f"{what}: wrong error {e}")
        return
    failures.append(f"{what}: accepted")


def main():
    rank, world = int(os.environ["RANK"]), int(os.environ["WORLD_SIZE"])
    local = int(os.environ.get("LOCAL_RANK", rank))
    torch.cuda.set_device(local)
    dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    ctx = Context(local, stream=torch.cuda.current_stream().cuda_stream)
    sharding.init_native(ctx)
    failures = []
    partial = Layer(ctx, 0.05, max_blocks=MAX_BLOCKS)
    owned = Layer(ctx, 0.05, max_blocks=MAX_BLOCKS)

    # 1 + 2: union check on the C2 and the corridor shape, and the guard on C2
    c2 = shape_submaps(ctx, "C2", rank, world, per_rank=2, frames=3, stride=2)
    c3 = shape_submaps(ctx, "C3", rank, world, per_rank=2, frames=10, stride=2)
    for name, (subs, poses) in (("C2", c2), ("corridor", c3)):
        owned.clear()
        getProjectedMapSharded(subs, poses, partial, owned)
        mine = union_check(ctx, owned, rank, world, name, failures)
        if name == "C2":
            plain = owned.generateMesh()
            differs = [None] * world
            dist.all_gather_object(differs, not same_bytes(plain, mine))
            if rank == 0 and not any(differs):
                failures.append("guard: plain cg_layer_mesh of the owned layers equals the sharded "
                                "mesh on every rank: the halo was not exercised")

    # 3a: the last rank passes no submaps, so its owned layer stays empty
    subs, poses = c2
    last = rank == world - 1
    owned.clear()
    getProjectedMapSharded([] if last else subs, poses[:0] if last else poses, partial, owned)
    if last and owned.num_blocks:
        failures.append("empty rank: the owned layer is not empty")
    union_check(ctx, owned, rank, world, "C2 with an empty rank", failures)

    # 3b: a colour block on a third rank.  A 2 x 2 x 2 block cube with the plane y = 16.1 voxels:
    # the vertices that cube (15, 15, z) of block (0, 0, z) puts on its x = 16 edges lie in block
    # (1, 1, z), which the colour lookup reads.  Blocks (0,0,z) -> rank 0, (1,0,z) and (0,1,z) ->
    # rank 1, (1,1,z) -> rank 2 (mod world); every block has its own colour.
    E = Layer(ctx, 0.05, max_blocks=MAX_BLOCKS)
    owner = {(0, 0): 0, (1, 0): 1 % world, (0, 1): 1 % world, (1, 1): 2 % world}
    lin = np.arange(4096)
    loc = np.stack([lin & 15, (lin >> 4) & 15, lin >> 8], -1)
    blocks = [(x, y, z) for z in (0, 1) for y in (0, 1) for x in (0, 1)]
    mine_b = np.array([b for b in blocks if owner[b[:2]] == rank], np.int32).reshape(-1, 3)
    vox = np.zeros((len(mine_b), 4096), VOXEL_DTYPE)
    for k, b in enumerate(mine_b):
        c = (b[None, :] * 16 + loc + 0.5) * 0.05
        vox[k]["distance"] = (c[:, 1] - 16.1 * 0.05) + 0.02 * c[:, 2]
        vox[k]["weight"] = 1.0
        vox[k]["rgba"] = (10 * b[0] + 1, 10 * b[1] + 2, 10 * b[2] + 3, 255)
    if len(mine_b):
        E.upload(mine_b, vox)
    mine = union_check(ctx, E, rank, world, "colour block on a third rank", failures, reset_flags=False)
    if rank == 0 and world >= 3:
        idx, begin, _, _, col = mine
        b0 = [i for i, b in enumerate(idx) if tuple(b) == (0, 0, 0)]
        far = np.array([11, 12, 3, 255], np.uint8)  # colour of block (1, 1, 0), held by rank 2
        if not b0 or not (col[begin[b0[0]]:begin[b0[0] + 1]] == far).all(axis=1).any():
            failures.append("third rank: no vertex of block (0,0,0) took its colour from (1,1,0)")

    # 3c: gather and mesh alternate three times; no peer mapping is opened after the first pair
    opened = []
    meshes = []
    for rep in range(3):
        owned.clear()
        getProjectedMapSharded(c2[0], c2[1], partial, owned)
        meshes.append(sharding.mesh_sharded(owned))
        opened.append(commPeerMappings(ctx)[0])
    if opened[1] != opened[0] or opened[2] != opened[0]:
        failures.append(f"alternating calls opened peer mappings again: {opened}")
    if not (same_bytes(meshes[0], meshes[1]) and same_bytes(meshes[0], meshes[2])):
        failures.append("alternating calls: the meshes differ between repetitions")

    # 4: errors seen by every rank, each followed by a successful call
    D = Layer(ctx, 0.05, max_blocks=MAX_BLOCKS)
    if rank < 2:
        v = np.zeros((1, 4096), VOXEL_DTYPE)
        v["weight"] = 1.0
        D.upload(np.array([[5, -7, 3]], np.int32), v)
    expect_invalid(lambda: sharding.mesh_sharded(D), "(5, -7, 3)", "key held by two ranks", failures)
    if not same_bytes(sharding.mesh_sharded(owned), meshes[0]):
        failures.append("the call after the duplicate-key error differs")
    X = Layer(ctx, 0.04 if rank == 1 else 0.05, max_blocks=MAX_BLOCKS)
    expect_invalid(lambda: sharding.mesh_sharded(X), "differs", "mismatched voxel sizes", failures)
    if not same_bytes(sharding.mesh_sharded(owned), meshes[0]):
        failures.append("the call after the voxel-size error differs")

    gathered = [None] * world
    dist.all_gather_object(gathered, failures)
    bad = [f"rank {r}: {f}" for r, fs in enumerate(gathered) for f in fs]
    if rank == 0:
        if bad:
            print("multigpu_mesh_check FAILED:\n  " + "\n  ".join(bad), flush=True)
        else:
            print(f"multigpu_mesh_check ok: world {world}, peer mappings opened {opened[0]}",
                  flush=True)
    capi.check(capi.load().cg_comm_destroy(ctx._h))  # peer mappings closed before layers go
    dist.barrier()
    for L in c2[0] + c3[0] + [partial, owned, E, D, X]:
        L.close()
    ctx.close()
    dist.destroy_process_group()
    sys.exit(1 if bad else 0)


if __name__ == "__main__":
    main()
