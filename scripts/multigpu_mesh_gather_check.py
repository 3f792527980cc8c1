#!/usr/bin/env python
"""Multi-GPU check of cg_mesh_gather_sharded, one process per GPU (torchrun, NCCL): the global map is
projected with cg_project_submaps_sharded, every rank meshes its owned layer with
cg_layer_mesh_sharded, and the block meshes are gathered onto one root.  The root's fetched mesh
and its connected mesh (cg_mesh_connect, the PLY's mesh) must be byte-identical to cg_layer_mesh and
cg_mesh_connect of one layer U holding the union of the owned layers (voxels and flags), built on
one GPU in a second context; every other rank's cg_mesh_fetch must be unchanged by the call.

  python -m torch.distributed.run --nnodes=1 --nproc-per-node N --master-addr 127.0.0.1 \\
      --master-port 29541 scripts/multigpu_mesh_gather_check.py

Cases: the C2 shape and a corridor shape (the shapes of multigpu_mesh_check.py), root 0 and root
world - 1, colour on / off, raised min_weight, and only_updated after some flags were reset; a rank
with an empty owned layer, that rank as the root, and every rank empty; ranks passing different
roots, one rank that ran plain cg_layer_mesh after the sharded mesh, one rank that ran
cg_esdf_free_points, and a repeated gather, each rejected on every rank and followed by a
successful call.  Prints "multigpu_mesh_gather_check ok" when everything holds.
"""
import os
import sys

import numpy as np
import torch
import torch.distributed as dist

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "scripts"))

from coxgraph_b200 import Context, Layer, capi, sharding  # noqa: E402
from coxgraph_b200.api import _fetch_mesh, getProjectedMapSharded  # noqa: E402
from multigpu_mesh_check import MAX_BLOCKS, same_bytes, shape_submaps  # noqa: E402

ARGS = [dict(), dict(use_color=False), dict(min_weight=0.5), dict(only_updated=True)]


def gather_check(ctx, ref_ctx, owned, rank, world, root, what, failures, kw=None):
    """mesh_sharded(**kw) on every rank, then mesh_gather(root): the root's mesh and connected mesh
    == cg_layer_mesh(U) and cg_mesh_connect; the other ranks' retained share unchanged."""
    kw = kw or {}
    held = [None] * world
    dist.all_gather_object(held, owned.download())
    mine = sharding.mesh_sharded(owned, **kw)
    out = sharding.mesh_gather(ctx, root)
    totals = (len(out[0]), len(out[2])) if rank == root else out
    if rank == root:
        gi = np.concatenate([h[0] for h in held])
        U = Layer(ref_ctx, 0.05, max_blocks=max(len(gi), 1) * 2)
        if len(gi):
            U.upload(gi, np.concatenate([h[1] for h in held]), np.concatenate([h[2] for h in held]))
        ref = U.generateMesh(**kw)
        if not same_bytes(out, ref):
            failures.append(f"{what} {kw} root {root}: gathered mesh differs from cg_layer_mesh(U)")
        if not same_bytes(owned.getConnectedMesh(), U.getConnectedMesh()):
            failures.append(f"{what} {kw} root {root}: connected mesh differs from U's")
        expected = (len(ref[0]), len(ref[2]))
        U.close()
    else:
        if not same_bytes(_fetch_mesh(ctx, len(mine[0]), len(mine[2])), mine):
            failures.append(f"{what} {kw} root {root}: rank {rank}'s retained mesh changed")
        expected = None
    both = [None] * world
    dist.all_gather_object(both, (totals, expected))
    if both[root][1] is not None and any(tuple(b[0]) != tuple(both[root][1]) for b in both):
        failures.append(f"{what} {kw} root {root}: global totals {[b[0] for b in both]}, "
                        f"expected {both[root][1]}")
    if rank == root and not kw:
        print(f"{what}: root {root}, {totals[0]} blocks, {totals[1]} vertices over {world} ranks",
              flush=True)


def reset_some_flags(owned):
    idx, vox, fl = owned.download()
    sel = np.arange(0, len(idx), 3)
    if len(sel):
        owned.upload(idx[sel], vox[sel], fl[sel] & np.uint8(0xFD))


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
    ref_ctx = Context(local)
    sharding.init_native(ctx)
    failures = []
    partial = Layer(ctx, 0.05, max_blocks=MAX_BLOCKS)
    owned = Layer(ctx, 0.05, max_blocks=MAX_BLOCKS)
    last = world - 1

    # 1: both shapes, roots 0 and world - 1, every argument combination
    c2 = shape_submaps(ctx, "C2", rank, world, per_rank=2, frames=3, stride=2)
    c3 = shape_submaps(ctx, "C3", rank, world, per_rank=2, frames=10, stride=2)
    for name, (subs, poses) in (("C2", c2), ("corridor", c3)):
        owned.clear()
        getProjectedMapSharded(subs, poses, partial, owned)
        for root in sorted({0, last}):
            for kw in ARGS:
                if kw.get("only_updated"):
                    reset_some_flags(owned)
                gather_check(ctx, ref_ctx, owned, rank, world, root, name, failures, kw)

    # 2: the last rank passes no submaps, so its owned layer stays empty; it is also the root
    subs, poses = c2
    owned.clear()
    getProjectedMapSharded([] if rank == last else subs, poses[:0] if rank == last else poses,
                           partial, owned)
    if rank == last and owned.num_blocks:
        failures.append("empty rank: the owned layer is not empty")
    for root in sorted({0, last}):
        gather_check(ctx, ref_ctx, owned, rank, world, root, "C2 with an empty rank", failures)
    # every rank empty
    owned.clear()
    gather_check(ctx, ref_ctx, owned, rank, world, 0, "every rank empty", failures)

    # 3: errors seen by every rank, each followed by a successful call
    owned.clear()
    getProjectedMapSharded(c2[0], c2[1], partial, owned)

    def good(what):
        gather_check(ctx, ref_ctx, owned, rank, world, 0, f"after {what}", failures)

    if world > 1:
        sharding.mesh_sharded(owned, fetch=False)
        expect_invalid(lambda: sharding.mesh_gather(ctx, rank % 2), "different roots",
                       "different roots", failures)
        good("different roots")
    sharding.mesh_sharded(owned, fetch=False)
    expect_invalid(lambda: sharding.mesh_gather(ctx, world), f"root {world}", "root out of range",
                   failures)
    good("a root out of range")
    sharding.mesh_sharded(owned, fetch=False)
    if rank == last:
        owned.generateMesh(fetch=False)
    expect_invalid(lambda: sharding.mesh_gather(ctx, 0), f"rank {last}'s retained mesh is from "
                   "cg_layer_mesh", "plain cg_layer_mesh on one rank", failures)
    good("plain cg_layer_mesh on one rank")
    if rank == 0:
        owned.updateEsdfBatch(fetch=False)
    sharding.mesh_sharded(owned, fetch=False)
    if rank == 0 and not len(owned.esdfFreePoints(0.1)):
        failures.append("cg_esdf_free_points found no free point")
    expect_invalid(lambda: sharding.mesh_gather(ctx, 0), "cg_esdf_free_points",
                   "cg_esdf_free_points on one rank", failures)
    good("cg_esdf_free_points on one rank")
    sharding.mesh_sharded(owned, fetch=False)
    sharding.mesh_gather(ctx, last)
    expect_invalid(lambda: sharding.mesh_gather(ctx, last), "gathered already", "repeated gather",
                   failures)
    good("a repeated gather")

    gathered = [None] * world
    dist.all_gather_object(gathered, failures)
    bad = [f"rank {r}: {f}" for r, fs in enumerate(gathered) for f in fs]
    if rank == 0:
        if bad:
            print("multigpu_mesh_gather_check FAILED:\n  " + "\n  ".join(bad), flush=True)
        else:
            print(f"multigpu_mesh_gather_check ok: world {world}", flush=True)
    capi.check(capi.load().cg_comm_destroy(ctx._h))  # peer mappings closed before layers go
    dist.barrier()
    for L in c2[0] + c3[0] + [partial, owned]:
        L.close()
    ref_ctx.close()
    ctx.close()
    dist.destroy_process_group()
    sys.exit(1 if bad else 0)


if __name__ == "__main__":
    main()
