#!/usr/bin/env python
"""Multi-GPU check of cg_reproject_submaps_sharded, one process per GPU (torchrun, NCCL): after every
step each rank's owned and partial layers must equal, exactly (block set, voxel bits, flags), what
cg_layer_clear(owned) + cg_project_submaps_sharded under the effective poses leaves on that rank.
The reference runs in a second context with its own communicator, on copies of the submaps.

  python -m torch.distributed.run --nnodes=1 --nproc-per-node N --master-addr 127.0.0.1 \\
      --master-port 29547 scripts/multigpu_reproject_check.py

Cases, on the C2 shape (every rank's submaps cover one room, ownership interleaves block by block)
and a corridor shape (consecutive corridor submaps on different ranks, the last rank starting with
none), under CG_REPROJECT_FULL_FRACTION=2 (block by block) and the default: a move on every rank,
moves on one rank only, a submap appended on one rank, a submap moved away so that blocks change
holders (removed on one rank, folded on another); cg_layer_mesh_sharded afterwards against
cg_layer_mesh of the union; a partial layer too small for an appended submap on one rank, which
fails on every rank without touching the owned layers, then a successful call after the fix.
Prints "multigpu_reproject_check ok" when everything holds.
"""
import os
import sys

import numpy as np
import torch
import torch.distributed as dist

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "scripts"))

import multigpu_mesh_check as mm  # noqa: E402
from coxgraph_b200 import Context, Layer, capi, sharding, synth  # noqa: E402
from coxgraph_b200.api import getProjectedMapSharded, reprojectSubmapsSharded  # noqa: E402

MAX_BLOCKS = 32768


def copy_to(layer, ctx):
    L = Layer(ctx, 0.05, max_blocks=8192)
    L.upload(*layer.download())
    return L


def same_layer(a, b):
    return (np.array_equal(a[0], b[0]) and np.array_equal(a[2], b[2])
            and all(np.array_equal(a[1][f].view(np.uint32) if f != "rgba" else a[1][f],
                                   b[1][f].view(np.uint32) if f != "rgba" else b[1][f])
                    for f in ("distance", "weight", "rgba")))


class Rank:
    def __init__(self, ctx, ref_ctx, rank, world):
        self.ctx, self.ref_ctx, self.rank, self.world = ctx, ref_ctx, rank, world
        self.partial = Layer(ctx, 0.05, max_blocks=MAX_BLOCKS)
        self.owned = Layer(ctx, 0.05, max_blocks=MAX_BLOCKS)
        self.ref_of = {}

    def ref(self, L):
        if id(L) not in self.ref_of:
            self.ref_of[id(L)] = copy_to(L, self.ref_ctx)
        return self.ref_of[id(L)]

    def check(self, subs, poses, what, failures):
        """This rank's layers against the fresh sharded projection (collective)."""
        P = Layer(self.ref_ctx, 0.05, max_blocks=MAX_BLOCKS)
        O = Layer(self.ref_ctx, 0.05, max_blocks=MAX_BLOCKS)
        getProjectedMapSharded([self.ref(L) for L in subs], poses, P, O)
        if not same_layer(self.owned.download(), O.download()):
            failures.append(f"{what}: owned layer differs from the fresh projection")
        if not same_layer(self.partial.download(), P.download()):
            failures.append(f"{what}: partial layer differs from the fresh projection")
        P.close()
        O.close()


def chain(R, name, subs, poses, extra, failures, block_by_block):
    """Chained steps on one shape; returns this rank's submaps and poses at the end."""
    rank, world = R.rank, R.world
    rng = np.random.default_rng(100 * rank + len(name))
    R.owned.clear()
    getProjectedMapSharded(subs, poses, R.partial, R.owned)
    R.check(subs, poses, f"{name} start", failures)
    cur = poses
    for kind in ("every rank", "one rank", "append", "holder change"):
        new = cur.copy()
        nsubs = list(subs)
        if kind == "every rank" and len(subs):
            new[0] = synth.perturb_pose(cur[0], rng, sigma_t=0.1, sigma_yaw_deg=2.0)
        if kind == "one rank" and rank == 0:
            for k in range(min(2, len(subs))):
                new[k] = synth.perturb_pose(cur[k], rng, sigma_t=0.1, sigma_yaw_deg=2.0)
        if kind == "append" and rank == world - 1:
            nsubs.append(extra)
            new = np.concatenate([new, synth.robot_map_offset(0)[None]])
        if kind == "holder change" and rank == 0:
            new[0, 4:7] += np.array([30.0, 0.0, 0.0], np.float32)
        changed, st = reprojectSubmapsSharded(nsubs, cur, new, R.partial, R.owned,
                                              eps_translation=1e-4, eps_rotation=1e-5)
        cur = np.where(changed[:, None], new, np.concatenate([cur, new[len(cur):]]))
        subs = nsubs
        what = f"{name} / {kind} / {'block by block' if block_by_block else 'default'}"
        R.check(subs, cur, what, failures)
        stats = [None] * world
        dist.all_gather_object(stats, (int(st.blocks_dirty), int(st.full_rebuild),
                                       int(st.blocks_folded), int(st.blocks_removed),
                                       int(st.submaps_added)))
        if len({(s[0], s[1]) for s in stats}) != 1:
            failures.append(f"{what}: ranks disagree on |D| or the full-rebuild decision: {stats}")
        if block_by_block and stats[0][1]:
            failures.append(f"{what}: full rebuild under CG_REPROJECT_FULL_FRACTION=2")
        if kind == "append" and stats[world - 1][4] != 1:
            failures.append(f"{what}: stats of the appending rank {stats[world - 1]}")
        if kind == "holder change" and block_by_block and name == "C2" and world > 1:
            if not (stats[0][3] > 0 and any(s[2] > 0 for s in stats[1:])):
                failures.append(f"{what}: no block removed on rank 0 and folded elsewhere: {stats}")
        if rank == 0:
            print(f"{what}: |D| {stats[0][0]}, (folded, removed) per rank "
                  f"{[(s[2], s[3]) for s in stats]}", flush=True)
    return subs, cur


def local_failure(R, subs, poses, extra, failures):
    """A partial layer too small for the submap rank 0 appends: every rank returns an error, no
    owned layer changes; after the fix (a full projection into the large partial layer) the next
    call succeeds."""
    rank, world = R.rank, R.world
    counts = [None] * world
    R.owned.clear()
    getProjectedMapSharded(subs, poses, R.partial, R.owned)
    dist.all_gather_object(counts, R.partial.num_blocks)
    small = Layer(R.ctx, 0.05, max_blocks=max(counts) + 1)
    R.owned.clear()
    getProjectedMapSharded(subs, poses, small, R.owned)
    before = R.owned.download()
    nsubs, new = list(subs), poses.copy()
    if rank == 0:
        nsubs.append(extra)
        far = synth.robot_map_offset(0)
        far[4:7] += np.array([0.0, 50.0, 0.0], np.float32)
        new = np.concatenate([new, far[None]])
    try:
        reprojectSubmapsSharded(nsubs, poses, new, small, R.owned)
        failures.append("local failure: the call succeeded")
    except capi.CgError as e:
        if e.status != capi.CG_ERR_POOL_FULL:
            failures.append(f"local failure: status {e.status} ({e})")
    if not same_layer(R.owned.download(), before):
        failures.append("local failure: the owned layer changed")
    R.owned.clear()
    getProjectedMapSharded(subs, poses, R.partial, R.owned)
    new = poses.copy()
    if len(subs):
        new[0] = synth.perturb_pose(poses[0], np.random.default_rng(rank), sigma_t=0.1,
                                    sigma_yaw_deg=2.0)
    changed, _ = reprojectSubmapsSharded(subs, poses, new, R.partial, R.owned)
    R.check(subs, np.where(changed[:, None], new, poses), "after the local failure", failures)
    small.close()


def main():
    rank, world = int(os.environ["RANK"]), int(os.environ["WORLD_SIZE"])
    local = int(os.environ.get("LOCAL_RANK", rank))
    torch.cuda.set_device(local)
    dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    ctx = Context(local, stream=torch.cuda.current_stream().cuda_stream)
    ref_ctx = Context(local, stream=torch.cuda.current_stream().cuda_stream)
    sharding.init_native(ctx)
    sharding.init_native(ref_ctx)
    failures = []
    R = Rank(ctx, ref_ctx, rank, world)
    c2 = mm.shape_submaps(ctx, "C2", rank, world, per_rank=3, frames=2, stride=4)
    c3 = mm.shape_submaps(ctx, "C3", rank, world, per_rank=2, frames=8, stride=4)
    extra = mm.fuse(ctx, synth.submap_frames(rank % 2, 50 + rank, 2, device=torch.device("cuda", local),
                                             stride=4))
    last = rank == world - 1
    c3 = ([], c3[1][:0]) if last else c3
    for fraction in ("2", None):
        if fraction:
            os.environ["CG_REPROJECT_FULL_FRACTION"] = fraction
        else:
            os.environ.pop("CG_REPROJECT_FULL_FRACTION", None)
        for name, (subs, poses) in (("C2", c2), ("corridor", c3)):
            chain(R, name, subs, poses, extra, failures, fraction is not None)
        mm.union_check(ctx, R.owned, rank, world, f"mesh after re-projection ({fraction})", failures,
                       reset_flags=False)
    local_failure(R, c2[0], c2[1], extra, failures)

    gathered = [None] * world
    dist.all_gather_object(gathered, failures)
    bad = [f"rank {r}: {f}" for r, fs in enumerate(gathered) for f in fs]
    if rank == 0:
        if bad:
            print("multigpu_reproject_check FAILED:\n  " + "\n  ".join(bad), flush=True)
        else:
            print(f"multigpu_reproject_check ok: world {world}", flush=True)
    capi.check(capi.load().cg_comm_destroy(ctx._h))
    capi.check(capi.load().cg_comm_destroy(ref_ctx._h))
    dist.barrier()
    for L in c2[0] + c3[0] + [extra, R.partial, R.owned] + list(R.ref_of.values()):
        L.close()
    ctx.close()
    ref_ctx.close()
    dist.destroy_process_group()
    sys.exit(1 if bad else 0)


if __name__ == "__main__":
    main()
