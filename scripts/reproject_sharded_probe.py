#!/usr/bin/env python
"""Timing of cg_reproject_submaps_sharded against what it replaces, one process per GPU (torchrun,
NCCL), on the C3 corridor shape (one robot per rank, robots 128 m apart, as in the benchmark's C3):

  incremental  cg_reproject_submaps_sharded after a pose-graph update (device time, maximum over
               the ranks);
  full         cg_layer_clear(owned) + cg_project_submaps_sharded under the same effective poses
               (device time, maximum over the ranks), run in a second context;
  vertices     cg_layer_mesh_sharded(only_updated) after cg_layer_reset_updated + the incremental
               call, against the full sharded mesh (summed over the ranks).

Cases: 1 submap moved, 1 % and 10 % of all submaps moved, 1 submap appended.  Every run also checks
that both layers of every rank are bit-identical to the full path (blocks, voxels, has_data).

  python -m torch.distributed.run --nnodes=1 --nproc-per-node N --master-addr 127.0.0.1 \\
      --master-port 29548 scripts/reproject_sharded_probe.py [--out result.json]

Prints one JSON line per case, with the card's name and power limit read in the same run.
"""
import argparse
import json
import os
import subprocess
import sys

import numpy as np
import torch
import torch.distributed as dist

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "scripts"))

from coxgraph_b200 import Context, Layer, capi, sharding, synth  # noqa: E402
from coxgraph_b200.api import getProjectedMapSharded, reprojectSubmapsSharded  # noqa: E402
from multigpu_mesh_check import fuse, shape_submaps  # noqa: E402

MAX_BLOCKS = 131072


def card(local):
    q = subprocess.run(["nvidia-smi", "-i", str(local), "--query-gpu=name,power.limit",
                        "--format=csv,noheader"], capture_output=True, text=True)
    return q.stdout.strip()


def device_ms(fn):
    stream = torch.cuda.current_stream()
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    dist.barrier()
    torch.cuda.synchronize()
    a.record(stream)
    out = fn()
    b.record(stream)
    torch.cuda.synchronize()
    return a.elapsed_time(b), out


def same_data(a, b):
    return (np.array_equal(a[0], b[0]) and np.array_equal(a[2] & 1, b[2] & 1)
            and np.array_equal(a[1]["distance"].view(np.uint32), b[1]["distance"].view(np.uint32))
            and np.array_equal(a[1]["weight"].view(np.uint32), b[1]["weight"].view(np.uint32))
            and np.array_equal(a[1]["rgba"], b[1]["rgba"]))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--submaps", type=int, default=64, help="corridor submaps per rank")
    ap.add_argument("--frames", type=int, default=6)
    ap.add_argument("--stride", type=int, default=2)
    ap.add_argument("--repeats", type=int, default=3)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    rank, world = int(os.environ["RANK"]), int(os.environ["WORLD_SIZE"])
    local = int(os.environ.get("LOCAL_RANK", rank))
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    dist.init_process_group("nccl", device_id=dev)
    ctx = Context(local, stream=torch.cuda.current_stream().cuda_stream)
    ref_ctx = Context(local, stream=torch.cuda.current_stream().cuda_stream)
    sharding.init_native(ctx)
    sharding.init_native(ref_ctx)
    subs, poses = shape_submaps(ctx, "C3", rank, world, args.submaps, frames=args.frames,
                                stride=args.stride, robot_per_rank=True)
    extra = fuse(ctx, synth.corridor_frames(args.submaps * args.frames, args.frames, robot=rank,
                                            advance=0.2, start_x=128.0 * rank, device=dev,
                                            stride=args.stride))
    ref_of = {}
    for L in subs + [extra]:
        R = Layer(ref_ctx, 0.05, max_blocks=8192)
        R.upload(*L.download())
        ref_of[id(L)] = R
    partial, owned = Layer(ctx, 0.05, max_blocks=MAX_BLOCKS), Layer(ctx, 0.05, max_blocks=MAX_BLOCKS)
    P2, O2 = Layer(ref_ctx, 0.05, max_blocks=MAX_BLOCKS), Layer(ref_ctx, 0.05, max_blocks=MAX_BLOCKS)
    total = world * args.submaps
    name = card(local)
    lines, failures = [], []
    for case, count in (("move 1", 1), ("move 1%", max(1, round(0.01 * total))),
                        ("move 10%", max(1, round(0.1 * total))), ("append 1", 0)):
        rng = np.random.default_rng(len(case) + count)  # the same choice on every rank
        picked = rng.choice(total, count, replace=False)
        t_inc, t_full, nv = [], [], None
        for rep in range(args.repeats):
            owned.clear()
            getProjectedMapSharded(subs, poses, partial, owned)
            owned.resetUpdated()
            nsubs, new = list(subs), poses.copy()
            for g in picked:
                if g // args.submaps == rank:
                    k = g % args.submaps
                    new[k] = synth.perturb_pose(poses[k], np.random.default_rng(int(g) + rep),
                                                sigma_t=0.05, sigma_yaw_deg=1.0)
            if case == "append 1" and rank == 0:
                nsubs.append(extra)
                new = np.concatenate([new, poses[-1:]])
            ti, (changed, st) = device_ms(lambda: reprojectSubmapsSharded(nsubs, poses, new, partial,
                                                                          owned))
            eff = np.where(changed[:, None], new, np.concatenate([poses, new[len(poses):]]))
            tf, _ = device_ms(lambda: (O2.clear(), getProjectedMapSharded(
                [ref_of[id(L)] for L in nsubs], eff, P2, O2)))
            t_inc.append(ti)
            t_full.append(tf)
            if not (same_data(owned.download(), O2.download())
                    and same_data(partial.download(), P2.download())):
                failures.append(f"{case}: layers differ from the full path")
            nv = (sharding.mesh_sharded(owned, only_updated=True, fetch=False)[1],
                  sharding.mesh_sharded(owned, fetch=False)[1], owned.num_blocks,
                  int(st.blocks_dirty), int(st.full_rebuild))
        per_rank = [None] * world
        dist.all_gather_object(per_rank, (t_inc, t_full, nv, failures))
        if rank == 0:
            inc = [max(p[0][i] for p in per_rank) for i in range(args.repeats)]
            full = [max(p[1][i] for p in per_rank) for i in range(args.repeats)]
            line = dict(probe="reproject_sharded", shape="C3", world=world, card=name,
                        submaps_per_rank=args.submaps, case=case, submaps_changed=count or 1,
                        global_blocks=sum(p[2][2] for p in per_rank),
                        blocks_dirty=per_rank[0][2][3], full_rebuild=per_rank[0][2][4],
                        incremental_ms=round(min(inc), 3), incremental_ms_all=[round(x, 3) for x in inc],
                        full_ms=round(min(full), 3), full_ms_all=[round(x, 3) for x in full],
                        vertices_only_updated=sum(p[2][0] for p in per_rank),
                        vertices_full=sum(p[2][1] for p in per_rank),
                        bit_identical=not any(p[3] for p in per_rank))
            print(json.dumps(line), flush=True)
            lines.append(line)
    if rank == 0 and args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            json.dump(lines, f, indent=1)
    capi.check(capi.load().cg_comm_destroy(ctx._h))
    capi.check(capi.load().cg_comm_destroy(ref_ctx._h))
    dist.barrier()
    for L in subs + [extra, partial, owned, P2, O2] + list(ref_of.values()):
        L.close()
    ctx.close()
    ref_ctx.close()
    dist.destroy_process_group()
    sys.exit(1 if failures else 0)


if __name__ == "__main__":
    main()
