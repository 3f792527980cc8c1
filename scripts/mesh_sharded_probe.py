#!/usr/bin/env python
"""Timing of cg_layer_mesh_sharded against the ways to mesh a sharded global map without it, one
process per GPU (torchrun, NCCL):

  sharded    cg_layer_mesh_sharded on every rank (count query, the mesh stays on the device):
             device time, maximum over the ranks;
  via host   today's alternative: every rank downloads its owned layer, rank 0 gathers them
             through the host, uploads them into one layer and runs cg_layer_mesh (host clock
             from a barrier to the end of the mesh on rank 0);
  resident   cg_layer_mesh of that gathered layer, already resident on one GPU (device time).

  python -m torch.distributed.run --nnodes=1 --nproc-per-node N --master-addr 127.0.0.1 \\
      --master-port 29524 scripts/mesh_sharded_probe.py [--out result.json]

Shapes: C2 (every rank's submaps cover the same room, ownership interleaves block by block) and
C3 (one robot per rank on the corridor scene, robots 128 m apart, as in the benchmark's C3).
Prints one JSON line per shape, with the card's name and power limit read in the same run.
"""
import argparse
import json
import os
import subprocess
import sys
import time

import numpy as np
import torch
import torch.distributed as dist

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "scripts"))

from coxgraph_b200 import Context, Layer, capi, sharding  # noqa: E402
from coxgraph_b200.api import getProjectedMapSharded  # noqa: E402
from multigpu_mesh_check import shape_submaps  # noqa: E402


def card(local):
    q = subprocess.run(["nvidia-smi", "-i", str(local), "--query-gpu=name,power.limit",
                        "--format=csv,noheader"], capture_output=True, text=True)
    return q.stdout.strip()


def device_ms(ctx, fn, repeats):
    stream = torch.cuda.current_stream()
    times = []
    for _ in range(repeats):
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        dist.barrier()
        torch.cuda.synchronize()
        a.record(stream)
        out = fn()
        b.record(stream)
        torch.cuda.synchronize()
        times.append(a.elapsed_time(b))
    return times, out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--c2-submaps", type=int, default=4, help="room submaps per rank (C2)")
    ap.add_argument("--c3-submaps", type=int, default=8, help="corridor submaps per rank (C3)")
    ap.add_argument("--repeats", type=int, default=6)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    rank, world = int(os.environ["RANK"]), int(os.environ["WORLD_SIZE"])
    local = int(os.environ.get("LOCAL_RANK", rank))
    torch.cuda.set_device(local)
    dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    ctx = Context(local, stream=torch.cuda.current_stream().cuda_stream)
    sharding.init_native(ctx)
    lines, keep = [], []
    for shape, per_rank, robot_per_rank in (("C2", args.c2_submaps, False),
                                            ("C3", args.c3_submaps, True)):
        subs, poses = shape_submaps(ctx, shape, rank, world, per_rank, frames=10, stride=1,
                                    robot_per_rank=robot_per_rank)
        partial = Layer(ctx, 0.05, max_blocks=65536)
        owned = Layer(ctx, 0.05, max_blocks=65536)
        getProjectedMapSharded(subs, poses, partial, owned)
        t_sh, (nb, nv) = device_ms(ctx, lambda: sharding.mesh_sharded(owned, fetch=False),
                                   args.repeats)
        # today's alternative: through the host to one GPU
        t_host = []
        U = None
        for _ in range(max(2, args.repeats // 2)):
            dist.barrier()
            t0 = time.perf_counter()
            mine = owned.download()
            gathered = [None] * world
            dist.all_gather_object(gathered, mine)
            if rank == 0:
                gi = np.concatenate([g[0] for g in gathered])
                if U is None:
                    U = Layer(ctx, 0.05, max_blocks=max(len(gi), 1) * 2)
                U.clear()
                U.upload(gi, np.concatenate([g[1] for g in gathered]),
                         np.concatenate([g[2] for g in gathered]))
                U.generateMesh(fetch=False)
                torch.cuda.synchronize()
                t_host.append((time.perf_counter() - t0) * 1e3)
        per_rank_t = [None] * world
        dist.all_gather_object(per_rank_t, (t_sh, nb, nv, owned.num_blocks))
        if rank == 0:
            t_res, (ub, uv) = device_ms(ctx, lambda: U.generateMesh(fetch=False), args.repeats)
        else:
            device_ms(ctx, lambda: None, args.repeats)
        if rank == 0:
            sh = [max(t[0][i] for t in per_rank_t) for i in range(args.repeats)]
            line = dict(probe="mesh_sharded", shape=shape, world=world, card=card(local),
                        blocks=[t[3] for t in per_rank_t], global_blocks=ub,
                        vertices_sharded=sum(t[2] for t in per_rank_t), vertices_resident=uv,
                        sharded_ms_max_over_ranks=round(min(sh[1:]), 3),
                        sharded_ms_all=[round(x, 3) for x in sh],
                        via_host_ms=round(min(t_host[1:]), 1),
                        via_host_ms_all=[round(x, 1) for x in t_host],
                        resident_ms=round(min(t_res[1:]), 3),
                        resident_ms_all=[round(x, 3) for x in t_res])
            print(json.dumps(line), flush=True)
            lines.append(line)
            U.close()
        keep += subs + [partial, owned]  # mapped into the peers until the communicator goes
        dist.barrier()
    if rank == 0 and args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            json.dump(lines, f, indent=1)
    capi.check(capi.load().cg_comm_destroy(ctx._h))
    dist.barrier()
    for L in keep:
        L.close()
    ctx.close()
    dist.destroy_process_group()


if __name__ == "__main__":
    main()
