#!/usr/bin/env python
"""Timing of the combined mesh of a sharded global map on one root rank (saveAndPubCombinedMesh's
output on several GPUs), one process per GPU (torchrun, NCCL), root = rank 0:

  sharded    cg_layer_mesh_sharded on every rank (count query): device time, maximum over ranks;
  gather     cg_mesh_gather_sharded to the root (count query): event time on the stream, maximum
             over the ranks (it includes the call's two host synchronisations);
  connect    cg_mesh_connect of the gathered mesh on the root (count query, the weld runs whole);
  via host   today's alternative: every rank downloads its owned layer, the root gathers them
             through the host, uploads them into one layer and runs cg_layer_mesh + cg_mesh_connect
             (host clock from a barrier to the end of the weld on the root);
  resident   cg_layer_mesh + cg_mesh_connect of that gathered layer, already resident on one GPU
             (device time);
  bytes      what the gather moves into the root: 12 B of block index and 4 B of vertex range per
             block, 28 B per vertex (position, normal, colour), summed over the other ranks.

  python -m torch.distributed.run --nnodes=1 --nproc-per-node N --master-addr 127.0.0.1 \\
      --master-port 29542 scripts/mesh_gather_probe.py [--out result.json]

Shapes: C2 (every rank's submaps cover the same room) and C3 (one robot per rank on the corridor
scene, robots 128 m apart), the shapes of scripts/mesh_sharded_probe.py.  Prints one JSON line per
shape, with the card's name and power limit read in the same run.
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
from coxgraph_b200.api import gatherMeshSharded, getProjectedMapSharded  # noqa: E402
from mesh_sharded_probe import card, device_ms  # noqa: E402
from multigpu_mesh_check import shape_submaps  # noqa: E402


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
    R = args.repeats
    for shape, per_rank, robot_per_rank in (("C2", args.c2_submaps, False),
                                            ("C3", args.c3_submaps, True)):
        subs, poses = shape_submaps(ctx, shape, rank, world, per_rank, frames=10, stride=1,
                                    robot_per_rank=robot_per_rank)
        partial = Layer(ctx, 0.05, max_blocks=65536)
        owned = Layer(ctx, 0.05, max_blocks=65536)
        getProjectedMapSharded(subs, poses, partial, owned)
        t_sh, t_ga, t_co = [], [], []
        for _ in range(R):
            t, (nb, nv) = device_ms(ctx, lambda: sharding.mesh_sharded(owned, fetch=False), 1)
            t_sh += t
            t, (gb, gv) = device_ms(ctx, lambda: gatherMeshSharded(ctx, 0, fetch=False), 1)
            t_ga += t
            t, _ = device_ms(ctx, lambda: owned.getConnectedMesh(fetch=False) if rank == 0 else None, 1)
            t_co += t
        conn = owned.getConnectedMesh(fetch=False) if rank == 0 else None
        # today's alternative: the owned layers through the host to one GPU, mesh and weld there
        t_host = []
        U = None
        for _ in range(max(2, R // 2)):
            dist.barrier()
            t0 = time.perf_counter()
            gathered = [None] * world
            dist.all_gather_object(gathered, owned.download())
            if rank == 0:
                gi = np.concatenate([g[0] for g in gathered])
                if U is None:
                    U = Layer(ctx, 0.05, max_blocks=max(len(gi), 1) * 2)
                U.clear()
                U.upload(gi, np.concatenate([g[1] for g in gathered]),
                         np.concatenate([g[2] for g in gathered]))
                U.generateMesh(fetch=False)
                U.getConnectedMesh(fetch=False)
                torch.cuda.synchronize()
                t_host.append((time.perf_counter() - t0) * 1e3)
        per_rank_t = [None] * world
        dist.all_gather_object(per_rank_t, (t_sh, t_ga, nb, nv, owned.num_blocks))
        if rank == 0:
            t_res, (ub, uv) = device_ms(ctx, lambda: (U.generateMesh(fetch=False),
                                                      U.getConnectedMesh(fetch=False))[0], R)
        else:
            device_ms(ctx, lambda: None, R)
        if rank == 0:
            sh = [max(t[0][i] for t in per_rank_t) for i in range(R)]
            ga = [max(t[1][i] for t in per_rank_t) for i in range(R)]
            moved = sum(16 * t[2] + 4 + 28 * t[3] for r, t in enumerate(per_rank_t) if r != 0 and t[2])
            line = dict(probe="mesh_gather", shape=shape, world=world, card=card(local),
                        blocks=[t[4] for t in per_rank_t], global_blocks=gb, global_vertices=gv,
                        resident_blocks=ub, resident_vertices=uv, connected_vertices=conn[0],
                        bytes_to_root=moved,
                        sharded_ms_max_over_ranks=round(min(sh[1:]), 3),
                        gather_ms_max_over_ranks=round(min(ga[1:]), 3),
                        gather_ms_all=[round(x, 3) for x in ga],
                        connect_root_ms=round(min(t_co[1:]), 3),
                        via_host_ms=round(min(t_host[1:]), 1),
                        via_host_ms_all=[round(x, 1) for x in t_host],
                        resident_mesh_connect_ms=round(min(t_res[1:]), 3))
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
