"""Multi-GPU plan of the server's global merge (DESIGN.md "Multi-GPU", SURVEY.md §8e).

The reference re-projects every submap of every robot into one global TSDF on one CPU thread
(cblox getProjectedMap(), reached from coxgraph/src/server/visualizer/server_visualizer.cpp:
123-126).  Here the submaps are sharded over the ranks of one box (one process per GPU):

  1. every rank projects ITS submaps into a *partial* global layer (no communication);
  2. a global block is owned by rank ``cg_block_owner(index) % world``; each rank packs its
     partial blocks grouped by owner (``cg_layer_pack_by_owner``);
  3. one all-to-all moves the records to their owners (NCCL over NVLink; P2P send/recv under
     gloo, which is what the CPU tests exercise);
  4. the owner folds the received records in ascending source-rank order with the 2-argument
     mergeLayerAintoLayerB (``cg_layer_merge_packed``).

Integration needs none of this: robots (and their submaps) are independent, so they are simply
assigned to ranks.  torch.distributed is plumbing only; the record format, the owner function and
every kernel live behind the C ABI.
"""
import ctypes as C

import numpy as np

from . import capi

RECORD_BYTES = capi.PACKED_BLOCK_BYTES


def assign_robots(num_robots, world_size):
    """robot r is fused on rank r % world_size (C3: one robot per GPU)."""
    return [[r for r in range(num_robots) if r % world_size == rank] for rank in range(world_size)]


def assign_submaps(num_robots, submaps_per_robot, world_size):
    """Global submap ids handled by each rank.  A robot's consecutive submaps stay together so
    that most of their mutual overlap is resolved inside one partial layer."""
    robots = assign_robots(num_robots, world_size)
    return [[r * submaps_per_robot + s for r in robots[rank] for s in range(submaps_per_robot)]
            for rank in range(world_size)]


def block_owners(block_idx, world_size):
    """Owner rank of every block index ([B,3] int32), computed by the library's own hash."""
    lib = capi.load()
    idx = np.ascontiguousarray(block_idx, np.int32).reshape(-1, 3)
    return np.array([lib.cg_block_owner(int(x), int(y), int(z), int(world_size))
                     for x, y, z in idx], dtype=np.int32)


def _all_gather_counts(send_counts, group):
    import torch
    import torch.distributed as dist
    world = dist.get_world_size(group)
    dev = "cuda" if dist.get_backend(group) == "nccl" else "cpu"
    mine = torch.tensor(send_counts, dtype=torch.int64, device=dev)
    out = [torch.empty_like(mine) for _ in range(world)]
    dist.all_gather(out, mine, group=group)
    return torch.stack(out).cpu().numpy()          # [src, dst]


def exchange_records(send, send_counts, group=None):
    """All-to-all of packed block records.

    send: uint8 tensor [n, RECORD_BYTES], rows grouped by destination rank (ascending);
    send_counts[d] rows go to rank d.  Returns (recv [m, RECORD_BYTES] grouped by SOURCE rank
    in ascending order, recv_counts)."""
    import torch
    import torch.distributed as dist
    world = dist.get_world_size(group)
    rank = dist.get_rank(group)
    assert send.dtype == torch.uint8 and send.dim() == 2 and send.shape[1] == RECORD_BYTES
    assert len(send_counts) == world and sum(send_counts) == send.shape[0]
    matrix = _all_gather_counts(list(send_counts), group)
    recv_counts = [int(matrix[src, rank]) for src in range(world)]
    recv = torch.empty((sum(recv_counts), RECORD_BYTES), dtype=torch.uint8, device=send.device)
    if dist.get_backend(group) == "nccl":
        dist.all_to_all_single(recv, send, output_split_sizes=recv_counts,
                               input_split_sizes=[int(c) for c in send_counts], group=group)
        return recv, recv_counts
    # generic path (gloo): pairwise exchange
    send_off = np.concatenate([[0], np.cumsum(send_counts)]).astype(int)
    recv_off = np.concatenate([[0], np.cumsum(recv_counts)]).astype(int)
    recv[recv_off[rank]:recv_off[rank + 1]] = send[send_off[rank]:send_off[rank + 1]]
    ops = []
    for peer in range(world):
        if peer == rank:
            continue
        if send_counts[peer]:
            ops.append(dist.P2POp(dist.isend, send[send_off[peer]:send_off[peer + 1]].contiguous(),
                                  peer, group=group))
        if recv_counts[peer]:
            ops.append(dist.P2POp(dist.irecv, recv[recv_off[peer]:recv_off[peer + 1]], peer,
                                  group=group))
    if ops:
        for req in dist.batch_isend_irecv(ops):
            req.wait()
    return recv, recv_counts


def gather_global(partial_layer, owned_layer, group=None):
    """Steps 2-4 on the GPU: pack `partial_layer` by owner, exchange, fold into `owned_layer`.
    Returns (blocks sent per destination, blocks received per source)."""
    import torch
    import torch.distributed as dist
    lib = capi.load()
    world = dist.get_world_size(group)
    n = partial_layer.num_blocks
    dev = torch.device("cuda", partial_layer.ctx.device)
    send = torch.empty((max(n, 1), RECORD_BYTES), dtype=torch.uint8, device=dev)
    counts = (C.c_uint64 * world)()
    capi.check(lib.cg_layer_pack_by_owner(partial_layer._h, world, C.c_void_p(send.data_ptr()),
                                          n, counts))
    send_counts = [int(c) for c in counts]
    torch.cuda.current_stream(dev).synchronize()
    recv, recv_counts = exchange_records(send[:n], send_counts, group)
    torch.cuda.current_stream(dev).synchronize()
    if recv.shape[0]:
        capi.check(lib.cg_layer_merge_packed(owned_layer._h, C.c_void_p(recv.data_ptr()),
                                             recv.shape[0]))
    return send_counts, recv_counts


def project_sharded(local_submaps, local_poses, partial_layer, owned_layer, group=None):
    """getProjectedMap() over all ranks: every rank passes the submaps assigned to it."""
    from .api import getProjectedMap
    partial_layer.removeAllBlocks()
    if len(local_submaps):
        getProjectedMap(local_submaps, local_poses, partial_layer)
    return gather_global(partial_layer, owned_layer, group)


def init_native(ctx, group=None):
    """cg_comm_init for every rank of a torch.distributed group: rank 0's ncclGetUniqueId goes
    round with broadcast_object_list (host plumbing only; the exchange itself is in the library,
    csrc/comm.cu)."""
    import torch.distributed as dist
    from .api import commInit, commUniqueId
    rank, world = dist.get_rank(group), dist.get_world_size(group)
    box = [commUniqueId() if rank == 0 else None]
    dist.broadcast_object_list(box, src=0, group=group)
    commInit(ctx, box[0], rank, world)


def project_sharded_native(local_submaps, local_poses, partial_layer, owned_layer):
    """project_sharded through the C ABI alone (cg_project_submaps_sharded): owner-pull over
    NVLink peer memory, no torch in the data path.  Needs init_native(ctx) once."""
    from .api import getProjectedMapSharded
    getProjectedMapSharded(local_submaps, local_poses, partial_layer, owned_layer)


def mesh_sharded(owned_layer, min_weight=1e-4, use_color=True, only_updated=False, fetch=True):
    """The mesh half of saveAndPubCombinedMesh over all ranks (cg_layer_mesh_sharded), after
    project_sharded_native: every rank meshes the blocks of its owned layer where they lie, reading
    the one-block halo from the peers.  Returns Layer.generateMesh's tuple for this rank's blocks;
    merged by block index, the ranks' results equal generateMesh of the gathered map."""
    from .api import generateMeshSharded
    return generateMeshSharded(owned_layer, min_weight, use_color, only_updated, fetch)
