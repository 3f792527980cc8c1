#!/usr/bin/env python
"""bench.py — TSDF points integrated/s and submap-merge voxels/s (BASELINE.json metric).

Workload (BASELINE.json configs[1], "two-client CVG-experiment shape"): robots x submaps of 25
synthetic 640x480 depth frames each, 5 cm voxels, 16 cm truncation, Merged integrator, every
fused submap merged into the rank's global TSDF.  One STEP = clear the submap layer, fuse the 25
frames of one submap (7.68 M points) into it, merge it into the global layer.

  python bench.py --gpus N --steps K --warmup W              our arm (CUDA, C ABI), config C2
  python bench.py --config C1|C3|C4|C5 ...                   the other BASELINE.json configs
  python bench.py --impl reference --gpus N --steps K ...    the CPU oracle port, all host threads

Multi-GPU (torchrun, one rank per GPU): robots shard over ranks, no data-path collective in the
timed region (weak scaling); time = max over ranks.
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

FRAMES_PER_SUBMAP = 25
VOXEL_SIZE = 0.05
CFG = dict(default_truncation_distance=0.16, max_ray_length_m=5.0, min_ray_length_m=0.1,
           use_const_weight=1, method=1)
WORKLOAD = ("C2 two-client CVG shape: per step one submap = 25 x 640x480 depth frames "
            "(7.68 M points), 5 cm voxels, 16 cm truncation, merged integrator, voxel carving, "
            "fused into a cleared submap layer then merged into the global TSDF")
BLOCK_BYTES = 49152
# the `config` object of the JSON line: the same for both arms (the driver compares them)
CONFIG = {"workload": WORKLOAD,
          "l2": "no explicit flush: each step streams > 300 MB of fresh points, keys and update "
                "lists (L2 is 126 MB) and a different submap than the step before"}


# ----------------------------------------------------------------------------- helpers
class ClockSampler:
    """SM clock and throttle reasons sampled DURING the timed region: NVML polled from a thread
    every 2 ms (the timed region is tens of ms, too short for `nvidia-smi -lms`)."""
    REASONS = {0x8: "hw_slowdown", 0x40: "hw_thermal_slowdown", 0x20: "sw_thermal_slowdown",
               0x4: "sw_power_cap"}

    def __init__(self, gpu_index):
        self.gpu = gpu_index
        self.sm, self.reasons, self.max_mhz = [], set(), None
        self._stop = threading.Event()
        self.thread = None
        self.err = None

    def _run(self):
        try:
            pynvml, h, get_reasons = self._nvml
            while True:
                self.sm.append(float(pynvml.nvmlDeviceGetClockInfo(h, pynvml.NVML_CLOCK_SM)))
                bits = int(get_reasons(h))
                for bit, name in self.REASONS.items():
                    if bits & bit:
                        self.reasons.add(name)
                if self._stop.wait(0.001):
                    break
        except Exception as e:  # noqa: BLE001 - reported in the JSON line
            self.err = f"nvml unavailable: {e}"

    def start(self):
        """NVML is initialised here, before the timed region; the thread only polls."""
        try:
            import pynvml
            pynvml.nvmlInit()
            h = pynvml.nvmlDeviceGetHandleByIndex(self.gpu)
            self.max_mhz = float(pynvml.nvmlDeviceGetMaxClockInfo(h, pynvml.NVML_CLOCK_SM))
            get_reasons = getattr(pynvml, "nvmlDeviceGetCurrentClocksEventReasons", None) or \
                pynvml.nvmlDeviceGetCurrentClocksThrottleReasons
            self._nvml = (pynvml, h, get_reasons)
        except Exception as e:  # noqa: BLE001
            self.err = f"nvml unavailable: {e}"
            return
        self.thread = threading.Thread(target=self._run, daemon=True)
        self.thread.start()

    def stop(self):
        self._stop.set()
        if self.thread:
            self.thread.join(timeout=2)
        out = {"sm_mhz": float(np.median(self.sm)) if self.sm else None,
               "sm_max_mhz": self.max_mhz, "samples": len(self.sm),
               "reasons": sorted(self.reasons)}
        if self.err:
            out["reasons"] = out["reasons"] + [self.err]
        return out


def measured_peak_gbs():
    try:
        with open(os.path.join(ROOT, "MEASURED_PEAKS.json")) as f:
            return float(json.load(f)["hbm_gbs"]), "measured (MEASURED_PEAKS.json)"
    except Exception:
        return 6650.0, "fallback (B200_PROFILING.md)"


def stage_alg_bytes(stage, n_pts, rays, pairs, general, blocks, b_in=0, b_out=0):
    """Compulsory HBM bytes of one pipeline stage (what it must read and write once; DESIGN.md
    §7.1), per step.  (ray, block) segments are not in the job statistics: estimated as visits /
    11.5, the ratio ncu shows at the C2 shape."""
    segs = pairs / 11.5
    table = {
        "point_keys": 20 * n_pts, "bundle_sort": 16 * n_pts, "bundle_scan": 8 * n_pts + 4 * rays,
        "gather_sorted": 40 * n_pts, "bundle_order": 12 * rays,
        "fold_wide": 8 * n_pts + 12 * rays, "fold_bundles": 8 * n_pts + 12 * rays,
        "bundle_rays": 48 * rays, "ray_scan": 24 * rays, "walk_segments": 24 * rays + 40 * segs,
        "segment_sort": 16 * segs, "block_accumulate": 40 * segs + 8 * general + 65536 * blocks,
        "pair_sort": 16 * general, "segments": 12 * general, "voxel_update": 44 * general,
        "replay_wide": 44 * general, "finalize": 98304 * blocks, "merge_mark": 8 * b_in,
        "merge_resample": BLOCK_BYTES * (b_in + 2 * b_out),
    }
    return float(table.get(stage, 0.0))


def roofline_record(prof, steps, step_ms, bytes_step, per_step, traffic_file="traffic.json"):
    """The `roofline` object of the JSON line.  The dominant stage is chosen over ALL stages of the
    step, library kernels (cub sorts / selects: no own launches) included and flagged; `frac` is
    that stage's own algorithmic bytes over its own time; `step_frac` — the contract figure of
    SURVEY.md §8d over the whole step — is the headline."""
    peak, peak_src = measured_peak_gbs()
    stages = {k: v for k, v in prof.items() if k != "transfer" and v[0] > 0}
    top = max(stages, key=lambda k: stages[k][0])
    top_ms = stages[top][0] / steps
    alg = stage_alg_bytes(top, **per_step)
    achieved = alg / (top_ms * 1e-3) / 1e9
    traffic = None
    try:  # dram bytes of one launch of that stage from the ncu capture of the same command
        if traffic_file:
            with open(os.path.join(ROOT, "profiles", traffic_file)) as f:
                traffic = json.load(f).get(top)
    except Exception:  # noqa: BLE001
        pass
    lib_ms = sum(v[0] for v in stages.values() if v[1] == 0) / steps
    return {"bound": "hbm", "kernel": top, "library_kernel": stages[top][1] == 0,
            "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak,
            "traffic": traffic, "peak_source": peak_src,
            "algorithmic_bytes_per_launch": alg, "ms_per_launch": top_ms,
            "step_frac": bytes_step / (step_ms * 1e-3) / 1e9 / peak,
            "step_algorithmic_bytes": bytes_step,
            "library_stages_ms_per_step": lib_ms,
            "note": "frac = the dominant stage's own compulsory bytes / its own time (a stage is "
                    "one kernel or one library call); step_frac = the step's contract bytes "
                    "(16 N + 2 x 49152 B_touched per call, 49152 (B_in + 2 B_out) per merge) / "
                    "the whole step: the headline fraction"}


def submap_of_step(step, rank, world):
    """(robot, submap) fused at `step` on `rank`.  The 2 x 20 submaps of the C2 shape shard over
    the ranks; every rank alternates between the two robots (their scenes differ in cost), so the
    per-rank work is the same at every N (weak scaling)."""
    return (step + rank) % 2, (step // 2 + 3 * rank) % 20


def host_frames(robot, submap, frames, device):
    from coxgraph_b200 import synth
    fr = synth.submap_frames(robot, submap % 20, frames, device=device)
    poses = np.stack([T for (T, _, _) in fr]).astype(np.float32)
    return poses, [p for (_, p, _) in fr], [c for (_, _, c) in fr]


# ----------------------------------------------------------------------------- reference arm
def run_reference(args, rank, world):
    """The reference's CPU implementation of the path (restated: oracle/, kind 'port'), with all
    host threads, on a bounded sample of every step."""
    if rank != 0:
        return
    from coxgraph_b200 import synth
    from oracle import oracle_py as orc
    threads = os.cpu_count() or 1
    ocfg = orc.default_config(**CFG)
    sample_frames = args.ref_frames
    og = orc.Layer(VOXEL_SIZE)
    t_int = t_merge = 0.0
    pts_total = vox_total = 0
    t_region = 0.0
    for step in range(args.warmup + args.steps):
        robot, sm = submap_of_step(step, 0, 1)
        poses, pts, cols = host_frames(robot, sm, sample_frames, "cpu")
        pts = [p.numpy() for p in pts]
        cols = [c.numpy() for c in cols]
        ol = orc.Layer(VOXEL_SIZE)
        t0 = time.perf_counter()
        for f in range(sample_frames):
            ol.integrate(ocfg, poses[f], pts[f], cols[f], threads=threads)
        t1 = time.perf_counter()
        og.merge_from(ol, synth.robot_map_offset(robot), threads=threads)
        t2 = time.perf_counter()
        if step >= args.warmup:
            t_int += t1 - t0
            t_merge += t2 - t1
            t_region += t2 - t0
            pts_total += sum(len(p) for p in pts)
            vox_total += 4096 * ol.num_blocks
    value = pts_total / t_region
    sample = (f"{sample_frames} of {FRAMES_PER_SUBMAP} frames per step "
              f"({sample_frames * 307200} points), then merge of that partial submap")
    line = {
        "impl": "reference", "metric": "tsdf_points_integrated_per_s", "value": value,
        "unit": "points/s", "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup,
        "ms_per_step": 1e3 * t_region / args.steps, "higher_is_better": True, "scaling": "weak",
        "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        # the same `config` object as our arm prints (the driver compares them); what this run
        # sampled is in cpu_baseline.sample
        "config": dict(CONFIG),
        "integrate": {"value": pts_total / t_int, "unit": "points/s"},
        "merge": {"value": vox_total / t_merge, "unit": "voxels/s"},
        "cpu_baseline": {"value": value, "unit": "points/s", "cores": threads, "kind": "port",
                         "sample": sample},
        "e2e": {"value": value, "unit": "points/s", "h2d_bytes_per_step": 0,
                "d2h_bytes_per_step": 0},
    }
    print(json.dumps(line), flush=True)


def layer_diff(got, ref):
    """Margins of a CUDA layer against the oracle's: block sets, max |d_d| / tol, max |d_w| / tol
    (tol = max(1e-5, 1e-4 |ref|), BASELINE.json north_star) and the colour LSB histogram."""
    gi, gv, _ = got
    ri, rv, _ = ref
    out = {"blocks": int(len(gi)), "blocks_oracle": int(len(ri)),
           "block_sets_equal": bool(gi.shape == ri.shape and np.array_equal(gi, ri))}
    if not out["block_sets_equal"]:
        out["within_tolerance"] = False
        return out
    for name in ("distance", "weight"):
        g, r = gv[name].astype(np.float64), rv[name].astype(np.float64)
        tol = np.maximum(1e-5, 1e-4 * np.abs(r))
        out[f"max_{name}_err_over_tol"] = float((np.abs(g - r) / tol).max(initial=0.0))
    dc = np.abs(gv["rgba"].astype(np.int16) - rv["rgba"].astype(np.int16)).max(axis=-1)
    out["colour_lsb_hist"] = [int(x) for x in np.bincount(dc.ravel(), minlength=4)[:8]]
    out["within_tolerance"] = bool(out["max_distance_err_over_tol"] <= 1.0 and
                                   out["max_weight_err_over_tol"] <= 1.0 and dc.max(initial=0) <= 1)
    return out


# whole blocks per layer whose voxels --dump-outputs writes: with every block index of the two C2
# layers (at most 4096 + 32768 blocks) that stays under 53 MB in all
DUMP_BLOCKS = 256


def dump_outputs(out_dir, layers, stats):
    """--dump-outputs: what the timed path hands its caller after its last step, as
    out_dir/<name>.npy.  Per layer: every block index (the (z,y,x) order of download()) and its
    flags, and distance, weight and rgba of DUMP_BLOCKS blocks (all of them when there are fewer),
    a seeded choice of rows of that list stored as <layer>_sample_rows; the voxel fields are float32,
    indices, flags and counters float64.  Per call statistics struct: one scalar per field."""
    os.makedirs(out_dir, exist_ok=True)
    arrays = {}
    for name, layer in layers.items():
        idx, vox, flags = layer.download()
        rows = np.arange(len(idx))
        if len(idx) > DUMP_BLOCKS:
            rows = np.sort(np.random.default_rng(0).choice(len(idx), DUMP_BLOCKS, replace=False))
        arrays[f"{name}_block_idx"] = idx.astype(np.float64)
        arrays[f"{name}_flags"] = flags.astype(np.float64)
        arrays[f"{name}_sample_rows"] = rows.astype(np.float64)
        arrays[f"{name}_distance"] = vox["distance"][rows].astype(np.float32)
        arrays[f"{name}_weight"] = vox["weight"][rows].astype(np.float32)
        arrays[f"{name}_rgba"] = vox["rgba"][rows].astype(np.float32)
    for name, st in stats.items():
        for field, _ in st._fields_:
            arrays[f"{name}_{field}"] = np.array(getattr(st, field), np.float64)
    for name, a in arrays.items():
        np.save(os.path.join(out_dir, f"{name}.npy"), a)
    return arrays


def time_sharded(subs, poses, partial, owned, ctx, barrier, max_over_ranks, sum_over_ranks, vox,
                 stream):
    """The server's global merge over all ranks, timed on the device (max over ranks): every rank
    projects its submaps into a partial layer and the partial blocks go to their owners.  Two
    exchanges are timed: `native` = cg_project_submaps_sharded (csrc/comm.cu: the owner's fold
    kernel pulls the blocks over NVLink peer memory, NCCL only as bootstrap and barrier, no host
    in the data path) — the headline — and `packed` = pack + NCCL all-to-all through
    torch.distributed + fold (round 1's path)."""
    import torch
    from coxgraph_b200 import sharding
    out = {"unit": "voxels/s"}
    native_err = None
    try:
        sharding.init_native(ctx)
    except Exception as exc:  # noqa: BLE001 - reported in the JSON line, the packed path still runs
        native_err = repr(exc)
    for name in ("native", "packed"):
        if name == "native" and native_err:
            out["native_error"] = native_err
            continue
        times = []
        for it in range(5):
            owned.clear()
            barrier()
            a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            a.record(stream)
            if name == "native":
                sharding.project_sharded_native(subs, poses, partial, owned)
            else:
                sharding.project_sharded(subs, poses, partial, owned)
            b.record(stream)
            barrier()
            times.append(max_over_ranks(a.elapsed_time(b)))
        ms = min(times[1:])
        out[name] = {"ms": ms, "value": vox / (ms * 1e-3),
                     "global_blocks": int(sum_over_ranks(float(owned.num_blocks)))}
    best = "native" if "native" in out else "packed"
    out.update(value=out[best]["value"], ms=out[best]["ms"], exchange=best,
               collective="owner-pull over NVLink peer memory (CUDA IPC), NCCL barrier"
               if best == "native" else "nccl all_to_all_single of packed blocks")
    return out


def sharded_parity(subs, poses, partial, owned, rank, world):
    """Parity evidence for the multi-GPU merge inside the bench run (the pytest for it is skipped
    on one-GPU boxes): the union of the ranks' owned layers after a sharded projection of a few
    submaps per rank, against the SINGLE-PROCESS oracle left fold of the same submaps in rank-major
    order (SURVEY.md §8e H6: the sharded plan re-associates the merge).  Rank 0 runs the oracle."""
    import torch.distributed as dist
    from coxgraph_b200 import sharding
    owned.clear()
    if partial.ctx.has_comm:
        sharding.project_sharded_native(subs, poses, partial, owned)
    else:
        sharding.project_sharded(subs, poses, partial, owned)
    mine = {"owned": owned.download(), "subs": [L.download() for L in subs],
            "poses": np.asarray(poses)}
    gathered = [None] * world if rank == 0 else None
    dist.gather_object(mine, gathered, dst=0)
    if rank != 0:
        return None
    from oracle import oracle_py as orc
    og = orc.Layer(VOXEL_SIZE)
    for r in range(world):
        for (idx, vox, fl), T in zip(gathered[r]["subs"], gathered[r]["poses"]):
            ol = orc.Layer(VOXEL_SIZE)
            ol.upload(idx, vox, fl)
            og.merge_from(ol, T)
    idx = np.concatenate([g["owned"][0] for g in gathered])
    vox = np.concatenate([g["owned"][1] for g in gathered])
    order = np.lexsort((idx[:, 0], idx[:, 1], idx[:, 2]))
    out = layer_diff((idx[order], vox[order], None), og.download())
    out["submaps"] = len(subs) * world
    out["oracle"] = "single-process left fold, rank-major submap order"
    return out


# ----------------------------------------------------------------------------- our arm
def run_ours(args, rank, world, local_rank):
    import torch
    import torch.distributed as dist
    from coxgraph_b200 import (Context, Layer, TsdfIntegrator, TsdfIntegratorConfig,
                               mergeLayerAintoLayerB, synth)

    try:  # run (and first-touch the pinned buffers) on the CPUs next to this rank's GPU
        import pynvml
        pynvml.nvmlInit()
        pynvml.nvmlDeviceSetCpuAffinity(pynvml.nvmlDeviceGetHandleByIndex(local_rank))
    except Exception:  # noqa: BLE001 - affinity is an optimisation only
        pass
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)
    # the context's stream at high priority: with pipelined calls its kernels (the second half of
    # the current job, the merge) are scheduled ahead of the next job's first half on the
    # library's second stream, which has default priority
    stream = torch.cuda.Stream(device=dev, priority=int(os.environ.get("CG_BENCH_STREAM_PRIORITY", "-1")))
    torch.cuda.set_stream(stream)
    ctx = Context(local_rank, stream=stream.cuda_stream)
    gcfg = TsdfIntegratorConfig(**CFG)
    submap = Layer(ctx, VOXEL_SIZE, max_blocks=4096)
    glob = Layer(ctx, VOXEL_SIZE, max_blocks=32768)
    integ = TsdfIntegrator(gcfg, submap)

    # ---- synthetic inputs (generated on the GPU with torch, outside every timed region)
    total_steps = args.warmup + args.steps
    pool_n = min(total_steps, args.pool)
    pool = []
    for s in range(pool_n):
        robot, sm = submap_of_step(s, rank, world)
        poses, pts, cols = host_frames(robot, sm, FRAMES_PER_SUBMAP, dev)
        d_pts = torch.cat(pts).contiguous()
        d_cols = torch.cat(cols).contiguous()
        offs = np.cumsum([0] + [len(p) for p in pts]).astype(np.uint64)
        h_pts = torch.empty(d_pts.shape, dtype=d_pts.dtype, pin_memory=True).copy_(d_pts)
        h_cols = torch.empty(d_cols.shape, dtype=d_cols.dtype, pin_memory=True).copy_(d_cols)
        pool.append(dict(robot=robot, poses=poses, d_pts=d_pts, d_cols=d_cols, offs=offs,
                         h_pts=h_pts.numpy(), h_cols=h_cols.numpy(),
                         T_M_S=synth.robot_map_offset(robot), n=int(offs[-1])))
    torch.cuda.synchronize()

    # ---- untimed accounting pass: per-frame B_touched (the byte model's definition) and the
    # merge block counts, for every pool submap
    for e in pool:
        if args.profile_mode:
            e.update(bytes_integrate=0, blocks_in=0, bytes_merge=0, voxels_in=0, rays=0, pairs=0,
                     general=0, per_frame_ms=0.0, per_frame_queued_ms=0.0)
            continue
        submap.clear()
        touched = 0
        ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        ev0.record(stream)
        for f in range(FRAMES_PER_SUBMAP):
            a, b = int(e["offs"][f]), int(e["offs"][f + 1])
            st = integ.integratePointCloud(e["poses"][f], e["d_pts"][a:b], e["d_cols"][a:b])
            touched += st.blocks_touched
        ev1.record(stream)
        torch.cuda.synchronize()
        e["per_frame_ms"] = ev0.elapsed_time(ev1) / FRAMES_PER_SUBMAP
        # the same 25 calls with the subscriber queue two deep (voxblox_ros TsdfServer holds the
        # next PointCloud2 while the current one is integrated): the layer-independent first half
        # of frame f+1 is queued before frame f is completed (cg_prepare_batch_device with one
        # frame + cg_integrate_prepared); same result as the plain calls
        submap.clear()

        def one(f):
            a, b = int(e["offs"][f]), int(e["offs"][f + 1])
            return (e["poses"][f:f + 1], e["d_pts"][a:b], e["d_cols"][a:b],
                    np.array([0, b - a], np.uint64))
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        integ.prepareBatch(0, *one(0))
        for f in range(FRAMES_PER_SUBMAP):
            if f + 1 < FRAMES_PER_SUBMAP:
                integ.prepareBatch((f + 1) % 2, *one(f + 1))
            integ.integratePrepared(f % 2)
        torch.cuda.synchronize()
        e["per_frame_queued_ms"] = (time.perf_counter() - t0) * 1e3 / FRAMES_PER_SUBMAP
        e["bytes_integrate"] = 16 * e["n"] + 2 * BLOCK_BYTES * touched
        submap.clear()
        st = integ.integrateBatch(e["poses"], e["d_pts"], e["d_cols"], e["offs"])
        e["rays"], e["pairs"] = int(st.rays), int(st.voxel_updates)
        e["general"] = int(st.general_updates)
        e["blocks_in"] = submap.num_blocks
        glob.clear()
        ms = mergeLayerAintoLayerB(submap, e["T_M_S"], glob)
        e["bytes_merge"] = BLOCK_BYTES * (ms.blocks_in + 2 * ms.blocks_out)
        e["voxels_in"] = 4096 * ms.blocks_in

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def max_over_ranks(x):
        if world == 1:
            return x
        t = torch.tensor([x], dtype=torch.float64, device=dev)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item())

    def sum_over_ranks(x):
        if world == 1:
            return x
        t = torch.tensor([x], dtype=torch.float64, device=dev)
        dist.all_reduce(t, op=dist.ReduceOp.SUM)
        return float(t.item())

    def all_ranks(x):
        """x of every rank, in rank order (tells imbalance from stalls: SCALE runs)."""
        if world == 1:
            return [float(x)]
        t = torch.tensor([x], dtype=torch.float64, device=dev)
        out = [torch.zeros_like(t) for _ in range(world)]
        dist.all_gather(out, t)
        return [float(o.item()) for o in out]

    # pinned result buffers for the e2e leg (the fused submap layer, voxblox layout)
    out_idx = torch.empty((4096, 3), dtype=torch.int32, pin_memory=True).numpy()
    out_vox_t = torch.empty((4096, 4096 * 12), dtype=torch.uint8, pin_memory=True)
    from coxgraph_b200 import VOXEL_DTYPE
    out_vox = out_vox_t.numpy().view(VOXEL_DTYPE).reshape(4096, 4096)
    out_flags = torch.empty((4096,), dtype=torch.uint8, pin_memory=True).numpy()

    def step_device(e, ev=None):
        submap.clear()
        if ev:
            ev[0].record(stream)
        integ.integrateBatch(e["poses"], e["d_pts"], e["d_cols"], e["offs"])
        if ev:
            ev[1].record(stream)
        mst = mergeLayerAintoLayerB(submap, e["T_M_S"], glob)
        if ev:
            ev[2].record(stream)
        return mst

    def run_e2e(entries, pipelined=True):
        """Every step: H2D of its inputs from pinned host memory (cg_stage_batch_async, double
        buffered: the copy of step k+1 is queued before step k is fused), fuse, merge, D2H of the
        fused submap in voxblox layout.  pipelined: the first half of step k+1 (points -> rays,
        cg_prepare_batch_staged) also runs while step k is fused.  Returns the D2H bytes."""
        d2h = 0
        if entries:
            integ.stageBatch(0, entries[0]["h_pts"], entries[0]["h_cols"])
            if pipelined:
                integ.prepareStaged(0, 0, entries[0]["poses"], entries[0]["offs"])
        for k, e in enumerate(entries):
            if k + 1 < len(entries):
                nxt = entries[k + 1]
                integ.stageBatch((k + 1) % 2, nxt["h_pts"], nxt["h_cols"])
                if pipelined:
                    integ.prepareStaged((k + 1) % 2, (k + 1) % 2, nxt["poses"], nxt["offs"])
            submap.clear()
            if pipelined:
                integ.integratePrepared(k % 2)
            else:
                integ.integrateStaged(k % 2, e["poses"], e["offs"])
            mergeLayerAintoLayerB(submap, e["T_M_S"], glob)
            idx, vox, fl = submap.download(out=(out_idx, out_vox, out_flags))
            d2h += len(idx) * (BLOCK_BYTES + 13)
        return d2h

    def run_pipelined(entries):
        """Inputs resident in HBM; the first half of step k+1 (cg_prepare_batch_device) is queued
        before step k is completed (cg_integrate_prepared) and merged.  Returns the MergeStats
        of the last step."""
        mst = None
        if entries:
            e = entries[0]
            integ.prepareBatch(0, e["poses"], e["d_pts"], e["d_cols"], e["offs"])
        for k, e in enumerate(entries):
            if k + 1 < len(entries):
                n = entries[k + 1]
                integ.prepareBatch((k + 1) % 2, n["poses"], n["d_pts"], n["d_cols"], n["offs"])
            submap.clear()
            integ.integratePrepared(k % 2)
            mst = mergeLayerAintoLayerB(submap, e["T_M_S"], glob)
        return mst

    results = {}
    # "device": inputs resident in HBM, no instrumentation (-> value); "profiled": the same steps
    # with the library's stage timers on (-> stages_ms_per_step, roofline); "e2e": host buffers
    legs = ("device", "profiled", "e2e") if args.profile_mode else \
        ("device", "profiled", "pipelined", "e2e", "e2e_plain")
    headline_leg = "pipelined" if "pipelined" in legs else "device"   # the leg `value` reports
    for leg in legs:
        glob.clear()
        if leg in ("device", "profiled"):
            for s in range(args.warmup):
                step_device(pool[s % pool_n])
        elif leg == "pipelined":
            run_pipelined([pool[s % pool_n] for s in range(args.warmup)])
        else:
            run_e2e([pool[s % pool_n] for s in range(args.warmup)], pipelined=(leg == "e2e"))
        sampler = ClockSampler(local_rank)
        evs = [[torch.cuda.Event(enable_timing=True) for _ in range(3)] for _ in range(args.steps)]
        ev_a, ev_b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        launches0 = ctx.kernel_launches
        if leg == "profiled":
            ctx.reset_profile()
            ctx.set_profiling(True)
        sampler.start()
        barrier()
        ev_a.record(stream)
        d2h = 0
        last_merge = None
        if leg in ("device", "profiled"):
            for k in range(args.steps):
                # profile mode: the last un-instrumented step sits in an NVTX range, so that ncu
                # captures exactly one step (--nvtx --nvtx-include "cg_step/")
                mark = args.profile_mode and leg == "device" and k == args.steps - 1
                if mark:
                    torch.cuda.nvtx.range_push("cg_step")
                last_merge = step_device(pool[(args.warmup + k) % pool_n], evs[k])
                if mark:
                    torch.cuda.nvtx.range_pop()
        elif leg == "pipelined":
            last_merge = run_pipelined([pool[(args.warmup + k) % pool_n] for k in range(args.steps)])
        else:
            d2h = run_e2e([pool[(args.warmup + k) % pool_n] for k in range(args.steps)],
                          pipelined=(leg == "e2e"))
        ev_b.record(stream)
        barrier()
        clocks = sampler.stop()
        ctx.set_profiling(False)
        total_ms = max_over_ranks(ev_a.elapsed_time(ev_b))
        used = [pool[(args.warmup + k) % pool_n] for k in range(args.steps)]
        res = dict(total_ms=total_ms, clocks=clocks, launches=ctx.kernel_launches - launches0,
                   per_rank_ms=[v / args.steps for v in all_ranks(ev_a.elapsed_time(ev_b))],
                   points=sum_over_ranks(sum(e["n"] for e in used)),
                   h2d=sum(16 * e["n"] for e in used) / args.steps, d2h=d2h / args.steps)
        if leg in ("device", "profiled"):
            res["int_ms"] = max_over_ranks(sum(a.elapsed_time(b) for (a, b, _) in evs))
            res["merge_ms"] = max_over_ranks(sum(b.elapsed_time(c) for (_, b, c) in evs))
            res["voxels"] = sum_over_ranks(sum(e["voxels_in"] for e in used))
            res["bytes_int"] = sum(e["bytes_integrate"] for e in used)
            res["bytes_merge"] = sum(e["bytes_merge"] for e in used)
            if leg == "profiled":
                res["profile"] = ctx.profile()
        results[leg] = res
        if args.dump_outputs and rank == 0 and leg == headline_leg:
            # before the next leg clears the layers; integ.last_stats is the last step's
            dump_outputs(args.dump_outputs, {"submap": submap, "global": glob},
                         {"integrate": integ.last_stats, "merge": last_merge})

    # ---- server-side global merge at the C2 shape: 2 robots x 20 submaps projected into one
    # global TSDF with cblox getProjectedMap() semantics (one call, batched on the device)
    project = None
    if not args.profile_mode and args.project_submaps > 0:
        from coxgraph_b200 import getProjectedMap
        subs, T_all = [], []
        for k in range(args.project_submaps):
            e = pool[k % pool_n]
            L = Layer(ctx, VOXEL_SIZE, max_blocks=1024)
            TsdfIntegrator(gcfg, L).integrateBatch(e["poses"], e["d_pts"], e["d_cols"], e["offs"])
            subs.append(L)
            # every copy gets its own pose (as after a pose-graph update) so that the copies do
            # not fall on top of each other
            rng = np.random.default_rng(1000 + k)
            T_all.append(synth.perturb_pose(e["T_M_S"], rng, sigma_t=0.4, sigma_yaw_deg=10.0))
        T_all = np.stack(T_all)
        big = Layer(ctx, VOXEL_SIZE, max_blocks=65536)
        times = []
        for it in range(4):
            big.clear()
            a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            a.record(stream)
            st = getProjectedMap(subs, T_all, big, want_stats=(it == 3))
            b.record(stream)
            torch.cuda.synchronize()
            times.append(a.elapsed_time(b))
        ms = max_over_ranks(min(times[1:3]))
        vox = sum_over_ranks(4096.0 * sum(L.num_blocks for L in subs))
        project = {"value": vox / (ms * 1e-3), "unit": "voxels/s", "submaps": args.project_submaps,
                   "ms": ms, "blocks_in": int(st.blocks_in), "blocks_out": int(st.blocks_out),
                   "global_blocks": big.num_blocks,
                   "hbm_frac": BLOCK_BYTES * (st.blocks_in + 2 * st.blocks_out) / (ms * 1e-3) / 1e9 /
                   measured_peak_gbs()[0]}
        # after a pose-graph update that moved a tenth of the submaps: incremental re-projection
        # (bit-identical to the full rebuild), then the mesh of the device-resident map — what
        # saveAndPubCombinedMesh does next (server_visualizer.cpp:123-126)
        from coxgraph_b200 import reprojectSubmaps
        rng = np.random.default_rng(7)
        rep_ms = []
        for it in range(3):
            big.clear()
            getProjectedMap(subs, T_all, big)
            T_new = T_all.copy()
            for k in rng.choice(len(subs), max(1, len(subs) // 10), replace=False):
                T_new[k] = synth.perturb_pose(T_all[k], rng)
            a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            a.record(stream)
            _, rst = reprojectSubmaps(subs, T_all, T_new, big)
            b.record(stream)
            torch.cuda.synchronize()
            rep_ms.append(a.elapsed_time(b))
        project["reproject_10pct_moved"] = {
            "ms": max_over_ranks(min(rep_ms[1:])), "submaps_moved": int(rst.submaps_moved),
            "blocks_dirty": int(rst.blocks_dirty), "candidates": int(rst.candidates)}
        mesh_ms = []
        for it in range(3):
            t0 = time.perf_counter()
            mesh = big.generateMesh()
            mesh_ms.append((time.perf_counter() - t0) * 1e3)
        dev_ms = []
        for it in range(3):
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            big.generateMesh(fetch=False)
            dev_ms.append((time.perf_counter() - t0) * 1e3)
        project["mesh"] = {"ms_with_d2h": max_over_ranks(min(mesh_ms[1:])),
                           "ms_device_only": max_over_ranks(min(dev_ms[1:])),
                           "triangles": int(len(mesh[2]) // 3), "blocks": big.num_blocks,
                           "d2h_bytes": int(len(mesh[2]) * 28),
                           "layer_bytes_not_downloaded": int(big.num_blocks * BLOCK_BYTES)}
        project["esdf"] = time_esdf(big, max_over_ranks)
        if world > 1:
            # the server's global merge over all ranks: every rank projects its submaps into a
            # partial layer, one NCCL all-to-all moves the partial blocks to their owners, the
            # owners fold them (coxgraph_b200/sharding.py); timed on the device, max over ranks
            from coxgraph_b200 import sharding
            partial = Layer(ctx, VOXEL_SIZE, max_blocks=65536)
            owned = Layer(ctx, VOXEL_SIZE, max_blocks=65536)
            project["sharded"] = time_sharded(subs, T_all, partial, owned, ctx, barrier,
                                              max_over_ranks, sum_over_ranks, vox, stream)
            project["sharded"]["submaps_total"] = args.project_submaps * world
            project["sharded"]["parity"] = sharded_parity(
                subs[:args.parity_submaps], T_all[:args.parity_submaps], partial, owned, rank, world)
            partial.close()
            owned.close()
        for L in subs:
            L.close()
        big.close()

    # ---- two fusion jobs in flight on this GPU (two contexts on their own streams, two host
    # threads; ctypes drops the GIL during the calls): the robots of the C2 shape are independent,
    # and the stages of one job are latency-bound with few warps, so two jobs overlap.  Reported
    # beside `value` (which stays one job at a time); N = 1 only.
    two_jobs = None
    if world == 1 and not args.profile_mode and pool_n >= 2:
        try:
            import threading
            lanes = []
            for j in range(2):
                c2 = Context(local_rank)
                lanes.append((c2, Layer(c2, VOXEL_SIZE, max_blocks=4096),
                              Layer(c2, VOXEL_SIZE, max_blocks=32768), pool[j::2]))

            def run_lane(lane, steps):
                c2, sub2, glob2, ents = lane
                integ2 = TsdfIntegrator(gcfg, sub2)
                for k in range(steps):
                    e = ents[k % len(ents)]
                    sub2.clear()
                    integ2.integrateBatch(e["poses"], e["d_pts"], e["d_cols"], e["offs"])
                    mergeLayerAintoLayerB(sub2, e["T_M_S"], glob2)
                c2.synchronize()

            for lane in lanes:
                run_lane(lane, max(args.warmup, len(lane[3])))   # scratch buffers, key box
            torch.cuda.synchronize()
            threads = [threading.Thread(target=run_lane, args=(lane, args.steps)) for lane in lanes]
            t0 = time.perf_counter()
            for t in threads:
                t.start()
            for t in threads:
                t.join()
            torch.cuda.synchronize()
            dt = time.perf_counter() - t0
            pts2 = sum(lane[3][k % len(lane[3])]["n"] for lane in lanes for k in range(args.steps))
            two_jobs = {"value": pts2 / dt, "unit": "points/s", "jobs_in_flight": 2,
                        "ms_per_submap": dt * 1e3 / (2 * args.steps),
                        "timing": "wall clock around both threads, device synchronised on both sides"}
            # the same with each lane issuing the pipelined calls of `value` (the two clients of the
            # C2 shape, one context each)
            def run_lane_pipelined(lane, steps):
                c2, sub2, glob2, ents = lane
                integ2 = TsdfIntegrator(gcfg, sub2)
                e = ents[0]
                integ2.prepareBatch(0, e["poses"], e["d_pts"], e["d_cols"], e["offs"])
                for k in range(steps):
                    e = ents[k % len(ents)]
                    if k + 1 < steps:
                        n = ents[(k + 1) % len(ents)]
                        integ2.prepareBatch((k + 1) % 2, n["poses"], n["d_pts"], n["d_cols"], n["offs"])
                    sub2.clear()
                    integ2.integratePrepared(k % 2)
                    mergeLayerAintoLayerB(sub2, e["T_M_S"], glob2)
                c2.synchronize()

            for lane in lanes:
                run_lane_pipelined(lane, 3)
            torch.cuda.synchronize()
            threads = [threading.Thread(target=run_lane_pipelined, args=(lane, args.steps))
                       for lane in lanes]
            t0 = time.perf_counter()
            for t in threads:
                t.start()
            for t in threads:
                t.join()
            torch.cuda.synchronize()
            dt = time.perf_counter() - t0
            two_jobs["pipelined"] = {"value": pts2 / dt, "unit": "points/s",
                                     "ms_per_submap": dt * 1e3 / (2 * args.steps)}
            # the same with host buffers: every lane stages its next submap (pinned memory,
            # double buffered), fuses, merges and reads the fused submap back, like the e2e leg
            def run_lane_e2e(lane, steps, bufs):
                c2, sub2, glob2, ents = lane
                integ2 = TsdfIntegrator(gcfg, sub2)
                integ2.stageBatch(0, ents[0]["h_pts"], ents[0]["h_cols"])
                for k in range(steps):
                    e = ents[k % len(ents)]
                    if k + 1 < steps:
                        nxt = ents[(k + 1) % len(ents)]
                        integ2.stageBatch((k + 1) % 2, nxt["h_pts"], nxt["h_cols"])
                    sub2.clear()
                    integ2.integrateStaged(k % 2, e["poses"], e["offs"])
                    mergeLayerAintoLayerB(sub2, e["T_M_S"], glob2)
                    sub2.download(out=bufs)
                c2.synchronize()

            bufs = [(out_idx, out_vox, out_flags),
                    (torch.empty((4096, 3), dtype=torch.int32, pin_memory=True).numpy(),
                     torch.empty((4096, 4096 * 12), dtype=torch.uint8, pin_memory=True).numpy()
                     .view(VOXEL_DTYPE).reshape(4096, 4096),
                     torch.empty((4096,), dtype=torch.uint8, pin_memory=True).numpy())]
            for lane, b in zip(lanes, bufs):
                run_lane_e2e(lane, 3, b)
            torch.cuda.synchronize()
            threads = [threading.Thread(target=run_lane_e2e, args=(lane, args.steps, b))
                       for lane, b in zip(lanes, bufs)]
            t0 = time.perf_counter()
            for t in threads:
                t.start()
            for t in threads:
                t.join()
            torch.cuda.synchronize()
            dt = time.perf_counter() - t0
            two_jobs["e2e"] = {"value": pts2 / dt, "unit": "points/s",
                               "ms_per_submap": dt * 1e3 / (2 * args.steps)}
            for c2, sub2, glob2, _ in lanes:
                sub2.close()
                glob2.close()
                c2.close()
        except Exception as exc:  # noqa: BLE001 - an extra figure must not take the bench line down
            two_jobs = dict(two_jobs or {}, error=repr(exc))

    # ---- the live path as a C++ host drives it: one integratePointCloud call per frame through
    # the C++ mirror (coxgraph_b200/host/coxgraph_b200.hpp) with pageable std::vector inputs —
    # what voxblox_ros TsdfServer / INTEGRATION.md's adapter pass (N = 1, rank 0 only)
    per_frame_host = None
    if rank == 0 and world == 1 and not args.profile_mode:
        try:
            import struct
            import tempfile
            binary = os.path.join(ROOT, "build", "host_api_check")
            if not os.path.exists(binary):
                subprocess.check_call(["make", "-C", ROOT, "-s", "build/host_api_check"])
            e = pool[0]
            with tempfile.NamedTemporaryFile(suffix=".bin", delete=False) as f:
                f.write(struct.pack("<Iff", FRAMES_PER_SUBMAP, VOXEL_SIZE,
                                    CFG["default_truncation_distance"]))
                f.write(np.asarray(e["T_M_S"], np.float32).tobytes())
                for k in range(FRAMES_PER_SUBMAP):
                    a, b = int(e["offs"][k]), int(e["offs"][k + 1])
                    f.write(np.asarray(e["poses"][k], np.float32).tobytes())
                    f.write(struct.pack("<I", b - a))
                    f.write(np.ascontiguousarray(e["h_pts"][a:b]).tobytes())
                    f.write(np.ascontiguousarray(e["h_cols"][a:b]).tobytes())
                path = f.name
            r = subprocess.run([binary, "time", path, "3"], capture_output=True, text=True,
                               timeout=120)
            os.unlink(path)
            per_frame_host = json.loads(r.stdout.strip().splitlines()[-1])
            per_frame_host["what"] = ("cg_integrate_pointcloud through the C++ mirror, pageable "
                                      "std::vector inputs (H2D inside the call)")
        except Exception as exc:  # noqa: BLE001 - an extra figure must not take the bench line down
            per_frame_host = {"error": repr(exc)}
        # the plain call with PAGEABLE host arrays for a whole step (what an adapter's std::vector
        # clouds are): cg_integrate_batch copies them through its worker threads and pinned bounce
        # buffer (csrc/host_stage.cu); the merge follows as in a step
        try:
            e = pool[0]
            pg_pts = np.array(e["h_pts"], copy=True)   # ordinary (pageable) numpy memory
            pg_cols = np.array(e["h_cols"], copy=True)
            t_pg = []
            for it in range(4):
                submap.clear()
                torch.cuda.synchronize()
                t0 = time.perf_counter()
                integ.integrateBatch(e["poses"], pg_pts, pg_cols, e["offs"])
                mergeLayerAintoLayerB(submap, e["T_M_S"], glob)
                torch.cuda.synchronize()
                t_pg.append((time.perf_counter() - t0) * 1e3)
            if isinstance(per_frame_host, dict):
                per_frame_host["pageable_step"] = {
                    "ms_per_step": min(t_pg[1:]), "points_per_s": e["n"] / (min(t_pg[1:]) * 1e-3),
                    "what": "one C2 step through cg_integrate_batch with pageable host arrays "
                            "(123 MB staged by the library's worker threads), then the merge"}
        except Exception as exc:  # noqa: BLE001
            if isinstance(per_frame_host, dict):
                per_frame_host["pageable_step"] = {"error": repr(exc)}

    # ---- CPU baseline beside it (rank 0, N = 1 only): the oracle, all host threads, bounded
    cpu = None
    if rank == 0 and world == 1 and not args.no_cpu_baseline and not args.profile_mode:
        from oracle import oracle_py as orc
        threads = os.cpu_count() or 1
        ocfg = orc.default_config(**CFG)
        e = pool[args.warmup % pool_n]
        ol = orc.Layer(VOXEL_SIZE)
        t0 = time.perf_counter()
        done = 0
        for f in range(FRAMES_PER_SUBMAP):
            a, b = int(e["offs"][f]), int(e["offs"][f + 1])
            ol.integrate(ocfg, e["poses"][f], e["h_pts"][a:b], e["h_cols"][a:b], threads=threads)
            done += b - a
            if time.perf_counter() - t0 > args.cpu_seconds:
                break
        t_cpu = time.perf_counter() - t0
        og = orc.Layer(VOXEL_SIZE)
        t1 = time.perf_counter()
        og.merge_from(ol, e["T_M_S"])          # single thread, as the reference merges
        t_m = time.perf_counter() - t1
        # the reference's own setting is integrator_threads: 8 (tsdf_server_euroc.yaml:10)
        ol8 = orc.Layer(VOXEL_SIZE)
        t8 = time.perf_counter()
        done8 = 0
        for f in range(min(5, FRAMES_PER_SUBMAP)):
            a, b = int(e["offs"][f]), int(e["offs"][f + 1])
            ol8.integrate(ocfg, e["poses"][f], e["h_pts"][a:b], e["h_cols"][a:b], threads=8)
            done8 += b - a
        t8 = time.perf_counter() - t8
        cpu = {"value": done / t_cpu, "unit": "points/s", "cores": threads, "kind": "port",
               "value_8_threads": done8 / t8,
               "sample": f"first {done // 307200} frames ({done} points) of one submap, "
                         f"{threads}-thread voxblox-style integrator (oracle port)",
               "merge_voxels_per_s": 4096 * ol.num_blocks / t_m, "merge_threads": 1}

    if rank == 0:
        dv, ee, ee_name = results["device"], results["e2e"], "staged copy + prepared first half"
        if "e2e_plain" in results and results["e2e_plain"]["total_ms"] < ee["total_ms"]:
            ee, ee_name = results["e2e_plain"], "staged copy, plain calls"
        dv["profile"] = results["profiled"]["profile"]
        used_dev = [pool[(args.warmup + k) % pool_n] for k in range(args.steps)]
        peak, peak_src = measured_peak_gbs()
        prof = dv["profile"]
        n_used = float(len(used_dev))
        per_step = dict(n_pts=sum(e["n"] for e in used_dev) / n_used,
                        rays=sum(e["rays"] for e in used_dev) / n_used,
                        pairs=sum(e["pairs"] for e in used_dev) / n_used,
                        general=sum(e["general"] for e in used_dev) / n_used,
                        blocks=sum(e["blocks_in"] for e in used_dev) / n_used,
                        b_in=sum(e["blocks_in"] for e in used_dev) / n_used,
                        b_out=sum(e["bytes_merge"] / BLOCK_BYTES - e["blocks_in"] for e in used_dev)
                        / n_used / 2)
        # headline: the pipelined loop (the first half of step k+1 is queued before step k is
        # completed: cg_prepare_batch_device / cg_integrate_prepared); the plain-call loop beside it
        hv = results[headline_leg]
        roof = roofline_record(prof, args.steps, hv["total_ms"] / args.steps,
                               (dv["bytes_int"] + dv["bytes_merge"]) / args.steps, per_step)
        line = {
            "metric": "tsdf_points_integrated_per_s",
            "value": hv["points"] / (hv["total_ms"] * 1e-3),
            "unit": "points/s", "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
            "ms_per_step": hv["total_ms"] / args.steps, "higher_is_better": True,
            "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "config": dict(CONFIG),
            "run": {"parallelism": f"submaps sharded over {world} GPU(s), no data-path collective",
                    "l2": "each step streams >300 MB of fresh points and update lists "
                          "(> 126 MB L2); distinct submap per step",
                    "pool_submaps": pool_n,
                    "pipelining": "value / e2e: the layer-independent first half of step k+1 "
                                  "(points -> rays) runs on a second stream beside the second "
                                  "half and the merge of step k; plain_calls / e2e_plain_calls: "
                                  "one cg_integrate_batch call after the other"
                    if "pipelined" in results else "none"},
            "plain_calls": {"value": dv["points"] / (dv["total_ms"] * 1e-3), "unit": "points/s",
                            "ms_per_step": dv["total_ms"] / args.steps},
            "project_submaps": project,
            "two_jobs_in_flight": two_jobs,
            # the live path: one integratePointCloud call per 640x480 frame (device-resident
            # input), as voxblox_ros TsdfServer makes them; the batch call above is the recover loop
            # (median over the pool's submaps: the first per-frame calls of a context grow its
            # scratch buffers, and a cudaMalloc / cudaFree is a stall of milliseconds)
            "per_frame_call": {"ms": float(np.median([e["per_frame_ms"] for e in pool])),
                               "points_per_s": 307200.0 /
                               max(1e-9, float(np.median([e["per_frame_ms"] for e in pool])) * 1e-3),
                               "what": "cg_integrate_pointcloud_device, input resident in HBM",
                               "queued_ms": float(np.median([e["per_frame_queued_ms"] for e in pool])),
                               "queued_what": "the same frames with the next one queued: "
                                              "cg_prepare_batch_device(frame f+1) before "
                                              "cg_integrate_prepared(frame f); wall clock",
                               "host_pageable": per_frame_host},
            "integrate": {"value": dv["points"] / (dv["int_ms"] * 1e-3), "unit": "points/s",
                          "ms_per_step": dv["int_ms"] / args.steps,
                          "hbm_frac_phase": dv["bytes_int"] / (dv["int_ms"] * 1e-3) / 1e9 / peak},
            "merge": {"value": dv["voxels"] / (dv["merge_ms"] * 1e-3), "unit": "voxels/s",
                      "ms_per_step": dv["merge_ms"] / args.steps,
                      "hbm_frac_phase": dv["bytes_merge"] / (dv["merge_ms"] * 1e-3) / 1e9 / peak},
            # host buffers: the faster of the two loops (both timed above); the copy of step k+1 is
            # staged while step k is fused in either, `pipelined` also starts its first half
            "e2e": {"value": ee["points"] / (ee["total_ms"] * 1e-3), "unit": "points/s",
                    "ms_per_step": ee["total_ms"] / args.steps,
                    "h2d_bytes_per_step": ee["h2d"], "d2h_bytes_per_step": ee["d2h"],
                    "loop": ee_name},
            "e2e_loops_ms_per_step": {k: results[k]["total_ms"] / args.steps
                                      for k in ("e2e", "e2e_plain") if k in results},
            "gpu_launches": hv["launches"],
            "roofline": roof,
            "per_rank_ms_per_step": hv.get("per_rank_ms"),
            "stages_ms_per_step": {k: v[0] / args.steps for k, v in prof.items()},
            "per_step": {"rays": sum(e["rays"] for e in used_dev) / args.steps,
                         "voxel_updates": sum(e["pairs"] for e in used_dev) / args.steps,
                         "ordered_updates": sum(e["general"] for e in used_dev) / args.steps,
                         "blocks_in": sum(e["blocks_in"] for e in used_dev) / args.steps},
            "clocks": dv["clocks"], "clocks_e2e": ee["clocks"],
            "cpu_baseline": cpu,
        }
        print(json.dumps(line), flush=True)
    submap.close()
    glob.close()
    ctx.close()
    if world > 1:
        dist.destroy_process_group()


def time_esdf(layer, max_over_ranks=lambda x: x, reps=3):
    """updateEsdfBatch on the device-resident merged map (map_server.h:141-145) + the traversable
    cloud (map_server.cpp:112-113); wall time around the calls (they synchronise).  min_distance
    0.1 m (coxgraph_client.yaml:69): with the 0.16 m truncation band of the bench scenes upstream's
    default 0.2 m would fix every observed voxel."""
    from coxgraph_b200 import esdfConfig
    cfg = esdfConfig(min_distance_m=0.1)
    ms, free_ms, st, n_free = [], [], None, 0
    for _ in range(reps):
        t0 = time.perf_counter()
        st = layer.updateEsdfBatch(cfg, fetch=False)
        ms.append((time.perf_counter() - t0) * 1e3)
        t0 = time.perf_counter()
        n_free = len(layer.esdfFreePoints(0.3))
        free_ms.append((time.perf_counter() - t0) * 1e3)
    best = max_over_ranks(min(ms[1:]))
    return {"ms": best, "blocks": int(st.blocks), "observed_voxels": int(st.observed_voxels),
            "fixed_voxels": int(st.fixed_voxels), "sweeps": int(st.sweeps),
            "block_passes": int(st.block_passes),
            "voxels_per_s": st.blocks * 4096.0 / (best * 1e-3),
            "free_points": {"ms_with_d2h": max_over_ranks(min(free_ms[1:])), "points": int(n_free),
                            "radius_m": 0.3},
            "what": "cg_layer_esdf_batch: fixed point of EsdfIntegrator's wavefront, min_distance 0.1 m, "
                    "max_distance 2 m; result stays on the device"}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--pool", type=int, default=6, help="distinct submaps kept resident")
    ap.add_argument("--ref-frames", type=int, default=FRAMES_PER_SUBMAP,
                    help="frames per step the reference arm fuses (25 = the whole step; fewer = a "
                         "bounded sample)")
    ap.add_argument("--cpu-seconds", type=float, default=12.0)
    ap.add_argument("--project-submaps", type=int, default=40,
                    help="submaps of the separate getProjectedMap timing (0 = skip)")
    ap.add_argument("--parity-submaps", type=int, default=3,
                    help="submaps per rank of the in-bench parity check of the sharded merge (N > 1)")
    ap.add_argument("--config", default="C2", choices=["C1", "C2", "C3", "C4", "C5"],
                    help="BASELINE.json config (default C2 = the headline; see configs.py docstrings)")
    ap.add_argument("--c4-blocks", type=int, default=2_000_000,
                    help="C4: integrate along the trajectory until this many blocks are allocated")
    ap.add_argument("--c3-submaps", type=int, default=64, help="C3 / C5: submaps per robot")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--profile-mode", action="store_true",
                    help="skip the accounting pass and the CPU baseline (for runs under ncu)")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="after the timed steps of the leg `value` reports, write what its last "
                         "step left (the fused submap, the global layer, the call statistics) as "
                         "DIR/<name>.npy; rank 0, config C2")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and (args.impl != "ours" or args.config != "C2"):
        ap.error("--dump-outputs covers the CUDA arm of config C2")
    args.warmup = max(args.warmup, 0)
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    if args.impl == "reference":
        run_reference(args, rank, world)
        return
    if args.warmup < 3:
        args.warmup = 3
    if args.config == "C2":
        run_ours(args, rank, world, local_rank)
    else:
        import bench_configs
        bench_configs.run(args, rank, world, local_rank)


if __name__ == "__main__":
    main()
