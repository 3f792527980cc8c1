"""Depth-image input against the cloud input at the C2 shape (25 frames of 640x480 per step, 5 cm
voxels, merged integrator, fused into a cleared submap then merged into the global layer), in one
process, the two alternating.  The depth jobs read synthetic 16UC1 depth + rgb8 images
(synth.render_depth_frame); the cloud jobs read the clouds depth_image_proc + TsdfServer build
from the same images (tests/depth_reference.py).  Prints one JSON line.

    python scripts/depth_e2e.py [--steps 20] [--warmup 3] [--rounds 3] [--pool 4]
"""
import argparse
import json
import os
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

FRAMES = 25
VOXEL_SIZE = 0.05
CFG = dict(default_truncation_distance=0.16, max_ray_length_m=5.0, min_ray_length_m=0.1,
           use_const_weight=1, method=1)   # bench.py's C2 config
BLOCK_BYTES = 4096 * 12


def card():
    try:
        out = subprocess.check_output(["nvidia-smi", "--query-gpu=name,power.limit",
                                       "--format=csv,noheader", "-i", "0"], text=True)
        name, power = [s.strip() for s in out.strip().split(",")]
        return name, power
    except (OSError, subprocess.CalledProcessError, ValueError):
        import torch
        return torch.cuda.get_device_name(0), "unknown"


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--rounds", type=int, default=3, help="alternations of depth and cloud legs")
    ap.add_argument("--pool", type=int, default=4, help="distinct submaps cycled through")
    args = ap.parse_args()
    import torch
    if not torch.cuda.is_available():
        raise SystemExit("depth_e2e.py needs a CUDA device")
    from coxgraph_b200 import (Context, Layer, TsdfIntegrator, TsdfIntegratorConfig, VOXEL_DTYPE,
                               mergeLayerAintoLayerB, synth)
    from tests import depth_reference as ref
    dev = torch.device("cuda", 0)
    pin = lambda t: torch.empty(t.shape, dtype=t.dtype, pin_memory=True).copy_(t)  # noqa: E731

    pool = []
    for s in range(args.pool):
        robot, sm = s % 2, s // 2
        poses = synth.trajectory(FRAMES, robot=robot, submap=sm, frames_per_submap=FRAMES)
        imgs = [synth.render_depth_frame(poses[f]) for f in range(FRAMES)]
        cam = imgs[0][2]
        depth = np.stack([d for d, _, _ in imgs])
        rgb = np.stack([c for _, c, _ in imgs])
        pts, cols, offs = ref.depth_batch_cloud(depth, rgb, cam)
        t_depth = torch.from_numpy(depth.view(np.int16))
        t_rgb, t_pts, t_cols = (torch.from_numpy(a) for a in (rgb, pts, cols))
        pool.append(dict(poses=poses.astype(np.float32), cam=cam, offs=offs, depth=depth, rgb=rgb,
                         d_depth=t_depth.to(dev), d_rgb=t_rgb.to(dev), d_pts=t_pts.to(dev),
                         d_cols=t_cols.to(dev), h_depth=pin(t_depth).numpy().view(np.uint16),
                         h_rgb=pin(t_rgb).numpy(), h_pts=pin(t_pts).numpy(),
                         h_cols=pin(t_cols).numpy(), pts=pts, cols=cols,
                         T_M_S=synth.robot_map_offset(robot)))
    torch.cuda.synchronize()
    ctx = Context(0)
    cfg = TsdfIntegratorConfig(**CFG)
    submap = Layer(ctx, VOXEL_SIZE, max_blocks=4096)
    glob = Layer(ctx, VOXEL_SIZE, max_blocks=32768)
    integ = TsdfIntegrator(cfg, submap)
    out_idx = torch.empty((4096, 3), dtype=torch.int32, pin_memory=True).numpy()
    out_vox = torch.empty((4096, 4096 * 12), dtype=torch.uint8, pin_memory=True).numpy() \
        .view(VOXEL_DTYPE).reshape(4096, 4096)
    out_flags = torch.empty((4096,), dtype=torch.uint8, pin_memory=True).numpy()

    # one step of each kind of job: (prepare on device, prepare staged, stage, integrate device,
    # integrate staged)
    def ops(kind):
        if kind == "depth":
            return dict(
                prep=lambda sl, e: integ.prepareDepth(sl, e["poses"], e["d_depth"], e["d_rgb"], e["cam"]),
                stage=lambda sl, e: integ.stageDepth(sl, e["h_depth"], e["h_rgb"], e["cam"]),
                prep_staged=lambda sl, e: integ.prepareDepthStaged(sl, sl, e["poses"], e["cam"]),
                plain=lambda e: integ.integrateDepthBatch(e["poses"], e["d_depth"], e["d_rgb"], e["cam"]),
                staged=lambda sl, e: integ.integrateDepthStaged(sl, e["poses"], e["cam"]))
        return dict(
            prep=lambda sl, e: integ.prepareBatch(sl, e["poses"], e["d_pts"], e["d_cols"], e["offs"]),
            stage=lambda sl, e: integ.stageBatch(sl, e["h_pts"], e["h_cols"]),
            prep_staged=lambda sl, e: integ.prepareStaged(sl, sl, e["poses"], e["offs"]),
            plain=lambda e: integ.integrateBatch(e["poses"], e["d_pts"], e["d_cols"], e["offs"]),
            staged=lambda sl, e: integ.integrateStaged(sl, e["poses"], e["offs"]))

    def loop(kind, leg, entries):
        o = ops(kind)
        if leg == "device_pipelined":
            o["prep"](0, entries[0])
        if leg.startswith("e2e"):
            o["stage"](0, entries[0])
            if leg == "e2e_pipelined":
                o["prep_staged"](0, entries[0])
        for k, e in enumerate(entries):
            nxt = entries[k + 1] if k + 1 < len(entries) else None
            sl = k % 2
            if nxt is not None and leg == "device_pipelined":
                o["prep"](1 - sl, nxt)
            if nxt is not None and leg.startswith("e2e"):
                o["stage"](1 - sl, nxt)
                if leg == "e2e_pipelined":
                    o["prep_staged"](1 - sl, nxt)
            submap.clear()
            if leg in ("device_pipelined", "e2e_pipelined"):
                integ.integratePrepared(sl)
            elif leg == "device_plain":
                o["plain"](e)
            else:
                o["staged"](sl, e)
            mergeLayerAintoLayerB(submap, e["T_M_S"], glob)
            if leg.startswith("e2e"):
                submap.download(out=(out_idx, out_vox, out_flags))

    def timed(kind, leg):
        warm = [pool[s % len(pool)] for s in range(args.warmup)]
        steps = [pool[(args.warmup + s) % len(pool)] for s in range(args.steps)]
        loop(kind, leg, warm)
        ctx.synchronize()
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        loop(kind, leg, steps)
        ctx.synchronize()
        return (time.perf_counter() - t0) * 1e3 / args.steps

    def per_frame(kind):
        """The drop-in per-frame call with pageable numpy inputs."""
        e = pool[0]
        submap.clear()
        ctx.synchronize()
        t0 = time.perf_counter()
        for f in range(FRAMES):
            if kind == "depth":
                integ.integrateDepthImage(e["poses"][f], e["depth"][f], e["rgb"][f], e["cam"])
            else:
                a, b = int(e["offs"][f]), int(e["offs"][f + 1])
                integ.integratePointCloud(e["poses"][f], e["pts"][a:b], e["cols"][a:b])
        ctx.synchronize()
        return (time.perf_counter() - t0) * 1e3 / FRAMES

    legs = ("device_pipelined", "device_plain", "e2e_pipelined", "e2e_plain")
    runs = {k: {leg: [] for leg in legs + ("per_frame_call",)} for k in ("depth", "cloud")}
    for _ in range(args.rounds):
        for kind in ("depth", "cloud"):
            for leg in legs:
                runs[kind][leg].append(timed(kind, leg))
            per_frame(kind)  # warm
            runs[kind]["per_frame_call"].append(per_frame(kind))

    # the depth_points stage: its own profiled pass over plain device steps
    ctx.set_profiling(True)
    ctx.reset_profile()
    loop("depth", "device_plain", [pool[s % len(pool)] for s in range(args.steps)])
    prof = ctx.profile()
    ctx.set_profiling(False)
    stage_ms = {k: v[0] / args.steps for k, v in prof.items() if v[0] > 0}

    # parity: the last pool entry through both inputs, fused into fresh layers
    e = pool[-1]
    layers = []
    for kind in ("depth", "cloud"):
        L = Layer(ctx, VOXEL_SIZE, max_blocks=4096)
        it = TsdfIntegrator(cfg, L)
        if kind == "depth":
            it.integrateDepthBatch(e["poses"], e["d_depth"], e["d_rgb"], e["cam"])
        else:
            it.integrateBatch(e["poses"], e["d_pts"], e["d_cols"], e["offs"])
        idx, vox, fl = L.download()
        layers.append(idx.tobytes() + vox.tobytes() + fl.tobytes())
        L.close()

    name, power = card()
    px = FRAMES * e["cam"]["width"] * e["cam"]["height"]
    summary = lambda xs: dict(median=float(np.median(xs)), min=float(min(xs)), max=float(max(xs)))  # noqa: E731
    print(json.dumps(dict(
        workload="C2 shape: 25 x 640x480 frames per step, merged, 5 cm voxels, merge included",
        card=name, power_limit=power, steps=args.steps, rounds=args.rounds,
        ms_per_step={k: {leg: summary(v) for leg, v in runs[k].items()} for k in runs},
        h2d_bytes_per_step=dict(depth=px * (2 + 3), cloud=int(np.mean([p["offs"][-1] for p in pool])) * 16),
        depth_points_ms_per_step=stage_ms.get("depth_points", 0.0),
        stages_ms_per_step_depth_plain=stage_ms,
        parity_last_step=layers[0] == layers[1])))
    submap.close()
    glob.close()
    ctx.close()


if __name__ == "__main__":
    main()
