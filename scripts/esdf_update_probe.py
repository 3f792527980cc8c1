"""Timing probe of the incremental ESDF (cg_layer_esdf_update) against the batch, at the C2 and C5
shapes, with a bit-identity check in the same run.

Each case starts from the map with the batch ESDF retained, applies one mutation, times the
update (CUDA events), then times the batch on the same layer and compares the two results.  The
map is put back before the next repeat.  The compare pass (k_esdf_compare) is timed in a separate
torch.profiler run.  Prints the card name and power limit first, then one JSON line per case.
    python scripts/esdf_update_probe.py [--repeats 3] [--c5-submaps 64]"""
import argparse
import json
import os
import subprocess
import sys

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
from coxgraph_b200 import (Context, Layer, TsdfIntegrator, TsdfIntegratorConfig, esdfConfig,  # noqa: E402
                           getProjectedMap, mergeLayerAintoLayerB, reprojectSubmaps, synth)

DEV = torch.device("cuda", 0)
CFG = TsdfIntegratorConfig(default_truncation_distance=0.16, use_const_weight=1, method=1)
ESDF = esdfConfig(min_distance_m=0.1)


def _card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"],
                       capture_output=True, text=True)
    return q.stdout.strip()


def _fuse(ctx, frames, max_blocks):
    L = Layer(ctx, 0.05, max_blocks=max_blocks)
    P = np.stack([T for (T, _, _) in frames]).astype(np.float32)
    pts = torch.cat([p for (_, p, _) in frames]).contiguous()
    cols = torch.cat([c for (_, _, c) in frames]).contiguous()
    offs = np.cumsum([0] + [len(p) for (_, p, _) in frames]).astype(np.uint64)
    TsdfIntegrator(CFG, L).integrateBatch(P, pts, cols, offs)
    return L


def _timed(fn):
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    torch.cuda.synchronize()
    a.record()
    out = fn()
    b.record()
    torch.cuda.synchronize()
    return a.elapsed_time(b), out


def _compare_ms(glob, mutate, restore):
    """k_esdf_compare's device time in one update, from torch.profiler."""
    from torch.profiler import ProfilerActivity, profile
    restore()
    glob.updateEsdfBatch(ESDF, fetch=False)
    mutate()
    torch.cuda.synchronize()
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        glob.updateEsdf(ESDF, fetch=False)
        torch.cuda.synchronize()
    us = sum(e.device_time_total for e in prof.key_averages() if "k_esdf_compare" in e.key)
    return us / 1e3


def run_case(name, glob, mutate, restore, repeats):
    upd, bat, rows = [], [], None
    for _ in range(repeats + 1):  # the first round warms up
        restore()
        glob.updateEsdfBatch(ESDF, fetch=False)
        mutate()
        t_u, (st, ust) = _timed(lambda: glob.updateEsdf(ESDF, fetch=False))
        got = glob.updateEsdf(ESDF)  # nothing changed since: returns the retained result
        t_b, _ = _timed(lambda: glob.updateEsdfBatch(ESDF, fetch=False))
        want = glob.updateEsdfBatch(ESDF)
        same = (np.array_equal(got["idx"], want["idx"]) and np.array_equal(got["packed"], want["packed"])
                and np.array_equal(got["distance"].view(np.uint32), want["distance"].view(np.uint32)))
        if not same:
            raise SystemExit(f"{name}: update and batch differ")
        upd.append(t_u)
        bat.append(t_b)
        rows = (st, ust)
    st, ust = rows
    out = {"case": name, "blocks": int(st.blocks), "blocks_changed": int(ust.blocks_changed),
           "blocks_removed": int(ust.blocks_removed), "blocks_region": int(ust.blocks_region),
           "region_fraction": round(ust.blocks_region / max(1, st.blocks), 4),
           "full_rebuild": int(ust.full_rebuild), "sweeps": int(st.sweeps),
           "update_ms": round(float(np.median(upd[1:])), 3), "batch_ms": round(float(np.median(bat[1:])), 3),
           "update_ms_all": [round(x, 3) for x in upd[1:]], "batch_ms_all": [round(x, 3) for x in bat[1:]],
           "compare_ms": round(_compare_ms(glob, mutate, restore), 3), "bit_identical": True}
    print(json.dumps(out), flush=True)


def c2(ctx, repeats):
    subs, poses = [], []
    for k in range(41):
        robot, sm = k % 2, k // 2
        subs.append(_fuse(ctx, synth.submap_frames(robot, sm % 20, 25, device=DEV), 1024))
        poses.append(synth.robot_map_offset(robot))
    poses = np.stack(poses)
    poses[40] = synth.perturb_pose(poses[40], np.random.default_rng(3), 0.5, 10.0)
    glob = Layer(ctx, 0.05, max_blocks=65536)

    def restore():
        glob.clear()
        getProjectedMap(subs[:40], poses[:40], glob)

    run_case("C2: 40-submap map + one merged submap", glob,
             lambda: mergeLayerAintoLayerB(subs[40], poses[40], glob), restore, repeats)


def c5(ctx, repeats, per_robot):
    subs = []
    for r in range(8):
        for sm in range(per_robot + (1 if r == 0 else 0)):
            fr = synth.corridor_frames(sm * 10, 10, robot=r, advance=0.2, start_x=128.0 * r, device=DEV)
            subs.append(_fuse(ctx, fr, 768))
    extra = subs.pop(per_robot)  # robot 0's next submap along the corridor
    rng = np.random.default_rng(5)
    base = np.stack([synth.perturb_pose(synth.robot_map_offset(0), rng, sigma_t=0.05, sigma_yaw_deg=1.0)
                     for _ in subs])
    glob = Layer(ctx, 0.05, max_blocks=262144)

    def restore():
        glob.clear()
        getProjectedMap(subs, base, glob)

    run_case(f"C5: {len(subs)}-submap map + one more submap", glob,
             lambda: mergeLayerAintoLayerB(extra, synth.robot_map_offset(0), glob), restore, repeats)
    for frac_name, count in (("one moved submap", 1), ("10 % moved", max(1, len(subs) // 10))):
        moved = rng.choice(len(subs), count, replace=False)
        new = base.copy()
        for k in moved:
            new[k] = synth.perturb_pose(base[k], rng, sigma_t=0.05, sigma_yaw_deg=1.0)
        run_case(f"C5: {len(subs)}-submap map, {frac_name} re-projected", glob,
                 lambda: reprojectSubmaps(subs, base, new, glob), restore, repeats)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--repeats", type=int, default=3)
    ap.add_argument("--c5-submaps", type=int, default=64, help="submaps per robot (8 robots)")
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("esdf_update_probe needs a CUDA device")
    print(json.dumps({"card": _card()}), flush=True)
    ctx = Context(0)
    c2(ctx, args.repeats)
    c5(ctx, args.repeats, args.c5_submaps)


if __name__ == "__main__":
    main()
