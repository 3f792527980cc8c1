"""Deterministic synthetic depth-camera streams (SURVEY.md §8d).

A closed analytic scene (room 12 x 8 x 3 m, spheres, boxes) is ray-cast exactly from a pinhole
camera in the optical frame (z forward, x right, y down), producing what the reference's
front-end hands to `integratePointCloud`: `points_C` (float32 N x 3), `colors` (uint8 N x 4) and
`T_G_C` (qw qx qy qz tx ty tz).  Every pixel hits something, so N = W * H exactly.  Written in
torch ops so the same code runs on the CPU (tests, here) and on the GPU (bench input generation,
outside every timed region).  This is workload plumbing, not part of the hot path.
"""
import math

import numpy as np
import torch

SEED = 0xC0C62A9F

# RealSense intrinsics, /root/reference/coxgraph/config/ncamera_rs.yaml:5-11
CAM_640x480 = dict(width=640, height=480, fx=611.16, fy=609.64, cx=323.45, cy=244.94)
CAM_1280x720 = dict(width=1280, height=720, fx=920.0, fy=920.0, cx=640.0, cy=360.0)

ROOM = (12.0, 8.0, 3.0)
# Objects stand along the two long walls and on the centre line, leaving two clear corridors
# (y = 2.8 and y = 5.2) for the robots: every camera keeps >= 0.9 m from every surface.
# (cx, cy, cz, r)
SPHERES = [(3.0, 1.0, 0.8, 0.8), (6.5, 0.9, 0.5, 0.5), (9.0, 1.1, 1.2, 0.6),
           (4.5, 7.0, 0.6, 0.6), (10.0, 6.9, 0.7, 0.7), (7.5, 7.2, 1.8, 0.4)]
# (xmin, ymin, zmin, xmax, ymax, zmax)
BOXES = [(1.0, 6.2, 0.0, 2.0, 7.6, 1.5), (5.0, 3.6, 0.0, 6.0, 4.4, 0.9),
         (8.0, 6.3, 0.0, 8.6, 7.7, 2.2), (10.5, 0.4, 0.0, 11.5, 1.4, 1.0)]


def quat_from_matrix(R):
    """Rotation matrix (3x3, float64) -> unit quaternion (w, x, y, z), w >= 0."""
    R = np.asarray(R, dtype=np.float64)
    t = np.trace(R)
    if t > 0:
        s = math.sqrt(t + 1.0) * 2
        q = [0.25 * s, (R[2, 1] - R[1, 2]) / s, (R[0, 2] - R[2, 0]) / s, (R[1, 0] - R[0, 1]) / s]
    elif R[0, 0] > R[1, 1] and R[0, 0] > R[2, 2]:
        s = math.sqrt(1.0 + R[0, 0] - R[1, 1] - R[2, 2]) * 2
        q = [(R[2, 1] - R[1, 2]) / s, 0.25 * s, (R[0, 1] + R[1, 0]) / s, (R[0, 2] + R[2, 0]) / s]
    elif R[1, 1] > R[2, 2]:
        s = math.sqrt(1.0 + R[1, 1] - R[0, 0] - R[2, 2]) * 2
        q = [(R[0, 2] - R[2, 0]) / s, (R[0, 1] + R[1, 0]) / s, 0.25 * s, (R[1, 2] + R[2, 1]) / s]
    else:
        s = math.sqrt(1.0 + R[2, 2] - R[0, 0] - R[1, 1]) * 2
        q = [(R[1, 0] - R[0, 1]) / s, (R[0, 2] + R[2, 0]) / s, (R[1, 2] + R[2, 1]) / s, 0.25 * s]
    q = np.array(q)
    q /= np.linalg.norm(q)
    if q[0] < 0:
        q = -q
    return q


def matrix_from_quat(q):
    w, x, y, z = [float(v) for v in q]
    return np.array([
        [1 - 2 * (y * y + z * z), 2 * (x * y - z * w), 2 * (x * z + y * w)],
        [2 * (x * y + z * w), 1 - 2 * (x * x + z * z), 2 * (y * z - x * w)],
        [2 * (x * z - y * w), 2 * (y * z + x * w), 1 - 2 * (x * x + y * y)]])


def camera_pose(position, yaw, pitch=0.0, roll=0.0):
    """World pose T_G_C (7 floats) of an optical-frame camera looking along world yaw."""
    base = np.array([[0.0, 0.0, 1.0], [-1.0, 0.0, 0.0], [0.0, -1.0, 0.0]])  # cam xyz -> world
    cy, sy = math.cos(yaw), math.sin(yaw)
    Rz = np.array([[cy, -sy, 0], [sy, cy, 0], [0, 0, 1.0]])
    cp, sp = math.cos(pitch), math.sin(pitch)
    Rx = np.array([[1.0, 0, 0], [0, cp, -sp], [0, sp, cp]])  # about camera x
    cr, sr = math.cos(roll), math.sin(roll)
    Rr = np.array([[cr, -sr, 0], [sr, cr, 0], [0, 0, 1.0]])  # about camera z
    R = Rz @ base @ Rx @ Rr
    q = quat_from_matrix(R)
    return np.concatenate([q, np.asarray(position, dtype=np.float64)]).astype(np.float32)


def compose(Ta, Tb):
    """T = Ta * Tb for (qw qx qy qz t) transforms (float64 maths, float32 result)."""
    Ra, Rb = matrix_from_quat(Ta[:4]), matrix_from_quat(Tb[:4])
    R = Ra @ Rb
    t = Ra @ np.asarray(Tb[4:], dtype=np.float64) + np.asarray(Ta[4:], dtype=np.float64)
    return np.concatenate([quat_from_matrix(R), t]).astype(np.float32)


def invert(T):
    R = matrix_from_quat(T[:4]).T
    t = -R @ np.asarray(T[4:], dtype=np.float64)
    return np.concatenate([quat_from_matrix(R), t]).astype(np.float32)


def trajectory(num_frames, robot=0, submap=0, frames_per_submap=None):
    """Smooth drive along one of the two corridors: ~1.5 cm per frame, the camera sweeping
    left-right across the wall and the objects in front of it (never axis-aligned)."""
    if frames_per_submap is None:
        frames_per_submap = num_frames
    poses = []
    lane = robot // 2
    for f in range(num_frames):
        k = submap * frames_per_submap + f
        u = (k % 500) / 500.0
        s = 0.03 * k
        if robot % 2 == 0:   # corridor A, driving +x, looking towards the y = 0 wall
            pos = (2.0 + 7.5 * u + 0.13 * lane, 2.8 + 0.15 * math.sin(0.35 * s + lane),
                   1.35 + 0.1 * math.sin(0.8 * s) - 0.07 * lane)
            yaw = -math.pi / 2 + 0.62 + 0.6 * math.sin(0.21 * s + 0.9 * lane)
        else:                # corridor B, driving -x, looking towards the y = 8 wall
            pos = (10.0 - 7.5 * u - 0.13 * lane, 5.2 + 0.15 * math.cos(0.3 * s + lane),
                   1.25 + 0.12 * math.cos(0.7 * s) + 0.07 * lane)
            yaw = math.pi / 2 - 0.58 + 0.6 * math.sin(0.17 * s + 0.7 * lane + 0.4)
        pitch = 0.07 * math.sin(0.5 * s + robot)
        roll = 0.03 * math.cos(0.4 * s)
        poses.append(camera_pose(pos, yaw, pitch, roll))
    return np.stack(poses)


def _hash_color(p):
    """Procedural colour = integer hash of floor(4 p); alpha 255.  p: [N,3] float32 tensor."""
    c = torch.floor(p * 4.0).to(torch.int64)
    h = (c[:, 0] * 73856093) ^ (c[:, 1] * 19349663) ^ (c[:, 2] * 83492791)
    h = h ^ (h >> 13)
    r = (h & 255).to(torch.uint8)
    g = ((h >> 8) & 255).to(torch.uint8)
    b = ((h >> 16) & 255).to(torch.uint8)
    a = torch.full_like(r, 255)
    return torch.stack([r, g, b, a], dim=1)


PERIOD = ROOM[0]      # the corridor scene repeats the room's objects every 12 m along x
CORRIDOR_CAP = 40.0   # virtual end walls this far ahead of / behind the camera (every pixel hits)


def render_frame(T_G_C, cam=CAM_640x480, device="cpu", near_box=False, stride=1, scene="room"):
    """Exact ray-cast of the scene.  Returns (points_C float32 [N,3], colors uint8 [N,4]).

    scene="room": the closed 12 x 8 x 3 m room.  scene="corridor": the same cross-section without
    end walls, the objects repeated every 12 m along x — an unbounded environment for the long
    trajectories of configs C3 / C4 / C5 (SURVEY.md §8d); rays along the axis end on a virtual wall
    40 m from the camera (far beyond max_ray: they become clearing rays)."""
    dev = torch.device(device)
    W, H = cam["width"], cam["height"]
    us = torch.arange(0, W, stride, device=dev, dtype=torch.float64)
    vs = torch.arange(0, H, stride, device=dev, dtype=torch.float64)
    v, u = torch.meshgrid(vs, us, indexing="ij")
    d_c = torch.stack([(u - cam["cx"]) / cam["fx"], (v - cam["cy"]) / cam["fy"],
                       torch.ones_like(u)], dim=-1).reshape(-1, 3)
    R = torch.tensor(matrix_from_quat(T_G_C[:4]), device=dev, dtype=torch.float64)
    o = torch.tensor(np.asarray(T_G_C[4:], dtype=np.float64), device=dev)
    d_w = d_c @ R.T
    inf = torch.full((d_w.shape[0],), float("inf"), device=dev, dtype=torch.float64)
    t_best = inf.clone()
    # room walls (camera is inside: take the exit distance)
    corridor = scene == "corridor"
    ox = float(T_G_C[4])
    for a in range(3):
        da = d_w[:, a]
        lo_a, hi_a = 0.0, ROOM[a]
        if corridor and a == 0:
            lo_a, hi_a = ox - CORRIDOR_CAP, ox + CORRIDOR_CAP
        t_hi = torch.where(da > 0, (hi_a - o[a]) / da, inf)
        t_lo = torch.where(da < 0, (lo_a - o[a]) / da, inf)
        t_best = torch.minimum(t_best, torch.minimum(t_hi, t_lo))
    # periodic copies of the objects that can be within sensor range of the camera
    shifts = [0.0]
    if corridor:
        k0 = math.floor(ox / PERIOD)
        shifts = [PERIOD * k for k in range(k0 - 1, k0 + 2)]
    spheres = [(cx + dx, cy, cz, r) for dx in shifts for (cx, cy, cz, r) in SPHERES]
    for (cx, cy, cz, r) in spheres:
        c = torch.tensor([cx, cy, cz], device=dev, dtype=torch.float64)
        oc = o - c
        A = (d_w * d_w).sum(1)
        B = 2.0 * (d_w * oc).sum(1)
        Cc = (oc * oc).sum() - r * r
        disc = B * B - 4 * A * Cc
        sq = torch.sqrt(torch.clamp(disc, min=0.0))
        t0 = (-B - sq) / (2 * A)
        t_hit = torch.where((disc > 0) & (t0 > 1e-6), t0, inf)
        t_best = torch.minimum(t_best, t_hit)
    boxes = [(x0 + dx, y0, z0, x1 + dx, y1, z1) for dx in shifts
             for (x0, y0, z0, x1, y1, z1) in BOXES]
    if near_box:  # a small object 5 cm in front of the lens: every point on it is closer than
        # min_ray_length_m and must be rejected (about a third of the frame)
        fwd = R[:, 2].cpu().numpy()
        oc_ = o.cpu().numpy()
        ctr = oc_ + 0.05 * fwd
        boxes.append((ctr[0] - 0.012, ctr[1] - 0.012, ctr[2] - 0.012,
                      ctr[0] + 0.012, ctr[1] + 0.012, ctr[2] + 0.012))
    for (x0, y0, z0, x1, y1, z1) in boxes:
        lo = torch.tensor([x0, y0, z0], device=dev, dtype=torch.float64)
        hi = torch.tensor([x1, y1, z1], device=dev, dtype=torch.float64)
        inv = 1.0 / d_w
        ta = (lo - o) * inv
        tb = (hi - o) * inv
        tmin = torch.minimum(ta, tb).max(dim=1).values
        tmax = torch.maximum(ta, tb).min(dim=1).values
        t_hit = torch.where((tmax >= tmin) & (tmin > 1e-6), tmin, inf)
        t_best = torch.minimum(t_best, t_hit)
    p_c = (d_c * t_best[:, None]).to(torch.float32)
    p_w = (o[None, :] + d_w * t_best[:, None]).to(torch.float32)
    colors = _hash_color(p_w + 1e-3)
    return p_c.contiguous(), colors.contiguous()


def render_depth_frame(T_G_C, cam=CAM_640x480, stride=1, scene="room", depth_encoding="16UC1"):
    """The frame render_frame casts, as the registered images a depth camera driver publishes.
    Returns (depth, rgb8 uint8 [H,W,3], camera dict): depth is z in millimetres rounded to nearest
    (uint16 [H,W], 16UC1) or z in metres (float32 [H,W], 32FC1); the colours are the hash colours
    of render_frame.  With stride > 1 the image is subsampled and the camera's intrinsics are
    scaled to match (pixel u of the result is pixel u * stride of the full image)."""
    pts, cols = render_frame(T_G_C, cam=cam, stride=stride, scene=scene)
    W = len(range(0, cam["width"], stride))
    H = len(range(0, cam["height"], stride))
    z = pts[:, 2].numpy().reshape(H, W)
    if depth_encoding == "16UC1":
        depth = np.clip(np.rint(z.astype(np.float64) * 1000.0), 0, 65535).astype(np.uint16)
    elif depth_encoding == "32FC1":
        depth = z.astype(np.float32)
    else:
        raise ValueError(f"unknown depth encoding {depth_encoding}")
    rgb = cols[:, :3].numpy().reshape(H, W, 3).copy()
    camera = dict(width=W, height=H, fx=cam["fx"] / stride, fy=cam["fy"] / stride,
                  cx=cam["cx"] / stride, cy=cam["cy"] / stride, depth_encoding=depth_encoding,
                  color_encoding="rgb8")
    return depth, rgb, camera


def submap_frames(robot, submap, frames, cam=CAM_640x480, device="cpu", stride=1):
    """Poses + rendered frames of one submap of one robot (robot map frame == world here)."""
    poses = trajectory(frames, robot=robot, submap=submap, frames_per_submap=frames)
    out = []
    for f in range(frames):
        pts, cols = render_frame(poses[f], cam=cam, device=device, stride=stride,
                                 near_box=((submap * frames + f) % 20 == 7))
        out.append((poses[f], pts, cols))
    return out


def corridor_trajectory(first_frame, num_frames, robot=0, advance=0.2, start_x=0.0):
    """Drive along the unbounded corridor scene: `advance` metres per frame in +x from
    start_x, robots on different lanes (y) and heights, the camera sweeping across the walls and
    the objects (never axis-aligned).  Frame k of a robot is the same whatever the batching."""
    poses = []
    for f in range(num_frames):
        k = first_frame + f
        s = 0.045 * k
        y = 2.6 + 0.35 * (robot % 8) + 0.12 * math.sin(0.31 * s + robot)
        z = 1.2 + 0.05 * (robot % 4) + 0.1 * math.sin(0.7 * s + 0.5 * robot)
        yaw = (-1.0 if robot % 2 == 0 else 1.0) * (math.pi / 2 - 0.75) + 0.55 * math.sin(0.23 * s + 0.8 * robot)
        pitch = 0.08 * math.sin(0.5 * s + robot)
        roll = 0.03 * math.cos(0.4 * s)
        poses.append(camera_pose((start_x + advance * k, y, z), yaw, pitch, roll))
    return np.stack(poses)


def corridor_frames(first_frame, num_frames, robot=0, advance=0.2, start_x=0.0, cam=CAM_640x480,
                    device="cpu", stride=1):
    """Poses + rendered frames [first_frame, first_frame + num_frames) of a corridor drive."""
    poses = corridor_trajectory(first_frame, num_frames, robot, advance, start_x)
    out = []
    for f in range(num_frames):
        pts, cols = render_frame(poses[f], cam=cam, device=device, stride=stride, scene="corridor")
        out.append((poses[f], pts, cols))
    return out


def robot_map_offset(robot):
    """Known SE(3) between robot map frames (SURVEY §8d C2: yaw 37 deg, t = (2.0,-1.5,0.1))."""
    if robot == 0:
        return np.array([1, 0, 0, 0, 0, 0, 0], dtype=np.float32)
    yaw = math.radians(37.0) * robot
    q = np.array([math.cos(yaw / 2), 0, 0, math.sin(yaw / 2)])
    t = np.array([2.0, -1.5, 0.1]) * robot
    return np.concatenate([q, t]).astype(np.float32)


def perturb_pose(T, rng, sigma_t=0.05, sigma_yaw_deg=1.0):
    """Seeded SE(3) perturbation emulating a pose-graph update (config C5)."""
    dyaw = math.radians(sigma_yaw_deg) * rng.standard_normal()
    dt = sigma_t * rng.standard_normal(3)
    d = np.concatenate([[math.cos(dyaw / 2), 0, 0, math.sin(dyaw / 2)], dt]).astype(np.float32)
    return compose(d, T)
