"""Host-side mirror of the reference's interface for the hot path, on top of the C ABI.

Names and argument meaning follow the calls the reference makes into voxblox / cblox:
  * ``TsdfIntegrator.integratePointCloud(T_G_C, points_C, colors, freespace_points=False)``
    — voxblox::TsdfIntegratorBase::integratePointCloud, called at
    coxgraph/include/coxgraph/map_comm/tsdf_recover.h:75;
  * ``mergeLayerAintoLayerB(layer_A, T_B_A, layer_B)`` — coxgraph/src/client/map_server.cpp:67-69;
  * ``getProjectedMap(submaps, poses, global_layer)`` — cblox SubmapCollection::getProjectedMap,
    reached from coxgraph/src/server/visualizer/server_visualizer.cpp:123-126;
  * ``Layer.removeAllBlocks()`` — tsdf_recover.h:62, map_server.cpp:65.
The C++ twin of this file is coxgraph_b200/host/coxgraph_b200.hpp.  Inputs may be numpy arrays
(host memory; copied by the library inside the call) or torch CUDA tensors (device memory on the
layer's GPU; no copy).  Errors raise CgError — the reference aborts through glog CHECK instead.
"""
import ctypes as C

import numpy as np

from . import capi

VOXEL_DTYPE = np.dtype([("distance", "<f4"), ("weight", "<f4"), ("rgba", "u1", (4,))])


def _is_cuda_tensor(x):
    return hasattr(x, "is_cuda") and bool(x.is_cuda)


def _ptr(a):
    return a.ctypes.data_as(C.c_void_p)


def TsdfIntegratorConfig(**overrides):
    """voxblox::TsdfIntegratorBase::Config with the upstream defaults."""
    cfg = capi.IntegratorConfig()
    capi.load().cg_integrator_config_default(C.byref(cfg))
    for k, v in overrides.items():
        if not hasattr(cfg, k):
            raise AttributeError(f"unknown integrator config field {k}")
        setattr(cfg, k, v)
    return cfg


def esdfConfig(**overrides):
    """voxblox::EsdfIntegrator::Config with upstream defaults."""
    cfg = capi.EsdfConfig()
    capi.load().cg_esdf_config_default(C.byref(cfg))
    for k, v in overrides.items():
        if not hasattr(cfg, k):
            raise AttributeError(k)
        setattr(cfg, k, v)
    return cfg


class Context:
    """One per GPU (per process rank)."""

    def __init__(self, device=0, stream=None):
        self._h = C.c_void_p()
        capi.check(capi.load().cg_context_create(int(device), C.c_void_p(stream or 0),
                                                 C.byref(self._h)))
        self.device = int(device)
        self.has_comm = False   # commInit done (multi-GPU merge through the C ABI)
        self.comm_rank = None   # this context's rank in its communicator

    def synchronize(self):
        capi.check(capi.load().cg_context_synchronize(self._h))

    def wait_stream(self, producer_stream):
        """Order the context's stream behind `producer_stream` (a raw cudaStream_t value)."""
        capi.check(capi.load().cg_context_wait_stream(self._h, C.c_void_p(producer_stream or 0)))

    def wait_torch(self):
        """Device tensors handed to the `*_device` entry points are read on the context's stream:
        order it behind torch's current stream, which produced them."""
        import torch
        self.wait_stream(torch.cuda.current_stream(self.device).cuda_stream)

    def set_profiling(self, enable=True):
        """Bracket every pipeline stage with CUDA events (voxblox::timing::Timer counterpart)."""
        capi.check(capi.load().cg_context_set_profiling(self._h, int(bool(enable))))

    def reset_profile(self):
        capi.check(capi.load().cg_context_reset_profile(self._h))

    def profile(self):
        """-> {stage: (accumulated ms, own kernel launches)}"""
        arr = (capi.StageProfile * 32)()
        n = C.c_size_t(0)
        capi.check(capi.load().cg_context_get_profile(self._h, arr, 32, C.byref(n)))
        return {arr[i].name.decode(): (arr[i].ms, int(arr[i].launches)) for i in range(n.value)}

    @property
    def kernel_launches(self):
        return int(capi.load().cg_context_kernel_launches(self._h))

    def close(self):
        if getattr(self, "_h", None):
            capi.load().cg_context_destroy(self._h)
            self._h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass


class Layer:
    """voxblox::Layer<TsdfVoxel> living in HBM (block hash + block pool)."""

    def __init__(self, ctx, voxel_size, voxels_per_side=16, max_blocks=4096):
        self.ctx = ctx
        self._h = C.c_void_p()
        capi.check(capi.load().cg_layer_create(ctx._h, float(voxel_size), int(voxels_per_side),
                                               int(max_blocks), C.byref(self._h)))
        self.voxel_size = float(np.float32(voxel_size))
        self.max_blocks = int(max_blocks)

    def close(self):
        if getattr(self, "_h", None) and getattr(self.ctx, "_h", None):
            capi.load().cg_layer_destroy(self._h)
        self._h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def removeAllBlocks(self):
        capi.check(capi.load().cg_layer_clear(self._h))

    clear = removeAllBlocks

    def removeBlocks(self, block_indices):
        """Layer::removeBlock for every listed (x, y, z) block index; returns how many existed."""
        idx = np.ascontiguousarray(block_indices, np.int32).reshape(-1, 3)
        removed = C.c_uint64(0)
        capi.check(capi.load().cg_layer_remove_blocks(self._h, len(idx), _ptr(idx),
                                                      C.byref(removed)))
        return int(removed.value)

    def removeBlock(self, block_index):
        return self.removeBlocks([block_index])

    def getNumberOfAllocatedBlocks(self):
        return int(capi.load().cg_layer_num_blocks(self._h))

    num_blocks = property(getNumberOfAllocatedBlocks)

    def block_indices(self):
        n = self.num_blocks
        idx = np.zeros((n, 3), np.int32)
        out = C.c_size_t(0)
        capi.check(capi.load().cg_layer_block_indices(self._h, n, _ptr(idx), C.byref(out)))
        return idx

    def download(self, out=None):
        """-> (block_idx int32 [B,3] sorted (z,y,x), voxels [B,4096] VOXEL_DTYPE, flags u8 [B]).

        `out` = (idx, voxels, flags) preallocated host arrays (e.g. views of pinned memory) with
        room for at least num_blocks blocks; slices of them are returned."""
        n = self.num_blocks
        if out is None:
            idx = np.zeros((n, 3), np.int32)
            vox = np.zeros((n, capi.VOXELS_PER_BLOCK), VOXEL_DTYPE)
            flags = np.zeros((n,), np.uint8)
            cap = n
        else:
            idx, vox, flags = out
            cap = min(len(idx), len(vox), len(flags))
        cnt = C.c_size_t(0)
        capi.check(capi.load().cg_layer_download(self._h, cap, _ptr(idx), _ptr(vox), _ptr(flags),
                                                 C.byref(cnt)))
        return idx[:n], vox[:n], flags[:n]

    def serializeLayerAsMsg(self, only_updated=False):
        """voxblox::serializeLayerAsMsg block payload: (block_idx int32 [B,3], data uint32
        [B, 12288]) — three words per voxel, colour packed a | b<<8 | g<<16 | r<<24."""
        lib = capi.load()
        n = C.c_size_t(0)
        capi.check(lib.cg_layer_serialize(self._h, int(bool(only_updated)), 0, None, None,
                                          C.byref(n)))
        idx = np.zeros((n.value, 3), np.int32)
        data = np.zeros((n.value, 3 * capi.VOXELS_PER_BLOCK), np.uint32)
        if n.value:
            capi.check(lib.cg_layer_serialize(self._h, int(bool(only_updated)), n.value, _ptr(idx),
                                              _ptr(data), C.byref(n)))
        return idx[:n.value], data[:n.value]

    def resetUpdated(self):
        capi.check(capi.load().cg_layer_reset_updated(self._h))

    def deserializeMsgToLayer(self, block_idx, data):
        idx = np.ascontiguousarray(block_idx, np.int32).reshape(-1, 3)
        words = np.ascontiguousarray(data, np.uint32).reshape(len(idx), 3 * capi.VOXELS_PER_BLOCK)
        capi.check(capi.load().cg_layer_deserialize(self._h, len(idx), _ptr(idx), _ptr(words)))

    def generateMesh(self, min_weight=1e-4, use_color=True, only_updated=False, fetch=True):
        """voxblox::MeshIntegrator<TsdfVoxel>::generateMesh on the device (marching cubes per
        block) -> (block_idx int32 [B,3] in (z,y,x) order, vertex_begin u32 [B+1], vertices f32
        [V,3], normals f32 [V,3], colors u8 [V,4]); three consecutive vertices = one triangle."""
        return _mesh(capi.load().cg_layer_mesh, self, min_weight, use_color, only_updated, fetch)

    def getConnectedMesh(self, fetch=True):
        """MeshLayer::getConnectedMesh (voxblox::createConnectedMesh) of the mesh the last
        generateMesh left on the device -> (vertices f32 [U,3], normals f32 [U,3], colors u8 [U,4],
        indices u32 [V]); with fetch=False only (U, V)."""
        lib = capi.load()
        nu, ni = C.c_size_t(0), C.c_size_t(0)
        capi.check(lib.cg_mesh_connect(self.ctx._h, 0, 0, None, None, None, None, C.byref(nu),
                                       C.byref(ni)))
        U, V = nu.value, ni.value
        if not fetch:
            return U, V
        v, n = np.zeros((U, 3), np.float32), np.zeros((U, 3), np.float32)
        c, idx = np.zeros((U, 4), np.uint8), np.zeros(V, np.uint32)
        if V:
            capi.check(lib.cg_mesh_connect(self.ctx._h, U, V, _ptr(v), _ptr(n), _ptr(c), _ptr(idx),
                                           C.byref(nu), C.byref(ni)))
        return v, n, c, idx

    def updateEsdfBatch(self, config=None, fetch=True):
        """voxblox::EsdfIntegrator::updateFromTsdfLayerBatch on the device
        (coxgraph/include/coxgraph/client/map_server.h:141-145).  The ESDF stays in the context;
        with fetch -> dict(idx int32 [B,3] in (z,y,x) order, distance f32 [B,4096], flags u8
        [B,4096] (1 observed, 2 hallucinated, 8 fixed), parent i8 [B,4096,3], stats)."""
        lib = capi.load()
        cfg = config if config is not None else esdfConfig()
        st = capi.EsdfStats()
        capi.check(lib.cg_layer_esdf_batch(self._h, C.byref(cfg), C.byref(st)))
        if not fetch:
            return st
        return self._fetch_esdf(st)

    def updateEsdf(self, config=None, fetch=True):
        """voxblox::EsdfIntegrator::updateFromTsdfLayer on the device: brings the ESDF retained in
        the context up to date with this layer, re-solving only the blocks within reach of what
        changed; the result is bit-identical to updateEsdfBatch(config).  Changes are found by
        content (the `updated` flags are left alone).  -> updateEsdfBatch's dict plus
        "update" (capi.EsdfUpdateStats); with fetch=False -> (stats, update stats)."""
        lib = capi.load()
        cfg = config if config is not None else esdfConfig()
        st, ust = capi.EsdfStats(), capi.EsdfUpdateStats()
        capi.check(lib.cg_layer_esdf_update(self._h, C.byref(cfg), C.byref(st), C.byref(ust)))
        if not fetch:
            return st, ust
        out = self._fetch_esdf(st)
        out["update"] = ust
        return out

    def _fetch_esdf(self, st):
        lib = capi.load()
        B = st.blocks
        idx = np.zeros((B, 3), np.int32)
        dist = np.zeros((B, capi.VOXELS_PER_BLOCK), np.float32)
        packed = np.zeros((B, capi.VOXELS_PER_BLOCK), np.uint32)
        if B:
            capi.check(lib.cg_esdf_fetch(self.ctx._h, B, _ptr(idx), _ptr(dist), _ptr(packed), None))
        parent = np.stack([(packed >> 24).astype(np.uint8).view(np.int8),
                           ((packed >> 16) & 0xFF).astype(np.uint8).view(np.int8),
                           ((packed >> 8) & 0xFF).astype(np.uint8).view(np.int8)], axis=-1)
        return dict(idx=idx, distance=dist, flags=(packed & 0xFF).astype(np.uint8), parent=parent,
                    packed=packed, stats=st)

    def esdfFreePoints(self, min_distance):
        """voxblox::createFreePointcloudFromEsdfLayer (coxgraph/src/client/map_server.cpp:112-113)
        on the ESDF the last updateEsdfBatch left in the context -> f32 [N,4] (x, y, z, distance)."""
        lib = capi.load()
        n = C.c_size_t(0)
        capi.check(lib.cg_esdf_free_points(self.ctx._h, float(min_distance), 0, None, C.byref(n)))
        out = np.zeros((n.value, 4), np.float32)
        if n.value:
            capi.check(lib.cg_esdf_free_points(self.ctx._h, float(min_distance), n.value, _ptr(out),
                                               C.byref(n)))
        return out

    def download_updated(self):
        """Blocks whose `updated` flag is set (Layer::getAllUpdatedBlocks), (z,y,x) order ->
        (block_idx int32 [B,3], voxels [B,4096] VOXEL_DTYPE, flags u8 [B])."""
        lib = capi.load()
        n = C.c_size_t(0)
        capi.check(lib.cg_layer_download_updated(self._h, 0, None, None, None, C.byref(n)))
        idx = np.zeros((n.value, 3), np.int32)
        vox = np.zeros((n.value, capi.VOXELS_PER_BLOCK), VOXEL_DTYPE)
        flags = np.zeros(n.value, np.uint8)
        if n.value:
            capi.check(lib.cg_layer_download_updated(self._h, n.value, _ptr(idx), _ptr(vox),
                                                     _ptr(flags), C.byref(n)))
        return idx, vox, flags

    def download_blocks(self, block_indices):
        """The listed blocks only -> (voxels [n,4096] VOXEL_DTYPE, flags u8 [n], found bool [n])."""
        idx = np.ascontiguousarray(block_indices, np.int32).reshape(-1, 3)
        vox = np.zeros((len(idx), capi.VOXELS_PER_BLOCK), VOXEL_DTYPE)
        flags = np.zeros(len(idx), np.uint8)
        found = np.zeros(len(idx), np.uint8)
        capi.check(capi.load().cg_layer_download_blocks(self._h, len(idx), _ptr(idx), _ptr(vox),
                                                        _ptr(flags), _ptr(found)))
        return vox, flags, found.astype(bool)

    def hash_stats(self):
        st = capi.HashStats()
        capi.check(capi.load().cg_layer_hash_stats(self._h, C.byref(st)))
        return st

    def upload(self, block_idx, voxels, flags=None):
        idx = np.ascontiguousarray(block_idx, np.int32).reshape(-1, 3)
        vox = np.ascontiguousarray(voxels, VOXEL_DTYPE).reshape(len(idx), capi.VOXELS_PER_BLOCK)
        fl = None if flags is None else np.ascontiguousarray(flags, np.uint8)
        capi.check(capi.load().cg_layer_upload(self._h, len(idx), _ptr(idx), _ptr(vox),
                                               None if fl is None else _ptr(fl)))


def _mesh(entry, layer, min_weight, use_color, only_updated, fetch):
    """cg_layer_mesh or cg_layer_mesh_sharded (`entry`), then cg_mesh_fetch: Layer.generateMesh."""
    nb, nv = C.c_size_t(0), C.c_size_t(0)
    capi.check(entry(layer._h, min_weight, int(use_color), int(only_updated), 0, 0, None, None,
                     None, None, None, C.byref(nb), C.byref(nv)))
    B, V = nb.value, nv.value
    if not fetch:  # the mesh stays on the device (cg_mesh_fetch copies it out later)
        return B, V
    return _fetch_mesh(layer.ctx, B, V)


def _fetch_mesh(ctx, B, V):
    """cg_mesh_fetch of the B blocks / V vertices retained in `ctx` -> generateMesh's tuple."""
    idx = np.zeros((B, 3), np.int32)
    begin = np.zeros(B + 1, np.uint32)
    v = np.zeros((V, 3), np.float32)
    n = np.zeros((V, 3), np.float32)
    c = np.zeros((V, 4), np.uint8)
    if B:
        capi.check(capi.load().cg_mesh_fetch(ctx._h, B, V, _ptr(idx), _ptr(begin),
                                             _ptr(v) if V else None, _ptr(n) if V else None,
                                             _ptr(c) if V else None))
    return idx, begin, v, n, c


class TsdfIntegrator:
    """Drop-in for voxblox::TsdfIntegratorBase (Simple / Merged) bound to one layer."""

    def __init__(self, config, layer):
        self.config = config
        self.layer = layer
        self.last_stats = capi.IntegrateStats()

    def integratePointCloud(self, T_G_C, points_C, colors, freespace_points=False):
        lib = capi.load()
        T = np.ascontiguousarray(T_G_C, np.float32).reshape(7)
        if _is_cuda_tensor(points_C):
            assert points_C.dtype.is_floating_point and points_C.element_size() == 4
            assert points_C.is_contiguous() and colors.is_contiguous() and _is_cuda_tensor(colors)
            n = points_C.numel() // 3
            assert colors.numel() * colors.element_size() == 4 * n
            self.layer.ctx.wait_torch()
            capi.check(lib.cg_integrate_pointcloud_device(
                self.layer._h, C.byref(self.config), _ptr(T), C.c_void_p(points_C.data_ptr()),
                C.c_void_p(colors.data_ptr()), n, int(freespace_points),
                C.byref(self.last_stats)))
        else:
            pts = np.ascontiguousarray(points_C, np.float32).reshape(-1, 3)
            cols = np.ascontiguousarray(colors, np.uint8).reshape(-1, 4)
            if len(pts) != len(cols):
                raise ValueError("points_C and colors differ in length")
            capi.check(lib.cg_integrate_pointcloud(
                self.layer._h, C.byref(self.config), _ptr(T), _ptr(pts), _ptr(cols), len(pts),
                int(freespace_points), C.byref(self.last_stats)))
        return self.last_stats

    def integrateBatch(self, poses, points_C, colors, frame_offsets, freespace_points=False):
        """F integratePointCloud calls (the loop of tsdf_recover.h:71-86) as one job."""
        lib = capi.load()
        P = np.ascontiguousarray(poses, np.float32).reshape(-1, 7)
        offs = np.ascontiguousarray(frame_offsets, np.uint64).reshape(-1)
        if len(offs) != len(P) + 1:
            raise ValueError("frame_offsets must have F+1 entries")
        if _is_cuda_tensor(points_C):
            assert points_C.is_contiguous() and colors.is_contiguous() and _is_cuda_tensor(colors)
            self.layer.ctx.wait_torch()
            capi.check(lib.cg_integrate_batch_device(
                self.layer._h, C.byref(self.config), len(P), _ptr(P),
                C.c_void_p(points_C.data_ptr()), C.c_void_p(colors.data_ptr()), _ptr(offs),
                int(freespace_points), C.byref(self.last_stats)))
        else:
            pts = np.ascontiguousarray(points_C, np.float32).reshape(-1, 3)
            cols = np.ascontiguousarray(colors, np.uint8).reshape(-1, 4)
            capi.check(lib.cg_integrate_batch(
                self.layer._h, C.byref(self.config), len(P), _ptr(P), _ptr(pts), _ptr(cols),
                _ptr(offs), int(freespace_points), C.byref(self.last_stats)))
        return self.last_stats


def _stage_batch(self, slot, points_C, colors):
    """Queue the host->device copy of a later integrateStaged(slot, ...) job (pinned numpy arrays;
    returns at once).  Keep the arrays alive until that job has returned."""
    pts = np.ascontiguousarray(points_C, np.float32).reshape(-1, 3)
    cols = np.ascontiguousarray(colors, np.uint8).reshape(-1, 4)
    if len(pts) != len(cols):
        raise ValueError("points_C and colors differ in length")
    capi.check(capi.load().cg_stage_batch_async(self.layer.ctx._h, int(slot), _ptr(pts), _ptr(cols),
                                                len(pts)))
    self._staged = getattr(self, "_staged", {})
    self._staged[int(slot)] = (pts, cols)


def _integrate_staged(self, slot, poses, frame_offsets, freespace_points=False):
    """integrateBatch on the inputs staged in `slot`."""
    P = np.ascontiguousarray(poses, np.float32).reshape(-1, 7)
    offs = np.ascontiguousarray(frame_offsets, np.uint64).reshape(-1)
    if len(offs) != len(P) + 1:
        raise ValueError("frame_offsets must have F+1 entries")
    capi.check(capi.load().cg_integrate_batch_staged(
        self.layer._h, C.byref(self.config), len(P), _ptr(P), int(slot), _ptr(offs),
        int(freespace_points), C.byref(self.last_stats)))
    getattr(self, "_staged", {}).pop(int(slot), None)
    return self.last_stats


def _prepare_batch(self, slot, poses, points_C, colors, frame_offsets, freespace_points=False):
    """Queue the layer-independent first half of a LATER integrateBatch job (device tensors) on the
    context's second stream; integratePrepared(slot) completes it.  Keep the tensors alive and
    unchanged until then."""
    P = np.ascontiguousarray(poses, np.float32).reshape(-1, 7)
    offs = np.ascontiguousarray(frame_offsets, np.uint64).reshape(-1)
    if len(offs) != len(P) + 1:
        raise ValueError("frame_offsets must have F+1 entries")
    assert _is_cuda_tensor(points_C) and _is_cuda_tensor(colors)
    assert points_C.is_contiguous() and colors.is_contiguous()
    self.layer.ctx.wait_torch()
    capi.check(capi.load().cg_prepare_batch_device(
        self.layer._h, C.byref(self.config), len(P), _ptr(P), C.c_void_p(points_C.data_ptr()),
        C.c_void_p(colors.data_ptr()), _ptr(offs), int(freespace_points), int(slot)))
    self._prepared = getattr(self, "_prepared", {})
    self._prepared[int(slot)] = (points_C, colors)


def _prepare_staged(self, slot, stage_slot, poses, frame_offsets, freespace_points=False):
    """The same for inputs staged with stageBatch(stage_slot, ...)."""
    P = np.ascontiguousarray(poses, np.float32).reshape(-1, 7)
    offs = np.ascontiguousarray(frame_offsets, np.uint64).reshape(-1)
    if len(offs) != len(P) + 1:
        raise ValueError("frame_offsets must have F+1 entries")
    capi.check(capi.load().cg_prepare_batch_staged(
        self.layer._h, C.byref(self.config), len(P), _ptr(P), int(stage_slot), _ptr(offs),
        int(freespace_points), int(slot)))


def _integrate_prepared(self, slot):
    capi.check(capi.load().cg_integrate_prepared(self.layer._h, int(slot),
                                                 C.byref(self.last_stats)))
    getattr(self, "_prepared", {}).pop(int(slot), None)
    return self.last_stats


def depthCamera(camera):
    """capi.DepthCamera from a DepthCamera, or from a dict with width, height, fx, fy, cx, cy (e.g.
    synth.CAM_640x480) and optional depth_encoding ("16UC1" / "32FC1", default "16UC1") and
    color_encoding ("rgb8", "rgba8", "bgr8", "bgra8", "mono8", default "rgb8")."""
    if isinstance(camera, capi.DepthCamera):
        return camera

    def enc(v, table):
        return table[v] if isinstance(v, str) else int(v)
    return capi.DepthCamera(int(camera["width"]), int(camera["height"]), float(camera["fx"]),
                            float(camera["fy"]), float(camera["cx"]), float(camera["cy"]),
                            enc(camera.get("depth_encoding", "16UC1"), capi.DEPTH_ENCODINGS),
                            enc(camera.get("color_encoding", "rgb8"), capi.COLOR_ENCODINGS))


def _depth_images(cam, F, depth, color, device):
    """Checks the images of F frames against the camera; numpy arrays (host) are made contiguous.
    -> (depth, color, pointer of depth, pointer of color)."""
    n = F * cam.width * cam.height
    depth_item = 2 if cam.depth_encoding == capi.DEPTH_16UC1 else 4
    color_bytes = n * capi.COLOR_PIXEL_BYTES.get(cam.color_encoding, 0)
    if device:
        assert _is_cuda_tensor(depth) and _is_cuda_tensor(color)
        assert depth.is_contiguous() and color.is_contiguous()
        ok = (depth.numel() == n and depth.element_size() == depth_item and
              color.numel() * color.element_size() == color_bytes)
        ptrs = (C.c_void_p(depth.data_ptr()), C.c_void_p(color.data_ptr()))
    else:
        dtype = np.uint16 if cam.depth_encoding == capi.DEPTH_16UC1 else np.float32
        depth = np.ascontiguousarray(depth, dtype)
        color = np.ascontiguousarray(color, np.uint8)
        ok = depth.size == n and color.size == color_bytes
        ptrs = (_ptr(depth), _ptr(color))
    if not ok:
        raise ValueError(f"images do not match {F} frames of {cam.width} x {cam.height} with the "
                         "camera's encodings")
    return depth, color, ptrs[0], ptrs[1]


def _integrate_depth_batch(self, poses, depth, color, camera):
    """F TsdfServer insertions of registered depth + colour images (depth_image_proc
    point_cloud_xyzrgb, the finite filter of convertPointcloud, integratePointCloud) as one job:
    depth [F,H,W] uint16 (16UC1) or float32 (32FC1), color [F,H,W,C].  numpy arrays (host) or
    contiguous CUDA tensors (device)."""
    cam = depthCamera(camera)
    P = np.ascontiguousarray(poses, np.float32).reshape(-1, 7)
    device = _is_cuda_tensor(depth)
    depth, color, dp, cp = _depth_images(cam, len(P), depth, color, device)
    lib = capi.load()
    if device:
        self.layer.ctx.wait_torch()
        capi.check(lib.cg_integrate_depth_batch_device(self.layer._h, C.byref(self.config), len(P),
                                                       _ptr(P), C.byref(cam), dp, cp,
                                                       C.byref(self.last_stats)))
    else:
        capi.check(lib.cg_integrate_depth_batch(self.layer._h, C.byref(self.config), len(P), _ptr(P),
                                                C.byref(cam), dp, cp, C.byref(self.last_stats)))
    return self.last_stats


def _integrate_depth_image(self, T_G_C, depth, color, camera):
    """One frame of integrateDepthBatch: depth [H,W], color [H,W,C]."""
    return self.integrateDepthBatch(np.asarray(T_G_C, np.float32).reshape(1, 7), depth, color,
                                    camera)


def _stage_depth(self, slot, depth, color, camera):
    """Queue the host->device copy of the images of a later integrateDepthStaged /
    prepareDepthStaged job (pinned numpy arrays; returns at once).  Keep them alive until then."""
    cam = depthCamera(camera)
    F = int(np.asarray(depth).size // max(1, cam.width * cam.height))
    depth, color, dp, cp = _depth_images(cam, F, depth, color, False)
    capi.check(capi.load().cg_stage_depth_async(self.layer.ctx._h, int(slot), C.byref(cam), F, dp, cp))
    self._staged = getattr(self, "_staged", {})
    self._staged[int(slot)] = (depth, color)


def _integrate_depth_staged(self, slot, poses, camera):
    """integrateDepthBatch on the images staged in `slot`."""
    cam = depthCamera(camera)
    P = np.ascontiguousarray(poses, np.float32).reshape(-1, 7)
    capi.check(capi.load().cg_integrate_depth_staged(self.layer._h, C.byref(self.config), len(P),
                                                     _ptr(P), C.byref(cam), int(slot),
                                                     C.byref(self.last_stats)))
    getattr(self, "_staged", {}).pop(int(slot), None)
    return self.last_stats


def _prepare_depth(self, slot, poses, depth, color, camera):
    """prepareBatch for a depth job (CUDA tensors); integratePrepared(slot) completes it."""
    cam = depthCamera(camera)
    P = np.ascontiguousarray(poses, np.float32).reshape(-1, 7)
    depth, color, dp, cp = _depth_images(cam, len(P), depth, color, True)
    self.layer.ctx.wait_torch()
    capi.check(capi.load().cg_prepare_depth_device(self.layer._h, C.byref(self.config), len(P),
                                                   _ptr(P), C.byref(cam), dp, cp, int(slot)))
    self._prepared = getattr(self, "_prepared", {})
    self._prepared[int(slot)] = (depth, color)


def _prepare_depth_staged(self, slot, stage_slot, poses, camera):
    """The same for images staged with stageDepth(stage_slot, ...)."""
    cam = depthCamera(camera)
    P = np.ascontiguousarray(poses, np.float32).reshape(-1, 7)
    capi.check(capi.load().cg_prepare_depth_staged(self.layer._h, C.byref(self.config), len(P),
                                                   _ptr(P), C.byref(cam), int(stage_slot), int(slot)))


TsdfIntegrator.integrateDepthBatch = _integrate_depth_batch
TsdfIntegrator.integrateDepthImage = _integrate_depth_image
TsdfIntegrator.stageDepth = _stage_depth
TsdfIntegrator.integrateDepthStaged = _integrate_depth_staged
TsdfIntegrator.prepareDepth = _prepare_depth
TsdfIntegrator.prepareDepthStaged = _prepare_depth_staged
TsdfIntegrator.stageBatch = _stage_batch
TsdfIntegrator.integrateStaged = _integrate_staged
TsdfIntegrator.prepareBatch = _prepare_batch
TsdfIntegrator.prepareStaged = _prepare_staged
TsdfIntegrator.integratePrepared = _integrate_prepared


def meshToFrames(ctx, mesh, interpolate_voxel_size, poses, stamps_sec):
    """voxblox::MeshConverter (coxgraph/include/coxgraph/map_comm/mesh_converter.h):
    convertToPointCloud + getNextPointcloud for every trajectory pose.
    -> (frame_offsets u64 [F+1], points_C f32 [N,3], colors u8 [N,4])."""
    lib = capi.load()
    m, keep = capi.make_mesh(mesh)
    P = np.ascontiguousarray(poses, np.float32).reshape(-1, 7)
    st = np.ascontiguousarray(stamps_sec, np.float64).reshape(-1)
    offs = np.zeros(len(P) + 1, np.uint64)
    capi.check(lib.cg_mesh_to_frames(ctx._h, C.byref(m), float(interpolate_voxel_size), len(P),
                                     _ptr(P), _ptr(st), _ptr(offs), None, None, 0))
    n = int(offs[-1])
    pts, cols = np.zeros((n, 3), np.float32), np.zeros((n, 4), np.uint8)
    if n:
        capi.check(lib.cg_mesh_to_frames(ctx._h, C.byref(m), float(interpolate_voxel_size), len(P),
                                         _ptr(P), _ptr(st), _ptr(offs), _ptr(pts), _ptr(cols), n))
    return offs, pts, cols


def recoverMesh(layer, config, mesh, interpolate_voxel_size, poses, stamps_sec):
    """TsdfRecover::processMesh (coxgraph/include/coxgraph/map_comm/tsdf_recover.h:59-99) on the
    device: clear the layer, mesh -> per-pose clouds, integrate them.  Returns IntegrateStats."""
    m, keep = capi.make_mesh(mesh)
    P = np.ascontiguousarray(poses, np.float32).reshape(-1, 7)
    st = np.ascontiguousarray(stamps_sec, np.float64).reshape(-1)
    stats = capi.IntegrateStats()
    capi.check(capi.load().cg_recover_mesh(layer._h, C.byref(config), C.byref(m),
                                           float(interpolate_voxel_size), len(P), _ptr(P), _ptr(st),
                                           C.byref(stats)))
    return stats


def mergeLayerAintoLayerB(layer_A, T_B_A, layer_B):
    """voxblox::mergeLayerAintoLayerB(layer_A, T_B_A, &layer_B); returns MergeStats."""
    T = np.ascontiguousarray(T_B_A, np.float32).reshape(7)
    st = capi.MergeStats()
    capi.check(capi.load().cg_merge_layer_into_layer(layer_A._h, _ptr(T), layer_B._h,
                                                     C.byref(st)))
    return st


def getProjectedMap(submap_layers, submap_poses, global_layer, want_stats=False):
    """cblox SubmapCollection::getProjectedMap(): merge every submap into global_layer in order."""
    n = len(submap_layers)
    P = np.ascontiguousarray(submap_poses, np.float32).reshape(n, 7)
    arr = (C.c_void_p * n)(*[l._h for l in submap_layers])
    st = capi.MergeStats()
    capi.check(capi.load().cg_project_submaps(arr, _ptr(P), n, global_layer._h,
                                              C.byref(st) if want_stats else None))
    return st if want_stats else None


def commUniqueId():
    """ncclGetUniqueId as bytes: made on one rank, handed to every rank by the host."""
    buf = (C.c_uint8 * 128)()
    capi.check(capi.load().cg_comm_get_unique_id(buf))
    return bytes(buf)


def commInit(ctx, unique_id, rank, nranks):
    """Communicator of the multi-GPU merge on the context's GPU (collective over the ranks)."""
    buf = (C.c_uint8 * 128).from_buffer_copy(unique_id)
    capi.check(capi.load().cg_comm_init(ctx._h, buf, int(rank), int(nranks)))
    ctx.has_comm = True
    ctx.comm_rank = int(rank)


def gatherGlobal(partial_layer, owned_layer):
    """Collective: every rank's partial global blocks go to their owners (fold over NVLink peer
    memory, ascending source rank).  Returns the number of blocks folded into owned_layer."""
    n = C.c_uint64(0)
    capi.check(capi.load().cg_gather_global(partial_layer._h, owned_layer._h, C.byref(n)))
    return int(n.value)


def getProjectedMapSharded(submap_layers, submap_poses, partial_layer, owned_layer):
    """getProjectedMap() over all ranks: this rank's submaps -> partial_layer, then gatherGlobal."""
    n = len(submap_layers)
    P = np.ascontiguousarray(submap_poses, np.float32).reshape(n, 7)
    arr = (C.c_void_p * max(n, 1))(*[l._h for l in submap_layers])
    capi.check(capi.load().cg_project_submaps_sharded(arr, _ptr(P) if n else None, n,
                                                      partial_layer._h, owned_layer._h, None))


def reprojectSubmapsSharded(submap_layers, poses_old, poses_new, partial_layer, owned_layer,
                            eps_translation=0.0, eps_rotation=0.0):
    """Collective: reprojectSubmaps over all ranks after getProjectedMapSharded.  This rank's
    first len(poses_old) submaps are the ones it projected last (with poses_old), the rest are new;
    poses_new has one pose per submap.  Afterwards partial_layer and owned_layer hold exactly what
    a fresh getProjectedMapSharded under the effective poses would leave; only the owned blocks
    whose holders or copies changed are folded again (and flagged updated).  Returns (changed
    mask, ReprojectShardedStats)."""
    n = len(submap_layers)
    Po = np.ascontiguousarray(poses_old, np.float32).reshape(-1, 7)
    Pn = np.ascontiguousarray(poses_new, np.float32).reshape(n, 7)
    arr = (C.c_void_p * max(n, 1))(*[l._h for l in submap_layers])
    changed = np.zeros(max(n, 1), np.uint8)
    st = capi.ReprojectShardedStats()
    capi.check(capi.load().cg_reproject_submaps_sharded(
        arr, n, len(Po), _ptr(Po) if len(Po) else None, _ptr(Pn) if n else None,
        float(eps_translation), float(eps_rotation), partial_layer._h, owned_layer._h,
        _ptr(changed), C.byref(st)))
    return changed[:n].astype(bool), st


def generateMeshSharded(owned_layer, min_weight=1e-4, use_color=True, only_updated=False,
                        fetch=True):
    """Collective: generateMesh over the sharded global map, every rank with its owned layer.  Each
    rank gets the meshes of the blocks it holds, byte for byte what generateMesh gives for them on
    one layer holding every rank's owned blocks (neighbour and colour blocks are read from the
    peers).  Same tuple as Layer.generateMesh."""
    return _mesh(capi.load().cg_layer_mesh_sharded, owned_layer, min_weight, use_color,
                 only_updated, fetch)


def gatherMeshSharded(ctx, root=0, fetch=True):
    """Collective, right after generateMeshSharded on every rank: the ranks' block meshes are
    gathered onto rank `root`, which then holds exactly what generateMesh leaves for one layer
    holding every rank's owned blocks (so getConnectedMesh there is the combined map's PLY mesh).
    Returns Layer.generateMesh's tuple on the root (with fetch=False only the global (B, V)) and
    the global (B, V) on the other ranks, whose own share stays retained."""
    nb, nv = C.c_size_t(0), C.c_size_t(0)
    capi.check(capi.load().cg_mesh_gather_sharded(ctx._h, int(root), C.byref(nb), C.byref(nv)))
    B, V = nb.value, nv.value
    if not fetch or ctx.comm_rank != int(root):
        return B, V
    return _fetch_mesh(ctx, B, V)


def commPeerMappings(ctx):
    """(peer mappings opened since commInit, open now) of the context's communicator."""
    opened, now = C.c_uint64(0), C.c_uint64(0)
    capi.check(capi.load().cg_comm_peer_mappings(ctx._h, C.byref(opened), C.byref(now)))
    return int(opened.value), int(now.value)


def reprojectSubmaps(submap_layers, poses_old, poses_new, global_layer, eps_translation=0.0,
                     eps_rotation=0.0):
    """Incremental getProjectedMap() after a pose-graph update (SURVEY §8f N1): global_layer must
    hold the projection under poses_old; afterwards it is bit-identical to a fresh projection with
    the moved submaps at poses_new.  Returns (changed mask, ReprojectStats)."""
    n = len(submap_layers)
    Po = np.ascontiguousarray(poses_old, np.float32).reshape(n, 7)
    Pn = np.ascontiguousarray(poses_new, np.float32).reshape(n, 7)
    arr = (C.c_void_p * n)(*[l._h for l in submap_layers])
    changed = np.zeros(n, np.uint8)
    st = capi.ReprojectStats()
    capi.check(capi.load().cg_reproject_submaps(arr, _ptr(Po), _ptr(Pn), n, float(eps_translation),
                                                float(eps_rotation), global_layer._h, _ptr(changed),
                                                C.byref(st)))
    return changed.astype(bool), st


def block_owner(block_idx, nranks):
    return int(capi.load().cg_block_owner(int(block_idx[0]), int(block_idx[1]),
                                          int(block_idx[2]), int(nranks)))
