"""ctypes binding of the CPU oracle (oracle/tsdf_oracle.{h,cc}).

TEST INFRASTRUCTURE ONLY: imported by tests/, __graft_entry__.smoke() and bench.py's
cpu_baseline / --impl reference legs.  The product (coxgraph_b200/) never imports this.
"""
import ctypes as C
import os
import subprocess

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
_LIB_PATH = os.path.join(_HERE, "_build", "libtsdf_oracle.so")

VOXELS_PER_BLOCK = 4096
VOXEL_DTYPE = np.dtype([("distance", "<f4"), ("weight", "<f4"), ("rgba", "u1", (4,))])
assert VOXEL_DTYPE.itemsize == 12
# orc_visit: one updateTsdfVoxel call (global voxel index, sdf, effective weight, ray colour)
VISIT_DTYPE = np.dtype([("idx", "<i4", (3,)), ("sdf", "<f4"), ("weight", "<f4"),
                        ("rgba", "u1", (4,))])
assert VISIT_DTYPE.itemsize == 24


class IntegratorConfig(C.Structure):
    """Mirror of orc_integrator_config (voxblox TsdfIntegratorBase::Config)."""

    _fields_ = [
        ("default_truncation_distance", C.c_float),
        ("max_weight", C.c_float),
        ("voxel_carving_enabled", C.c_int32),
        ("min_ray_length_m", C.c_float),
        ("max_ray_length_m", C.c_float),
        ("use_const_weight", C.c_int32),
        ("allow_clear", C.c_int32),
        ("use_weight_dropoff", C.c_int32),
        ("use_sparsity_compensation_factor", C.c_int32),
        ("sparsity_compensation_factor", C.c_float),
        ("enable_anti_grazing", C.c_int32),
        ("method", C.c_int32),
        ("integration_order_mode", C.c_int32),
        ("start_voxel_subsampling_factor", C.c_float),
        ("max_consecutive_ray_collisions", C.c_int32),
    ]


class EsdfConfig(C.Structure):
    """Mirror of orc_esdf_config (voxblox EsdfIntegrator::Config)."""

    _fields_ = [
        ("max_distance_m", C.c_float),
        ("default_distance_m", C.c_float),
        ("min_distance_m", C.c_float),
        ("min_diff_m", C.c_float),
        ("min_weight", C.c_float),
        ("num_buckets", C.c_int32),
        ("multi_queue", C.c_int32),
        ("add_occupied_crust", C.c_int32),
    ]


def build(force=False):
    if force or not os.path.exists(_LIB_PATH) or os.path.getmtime(_LIB_PATH) < max(
        os.path.getmtime(os.path.join(_HERE, f)) for f in ("tsdf_oracle.cc", "tsdf_oracle.h")
    ):
        subprocess.check_call(["make", "-C", _HERE, "-s"])
    return _LIB_PATH


_lib = None


def lib():
    global _lib
    if _lib is None:
        _lib = C.CDLL(build())
        L = _lib
        L.orc_layer_create.restype = C.c_void_p
        L.orc_layer_create.argtypes = [C.c_float, C.c_int32]
        L.orc_layer_destroy.argtypes = [C.c_void_p]
        L.orc_layer_clear.argtypes = [C.c_void_p]
        L.orc_layer_num_blocks.restype = C.c_size_t
        L.orc_layer_num_blocks.argtypes = [C.c_void_p]
        L.orc_layer_download.argtypes = [C.c_void_p] * 4
        L.orc_layer_upload.argtypes = [C.c_void_p] * 4 + [C.c_size_t]
        L.orc_default_config.argtypes = [C.POINTER(IntegratorConfig)]
        L.orc_integrate_pointcloud.restype = C.c_int32
        L.orc_integrate_pointcloud.argtypes = [
            C.c_void_p, C.POINTER(IntegratorConfig), C.c_void_p, C.c_void_p, C.c_void_p,
            C.c_size_t, C.c_int32, C.POINTER(C.c_uint64)]
        L.orc_integrate_pointcloud_traced.restype = C.c_int32
        L.orc_integrate_pointcloud_traced.argtypes = [
            C.c_void_p, C.POINTER(IntegratorConfig), C.c_void_p, C.c_void_p, C.c_void_p,
            C.c_size_t, C.c_int32, C.POINTER(C.c_uint64), C.POINTER(C.c_void_p),
            C.POINTER(C.c_size_t)]
        L.orc_trace_free.argtypes = [C.c_void_p]
        L.orc_integrate_pointcloud_mt.restype = C.c_int32
        L.orc_integrate_pointcloud_mt.argtypes = [
            C.c_void_p, C.POINTER(IntegratorConfig), C.c_void_p, C.c_void_p, C.c_void_p,
            C.c_size_t, C.c_int32, C.c_int32]
        L.orc_merge_layer_into_layer.restype = C.c_int32
        L.orc_merge_layer_into_layer.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p,
                                                 C.POINTER(C.c_uint64)]
        L.orc_merge_layer_into_layer_mt.restype = C.c_int32
        L.orc_merge_layer_into_layer_mt.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p, C.c_int32,
                                                    C.POINTER(C.c_uint64)]
        L.orc_merge_layer_aligned.restype = C.c_int32
        L.orc_merge_layer_aligned.argtypes = [C.c_void_p, C.c_void_p]
        L.orc_mesh_to_frames.restype = C.c_size_t
        L.orc_mesh_to_frames.argtypes = [C.c_void_p, C.c_float, C.c_size_t, C.c_void_p, C.c_void_p,
                                         C.c_void_p, C.c_void_p, C.c_void_p, C.c_size_t]
        L.orc_transform_point.argtypes = [C.c_void_p] * 3
        L.orc_inverse_transform.argtypes = [C.c_void_p] * 2
        L.orc_cast_ray.restype = C.c_size_t
        L.orc_cast_ray.argtypes = [C.c_void_p, C.c_void_p, C.c_int32, C.c_int32, C.c_float,
                                   C.c_float, C.c_float, C.c_int32, C.c_void_p, C.c_size_t]
        L.orc_layer_mesh.restype = C.c_size_t
        L.orc_layer_mesh.argtypes = [C.c_void_p, C.c_float, C.c_int32, C.c_int32, C.c_void_p,
                                     C.c_void_p, C.c_void_p, C.c_void_p, C.c_size_t]
        L.orc_connect_mesh.restype = C.c_size_t
        L.orc_connect_mesh.argtypes = [C.c_void_p, C.c_size_t, C.c_void_p, C.c_void_p]
        L.orc_triangle_table.restype = C.POINTER(C.c_int)
        L.orc_triangle_table.argtypes = []
        L.orc_esdf_default_config.argtypes = [C.POINTER(EsdfConfig)]
        L.orc_esdf_batch.restype = C.c_void_p
        L.orc_esdf_batch.argtypes = [C.c_void_p, C.POINTER(EsdfConfig)]
        L.orc_esdf_destroy.argtypes = [C.c_void_p]
        L.orc_esdf_num_blocks.restype = C.c_size_t
        L.orc_esdf_num_blocks.argtypes = [C.c_void_p]
        L.orc_esdf_updates.restype = C.c_uint64
        L.orc_esdf_updates.argtypes = [C.c_void_p]
        L.orc_esdf_download.argtypes = [C.c_void_p] * 5
        L.orc_esdf_free_points.restype = C.c_size_t
        L.orc_esdf_free_points.argtypes = [C.c_void_p, C.c_float, C.c_void_p, C.c_size_t]
        L.orc_interp_voxel.restype = C.c_int32
        L.orc_interp_voxel.argtypes = [C.c_void_p, C.c_void_p, C.c_int32, C.POINTER(C.c_float),
                                       C.POINTER(C.c_float), C.c_void_p]
    return _lib


def default_config(**over):
    cfg = IntegratorConfig()
    lib().orc_default_config(C.byref(cfg))
    for k, v in over.items():
        if not hasattr(cfg, k):
            raise AttributeError(k)
        setattr(cfg, k, v)
    return cfg


def default_esdf_config(**over):
    cfg = EsdfConfig()
    lib().orc_esdf_default_config(C.byref(cfg))
    for k, v in over.items():
        if not hasattr(cfg, k):
            raise AttributeError(k)
        setattr(cfg, k, v)
    return cfg


def _f32(a, shape=None):
    a = np.ascontiguousarray(a, dtype=np.float32)
    if shape is not None:
        a = a.reshape(shape)
    return a


def _ptr(a):
    return a.ctypes.data_as(C.c_void_p)


class Layer:
    """Oracle Layer<TsdfVoxel>."""

    def __init__(self, voxel_size, voxels_per_side=16):
        self._h = lib().orc_layer_create(float(voxel_size), int(voxels_per_side))
        if not self._h:
            raise ValueError("bad layer parameters")
        self.voxel_size = float(np.float32(voxel_size))
        self.last_blocks_touched = 0
        self.last_blocks_out = 0

    def __del__(self):
        if getattr(self, "_h", None) and _lib is not None:  # module globals are gone at shutdown
            _lib.orc_layer_destroy(self._h)
            self._h = None

    def clear(self):
        lib().orc_layer_clear(self._h)

    @property
    def num_blocks(self):
        return lib().orc_layer_num_blocks(self._h)

    def integrate(self, cfg, T_G_C, points, colors, freespace=False, threads=0, trace=False):
        """integratePointCloud.  trace=True (single thread only) returns every voxel update of
        the call in order as a VISIT_DTYPE array."""
        pts = _f32(points, (-1, 3))
        cols = np.ascontiguousarray(colors, dtype=np.uint8).reshape(-1, 4)
        assert len(pts) == len(cols)
        T = _f32(T_G_C, (7,))
        if trace and threads and threads > 0:
            raise ValueError("the visit trace needs the single-threaded integrator (threads=0)")
        if trace:
            touched, buf, n = C.c_uint64(0), C.c_void_p(), C.c_size_t(0)
            rc = lib().orc_integrate_pointcloud_traced(self._h, C.byref(cfg), _ptr(T), _ptr(pts),
                                                       _ptr(cols), len(pts), int(freespace),
                                                       C.byref(touched), C.byref(buf), C.byref(n))
            if rc != 0:
                raise RuntimeError(f"oracle integrate failed rc={rc}")
            self.last_blocks_touched = touched.value
            out = np.zeros(n.value, VISIT_DTYPE)
            if n.value:
                C.memmove(out.ctypes.data, buf, n.value * VISIT_DTYPE.itemsize)
                lib().orc_trace_free(buf)
            return out
        if threads and threads > 0:
            rc = lib().orc_integrate_pointcloud_mt(self._h, C.byref(cfg), _ptr(T), _ptr(pts),
                                                   _ptr(cols), len(pts), int(freespace), threads)
        else:
            touched = C.c_uint64(0)
            rc = lib().orc_integrate_pointcloud(self._h, C.byref(cfg), _ptr(T), _ptr(pts),
                                                _ptr(cols), len(pts), int(freespace),
                                                C.byref(touched))
            self.last_blocks_touched = touched.value
        if rc != 0:
            raise RuntimeError(f"oracle integrate failed rc={rc}")

    def merge_from(self, layer_a, T_B_A, threads=0):
        """mergeLayerAintoLayerB(layer_a, T_B_A, self)."""
        T = _f32(T_B_A, (7,))
        out = C.c_uint64(0)
        if threads and threads > 1:
            rc = lib().orc_merge_layer_into_layer_mt(layer_a._h, _ptr(T), self._h, threads,
                                                     C.byref(out))
        else:
            rc = lib().orc_merge_layer_into_layer(layer_a._h, _ptr(T), self._h, C.byref(out))
        self.last_blocks_out = out.value
        if rc != 0:
            raise RuntimeError(f"oracle merge failed rc={rc}")

    def merge_aligned_from(self, layer_a):
        """2-argument mergeLayerAintoLayerB(layer_a, self) (same grid, voxel-wise)."""
        if lib().orc_merge_layer_aligned(layer_a._h, self._h) != 0:
            raise RuntimeError("oracle aligned merge failed")

    def download(self):
        """-> (block_idx int32 [B,3] sorted (z,y,x), voxels [B,4096] VOXEL_DTYPE, flags u8 [B])."""
        n = self.num_blocks
        idx = np.zeros((n, 3), np.int32)
        vox = np.zeros((n, VOXELS_PER_BLOCK), VOXEL_DTYPE)
        flags = np.zeros((n,), np.uint8)
        if n:
            lib().orc_layer_download(self._h, _ptr(idx), _ptr(vox), _ptr(flags))
        return idx, vox, flags

    def upload(self, idx, vox, flags=None):
        idx = np.ascontiguousarray(idx, np.int32).reshape(-1, 3)
        vox = np.ascontiguousarray(vox, VOXEL_DTYPE).reshape(len(idx), VOXELS_PER_BLOCK)
        fl = None if flags is None else np.ascontiguousarray(flags, np.uint8)
        lib().orc_layer_upload(self._h, _ptr(idx), _ptr(vox), None if fl is None else _ptr(fl),
                               len(idx))

    def mesh(self, min_weight=1e-4, use_color=True, only_updated=False):
        """MeshIntegrator::generateMesh -> (vertex_begin u32 [B+1], vertices f32 [V,3],
        normals f32 [V,3], colors u8 [V,4]); blocks in (z,y,x) order."""
        nb = self.num_blocks
        begin = np.zeros(nb + 1, np.uint32)
        n = lib().orc_layer_mesh(self._h, min_weight, int(use_color), int(only_updated),
                                 _ptr(begin), None, None, None, 0)
        v = np.zeros((n, 3), np.float32)
        nr = np.zeros((n, 3), np.float32)
        c = np.zeros((n, 4), np.uint8)
        if n:
            lib().orc_layer_mesh(self._h, min_weight, int(use_color), int(only_updated),
                                 _ptr(begin), _ptr(v), _ptr(nr), _ptr(c), n)
        return begin, v, nr, c

    def esdf_batch(self, cfg=None, free_min_distance=None):
        """EsdfIntegrator::updateFromTsdfLayerBatch on this TSDF layer -> dict(idx int32 [B,3] in
        (z,y,x) order, distance f32 [B,4096], flags u8 [B,4096] (1 observed, 2 hallucinated,
        4 in_queue, 8 fixed), parent i8 [B,4096,3], updates); with free_min_distance also
        free_points f32 [N,4] (createFreePointcloudFromEsdfLayer)."""
        cfg = cfg if cfg is not None else default_esdf_config()
        h = lib().orc_esdf_batch(self._h, C.byref(cfg))
        try:
            n = lib().orc_esdf_num_blocks(h)
            out = dict(idx=np.zeros((n, 3), np.int32),
                       distance=np.zeros((n, VOXELS_PER_BLOCK), np.float32),
                       flags=np.zeros((n, VOXELS_PER_BLOCK), np.uint8),
                       parent=np.zeros((n, VOXELS_PER_BLOCK, 3), np.int8),
                       updates=lib().orc_esdf_updates(h))
            if n:
                lib().orc_esdf_download(h, _ptr(out["idx"]), _ptr(out["distance"]),
                                        _ptr(out["flags"]), _ptr(out["parent"]))
            if free_min_distance is not None:
                m = lib().orc_esdf_free_points(h, float(free_min_distance), None, 0)
                pts = np.zeros((m, 4), np.float32)
                if m:
                    lib().orc_esdf_free_points(h, float(free_min_distance), _ptr(pts), m)
                out["free_points"] = pts
        finally:
            lib().orc_esdf_destroy(h)
        return out

    def interp(self, pos, interpolate=True):
        p = _f32(pos, (3,))
        d, w = C.c_float(0), C.c_float(0)
        rgba = np.zeros(4, np.uint8)
        ok = lib().orc_interp_voxel(self._h, _ptr(p), int(interpolate), C.byref(d), C.byref(w),
                                    _ptr(rgba))
        return bool(ok), d.value, w.value, rgba


def connect_mesh(vertices):
    """voxblox::createConnectedMesh on a flat triangle list -> (indices u32 [V], first_old u32 [U]:
    the old index of every unique vertex, in order of first occurrence)."""
    v = _f32(vertices, (-1, 3))
    idx = np.zeros(len(v), np.uint32)
    first = np.zeros(len(v), np.uint32)
    u = lib().orc_connect_mesh(_ptr(v), len(v), _ptr(idx), _ptr(first)) if len(v) else 0
    return idx, first[:u].copy()


def triangle_table():
    """kTriangleTable as an int array [256, 16]."""
    return np.ctypeslib.as_array(lib().orc_triangle_table(), shape=(256, 16)).copy()


def transform_point(T, p):
    out = np.zeros(3, np.float32)
    lib().orc_transform_point(_ptr(_f32(T, (7,))), _ptr(_f32(p, (3,))), _ptr(out))
    return out


def inverse_transform(T):
    out = np.zeros(7, np.float32)
    lib().orc_inverse_transform(_ptr(_f32(T, (7,))), _ptr(out))
    return out


def cast_ray(origin, point_G, clearing, carving, max_ray, voxel_size_inv, trunc,
             cast_from_origin=True, cap=100000):
    out = np.zeros((cap, 3), np.int64)
    n = lib().orc_cast_ray(_ptr(_f32(origin, (3,))), _ptr(_f32(point_G, (3,))), int(clearing),
                           int(carving), float(max_ray), float(voxel_size_inv), float(trunc),
                           int(cast_from_origin), _ptr(out), cap)
    return out[: min(n, cap)].copy()


class _Mesh(C.Structure):  # orc_mesh
    _fields_ = [("num_blocks", C.c_size_t), ("block_index", C.c_void_p),
                ("block_has_history", C.c_void_p), ("vertex_begin", C.c_void_p),
                ("x", C.c_void_p), ("y", C.c_void_p), ("z", C.c_void_p),
                ("r", C.c_void_p), ("g", C.c_void_p), ("b", C.c_void_p),
                ("hist_begin", C.c_void_p), ("hist", C.c_void_p),
                ("block_edge_length", C.c_float)]


def mesh_to_frames(mesh, interpolate_voxel_size, poses, stamps_sec):
    """MeshConverter::convertToPointCloud + getNextPointcloud per pose (mesh_converter.h:74-209).
    mesh: dict of numpy arrays (see coxgraph_b200.capi.make_mesh for the keys).
    -> (frame_offsets u64 [F+1], points_C f32 [N,3], colors u8 [N,4])."""
    spec = [("block_index", np.int32), ("block_has_history", np.uint8), ("vertex_begin", np.uint32),
            ("x", np.uint16), ("y", np.uint16), ("z", np.uint16), ("r", np.uint8), ("g", np.uint8),
            ("b", np.uint8), ("hist_begin", np.uint32), ("hist", np.uint32)]
    keep, m = [], _Mesh()
    for name, dt in spec:
        a = np.ascontiguousarray(mesh[name], dt)
        keep.append(a)
        setattr(m, name, a.ctypes.data)
    m.num_blocks = len(keep[1])
    m.block_edge_length = float(mesh["block_edge_length"])
    P = np.ascontiguousarray(poses, np.float32).reshape(-1, 7)
    st = np.ascontiguousarray(stamps_sec, np.float64).reshape(-1)
    offs = np.zeros(len(P) + 1, np.uint64)
    n = lib().orc_mesh_to_frames(C.byref(m), float(interpolate_voxel_size), len(P), P.ctypes.data,
                                 st.ctypes.data, offs.ctypes.data, None, None, 0)
    pts, cols = np.zeros((n, 3), np.float32), np.zeros((n, 4), np.uint8)
    if n:
        lib().orc_mesh_to_frames(C.byref(m), float(interpolate_voxel_size), len(P), P.ctypes.data,
                                 st.ctypes.data, offs.ctypes.data, pts.ctypes.data, cols.ctypes.data, n)
    return offs, pts, cols
