"""ctypes binding of the C ABI in include/coxgraph_b200.h.

The shared library is the product; this file only declares its symbols.  There is no Python or
CPU fallback: if the library is missing (not built) importing fails loudly, and if no CUDA
device is present `cg_context_create` fails with CG_ERR_CUDA.
"""
import ctypes as C
import os

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, "lib", "libcoxgraph_b200.so")

CG_OK = 0
CG_ERR_INVALID_ARG = -1
CG_ERR_CUDA = -2
CG_ERR_POOL_FULL = -3
CG_ERR_OUT_OF_RANGE = -4
CG_ERR_UNSUPPORTED = -5

METHOD_SIMPLE, METHOD_MERGED, METHOD_FAST = 0, 1, 2
ORDER_MIXED, ORDER_NATURAL = 0, 1

VOXELS_PER_BLOCK = 4096
BLOCK_BYTES = 49152
PACKED_BLOCK_BYTES = 16 + BLOCK_BYTES


class IntegratorConfig(C.Structure):
    """cg_integrator_config == voxblox::TsdfIntegratorBase::Config."""

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


class IntegrateStats(C.Structure):
    _fields_ = [("points_in", C.c_uint64), ("rays", C.c_uint64), ("voxel_updates", C.c_uint64),
                ("general_updates", C.c_uint64), ("blocks_touched", C.c_uint64), ("blocks_allocated", C.c_uint64),
                ("points_beyond_reach", C.c_uint64)]


DEPTH_16UC1, DEPTH_32FC1 = 0, 1
COLOR_RGB8, COLOR_RGBA8, COLOR_BGR8, COLOR_BGRA8, COLOR_MONO8 = 0, 1, 2, 3, 4
# sensor_msgs/Image encodings -> cg_depth_encoding / cg_color_encoding
DEPTH_ENCODINGS = {"16UC1": DEPTH_16UC1, "mono16": DEPTH_16UC1, "32FC1": DEPTH_32FC1}
COLOR_ENCODINGS = {"rgb8": COLOR_RGB8, "rgba8": COLOR_RGBA8, "bgr8": COLOR_BGR8, "bgra8": COLOR_BGRA8,
                   "mono8": COLOR_MONO8}
COLOR_PIXEL_BYTES = {COLOR_RGB8: 3, COLOR_RGBA8: 4, COLOR_BGR8: 3, COLOR_BGRA8: 4, COLOR_MONO8: 1}


class DepthCamera(C.Structure):
    """cg_depth_camera: CameraInfo intrinsics as image_geometry::PinholeCameraModel reports them
    (fx = P[0], fy = P[5], cx = P[2], cy = P[6]) and the encodings of the two images."""

    _fields_ = [("width", C.c_int32), ("height", C.c_int32), ("fx", C.c_double),
                ("fy", C.c_double), ("cx", C.c_double), ("cy", C.c_double),
                ("depth_encoding", C.c_int32), ("color_encoding", C.c_int32)]


class Mesh(C.Structure):
    """cg_mesh: voxblox_msgs/Mesh (with observation history) flattened into plain arrays."""

    _fields_ = [("num_blocks", C.c_size_t), ("block_index", C.c_void_p),
                ("block_has_history", C.c_void_p), ("vertex_begin", C.c_void_p),
                ("x", C.c_void_p), ("y", C.c_void_p), ("z", C.c_void_p),
                ("r", C.c_void_p), ("g", C.c_void_p), ("b", C.c_void_p),
                ("hist_begin", C.c_void_p), ("hist", C.c_void_p),
                ("block_edge_length", C.c_float)]


def make_mesh(mesh):
    """dict of numpy arrays -> (Mesh struct, keep-alive list).  Keys: block_index [B,3] i32,
    block_has_history [B] u8, vertex_begin [B+1] u32, x/y/z [V] u16, r/g/b [V] u8,
    hist_begin [V/3+1] u32, hist [H] u32, block_edge_length."""
    import numpy as np
    spec = [("block_index", np.int32), ("block_has_history", np.uint8), ("vertex_begin", np.uint32),
            ("x", np.uint16), ("y", np.uint16), ("z", np.uint16), ("r", np.uint8), ("g", np.uint8),
            ("b", np.uint8), ("hist_begin", np.uint32), ("hist", np.uint32)]
    keep, m = [], Mesh()
    for name, dt in spec:
        a = np.ascontiguousarray(mesh[name], dt)
        keep.append(a)
        setattr(m, name, a.ctypes.data)
    m.num_blocks = len(keep[1])
    m.block_edge_length = float(mesh["block_edge_length"])
    return m, keep


class StageProfile(C.Structure):
    _fields_ = [("name", C.c_char * 32), ("ms", C.c_double), ("launches", C.c_uint64)]


class HashStats(C.Structure):
    _fields_ = [("num_blocks", C.c_uint64), ("max_blocks", C.c_uint64),
                ("hash_capacity", C.c_uint64), ("load_factor", C.c_double),
                ("mean_probe_length", C.c_double), ("max_probe_length", C.c_uint64)]


class MergeStats(C.Structure):
    _fields_ = [("blocks_in", C.c_uint64), ("blocks_candidate", C.c_uint64),
                ("blocks_out", C.c_uint64)]


class ReprojectStats(C.Structure):
    _fields_ = [("submaps_moved", C.c_uint64), ("blocks_dirty", C.c_uint64),
                ("candidates", C.c_uint64), ("blocks_folded", C.c_uint64),
                ("blocks_removed", C.c_uint64), ("full_rebuild", C.c_uint64)]


class EsdfConfig(C.Structure):
    """cg_esdf_config == voxblox::EsdfIntegrator::Config."""

    _fields_ = [("max_distance_m", C.c_float), ("default_distance_m", C.c_float),
                ("min_distance_m", C.c_float), ("min_diff_m", C.c_float), ("min_weight", C.c_float),
                ("num_buckets", C.c_int32), ("multi_queue", C.c_int32),
                ("add_occupied_crust", C.c_int32), ("full_euclidean_distance", C.c_int32)]


class EsdfStats(C.Structure):
    _fields_ = [("blocks", C.c_uint64), ("observed_voxels", C.c_uint64),
                ("fixed_voxels", C.c_uint64), ("sweeps", C.c_uint64), ("block_passes", C.c_uint64)]


class EsdfUpdateStats(C.Structure):
    _fields_ = [("blocks_changed", C.c_uint64), ("blocks_removed", C.c_uint64),
                ("blocks_region", C.c_uint64), ("full_rebuild", C.c_int32), ("reserved", C.c_int32)]


# every symbol include/coxgraph_b200.h declares: name -> (restype, argtypes)
_P = C.c_void_p
SYMBOLS = {
    "cg_last_error": (C.c_char_p, []),
    "cg_version": (C.c_char_p, []),
    "cg_context_create": (C.c_int32, [C.c_int32, _P, C.POINTER(_P)]),
    "cg_context_destroy": (C.c_int32, [_P]),
    "cg_context_synchronize": (C.c_int32, [_P]),
    "cg_context_wait_stream": (C.c_int32, [_P, _P]),
    "cg_context_set_profiling": (C.c_int32, [_P, C.c_int32]),
    "cg_context_get_profile": (C.c_int32, [_P, _P, C.c_size_t, C.POINTER(C.c_size_t)]),
    "cg_context_reset_profile": (C.c_int32, [_P]),
    "cg_context_kernel_launches": (C.c_uint64, [_P]),
    "cg_layer_create": (C.c_int32, [_P, C.c_float, C.c_int32, C.c_size_t, C.POINTER(_P)]),
    "cg_layer_destroy": (C.c_int32, [_P]),
    "cg_layer_clear": (C.c_int32, [_P]),
    "cg_layer_remove_blocks": (C.c_int32, [_P, C.c_size_t, _P, C.POINTER(C.c_uint64)]),
    "cg_layer_num_blocks": (C.c_int64, [_P]),
    "cg_layer_voxel_size": (C.c_float, [_P]),
    "cg_layer_download": (C.c_int32, [_P, C.c_size_t, _P, _P, _P, C.POINTER(C.c_size_t)]),
    "cg_layer_download_updated": (C.c_int32, [_P, C.c_size_t, _P, _P, _P, C.POINTER(C.c_size_t)]),
    "cg_layer_download_blocks": (C.c_int32, [_P, C.c_size_t, _P, _P, _P, _P]),
    "cg_layer_hash_stats": (C.c_int32, [_P, C.POINTER(HashStats)]),
    "cg_layer_upload": (C.c_int32, [_P, C.c_size_t, _P, _P, _P]),
    "cg_layer_serialize": (C.c_int32, [_P, C.c_int32, C.c_size_t, _P, _P, C.POINTER(C.c_size_t)]),
    "cg_layer_reset_updated": (C.c_int32, [_P]),
    "cg_layer_deserialize": (C.c_int32, [_P, C.c_size_t, _P, _P]),
    "cg_layer_block_indices": (C.c_int32, [_P, C.c_size_t, _P, C.POINTER(C.c_size_t)]),
    "cg_integrator_config_default": (None, [C.POINTER(IntegratorConfig)]),
    "cg_integrate_pointcloud": (C.c_int32, [_P, C.POINTER(IntegratorConfig), _P, _P, _P,
                                            C.c_size_t, C.c_int32, C.POINTER(IntegrateStats)]),
    "cg_integrate_pointcloud_device": (C.c_int32, [_P, C.POINTER(IntegratorConfig), _P, _P, _P,
                                                   C.c_size_t, C.c_int32,
                                                   C.POINTER(IntegrateStats)]),
    "cg_integrate_batch": (C.c_int32, [_P, C.POINTER(IntegratorConfig), C.c_size_t, _P, _P, _P, _P,
                                       C.c_int32, C.POINTER(IntegrateStats)]),
    "cg_integrate_batch_device": (C.c_int32, [_P, C.POINTER(IntegratorConfig), C.c_size_t, _P, _P,
                                              _P, _P, C.c_int32, C.POINTER(IntegrateStats)]),
    "cg_stage_batch_async": (C.c_int32, [_P, C.c_int32, _P, _P, C.c_size_t]),
    "cg_integrate_batch_staged": (C.c_int32, [_P, C.POINTER(IntegratorConfig), C.c_size_t, _P,
                                              C.c_int32, _P, C.c_int32, C.POINTER(IntegrateStats)]),
    "cg_prepare_batch_device": (C.c_int32, [_P, C.POINTER(IntegratorConfig), C.c_size_t, _P, _P, _P,
                                            _P, C.c_int32, C.c_int32]),
    "cg_prepare_batch_staged": (C.c_int32, [_P, C.POINTER(IntegratorConfig), C.c_size_t, _P,
                                            C.c_int32, _P, C.c_int32, C.c_int32]),
    "cg_integrate_prepared": (C.c_int32, [_P, C.c_int32, C.POINTER(IntegrateStats)]),
    "cg_integrate_depth_batch": (C.c_int32, [_P, C.POINTER(IntegratorConfig), C.c_size_t, _P,
                                             C.POINTER(DepthCamera), _P, _P,
                                             C.POINTER(IntegrateStats)]),
    "cg_integrate_depth_batch_device": (C.c_int32, [_P, C.POINTER(IntegratorConfig), C.c_size_t, _P,
                                                    C.POINTER(DepthCamera), _P, _P,
                                                    C.POINTER(IntegrateStats)]),
    "cg_stage_depth_async": (C.c_int32, [_P, C.c_int32, C.POINTER(DepthCamera), C.c_size_t, _P, _P]),
    "cg_integrate_depth_staged": (C.c_int32, [_P, C.POINTER(IntegratorConfig), C.c_size_t, _P,
                                              C.POINTER(DepthCamera), C.c_int32,
                                              C.POINTER(IntegrateStats)]),
    "cg_prepare_depth_device": (C.c_int32, [_P, C.POINTER(IntegratorConfig), C.c_size_t, _P,
                                            C.POINTER(DepthCamera), _P, _P, C.c_int32]),
    "cg_prepare_depth_staged": (C.c_int32, [_P, C.POINTER(IntegratorConfig), C.c_size_t, _P,
                                            C.POINTER(DepthCamera), C.c_int32, C.c_int32]),
    "cg_mesh_to_frames": (C.c_int32, [_P, C.POINTER(Mesh), C.c_float, C.c_size_t, _P, _P, _P, _P, _P,
                                      C.c_size_t]),
    "cg_recover_mesh": (C.c_int32, [_P, C.POINTER(IntegratorConfig), C.POINTER(Mesh), C.c_float,
                                    C.c_size_t, _P, _P, C.POINTER(IntegrateStats)]),
    "cg_merge_layer_into_layer": (C.c_int32, [_P, _P, _P, C.POINTER(MergeStats)]),
    "cg_project_submaps": (C.c_int32, [_P, _P, C.c_size_t, _P, C.POINTER(MergeStats)]),
    "cg_layer_mesh": (C.c_int32, [_P, C.c_float, C.c_int32, C.c_int32, C.c_size_t, C.c_size_t, _P, _P,
                                  _P, _P, _P, C.POINTER(C.c_size_t), C.POINTER(C.c_size_t)]),
    "cg_mesh_fetch": (C.c_int32, [_P, C.c_size_t, C.c_size_t, _P, _P, _P, _P, _P]),
    "cg_mesh_connect": (C.c_int32, [_P, C.c_size_t, C.c_size_t, _P, _P, _P, _P,
                                    C.POINTER(C.c_size_t), C.POINTER(C.c_size_t)]),
    "cg_esdf_config_default": (None, [C.POINTER(EsdfConfig)]),
    "cg_layer_esdf_batch": (C.c_int32, [_P, C.POINTER(EsdfConfig), C.POINTER(EsdfStats)]),
    "cg_layer_esdf_update": (C.c_int32, [_P, C.POINTER(EsdfConfig), C.POINTER(EsdfStats),
                                         C.POINTER(EsdfUpdateStats)]),
    "cg_esdf_fetch": (C.c_int32, [_P, C.c_size_t, _P, _P, _P, C.POINTER(C.c_size_t)]),
    "cg_esdf_free_points": (C.c_int32, [_P, C.c_float, C.c_size_t, _P, C.POINTER(C.c_size_t)]),
    "cg_reproject_submaps": (C.c_int32, [_P, _P, _P, C.c_size_t, C.c_float, C.c_float, _P, _P,
                                         C.POINTER(ReprojectStats)]),
    "cg_block_owner": (C.c_int32, [C.c_int32, C.c_int32, C.c_int32, C.c_int32]),
    "cg_layer_pack_by_owner": (C.c_int32, [_P, C.c_int32, _P, C.c_size_t, _P]),
    "cg_layer_merge_packed": (C.c_int32, [_P, _P, C.c_size_t]),
    "cg_comm_get_unique_id": (C.c_int32, [_P]),
    "cg_comm_init": (C.c_int32, [_P, _P, C.c_int32, C.c_int32]),
    "cg_comm_destroy": (C.c_int32, [_P]),
    "cg_gather_global": (C.c_int32, [_P, _P, C.POINTER(C.c_uint64)]),
    "cg_project_submaps_sharded": (C.c_int32, [_P, _P, C.c_size_t, _P, _P, C.POINTER(MergeStats)]),
    "cg_layer_mesh_sharded": (C.c_int32, [_P, C.c_float, C.c_int32, C.c_int32, C.c_size_t, C.c_size_t,
                                          _P, _P, _P, _P, _P, C.POINTER(C.c_size_t),
                                          C.POINTER(C.c_size_t)]),
    "cg_comm_peer_mappings": (C.c_int32, [_P, C.POINTER(C.c_uint64), C.POINTER(C.c_uint64)]),
    "cg_debug_selftest": (C.c_int32, [_P, C.c_int32, C.c_uint64, C.POINTER(C.c_uint64)]),
}

_lib = None


def load():
    """Load libcoxgraph_b200.so; raise if it has not been built (no fallback)."""
    global _lib
    if _lib is None:
        if not os.path.exists(LIB_PATH):
            raise RuntimeError(
                f"{LIB_PATH} is missing: build it with `make` or __graft_entry__.build(). "
                "coxgraph_b200 has no CPU/Python fallback.")
        lib = C.CDLL(LIB_PATH)
        for name, (res, args) in SYMBOLS.items():
            fn = getattr(lib, name)  # AttributeError if the symbol is not exported
            fn.restype = res
            fn.argtypes = args
        _lib = lib
    return _lib


class CgError(RuntimeError):
    def __init__(self, status, message):
        super().__init__(f"coxgraph_b200 error {status}: {message}")
        self.status = status


def check(status):
    if status != CG_OK:
        raise CgError(status, load().cg_last_error().decode("utf-8", "replace"))
