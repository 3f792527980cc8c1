/*
 * coxgraph_b200.h — C ABI of the B200-native TSDF fusion engine for coxgraph's hot path.
 *
 * This is the drop-in boundary: a plain `extern "C"` shared library (libcoxgraph_b200.so),
 * opaque handles, POD structs, plain pointers and sizes.  No torch, STL or exceptions cross
 * it.  Every entry point names the reference interface it replaces (paths are relative to
 * the reference checkout, mfkiwl/coxgraph).  The arithmetic itself lives in the reference's
 * un-vendored dependency voxblox ([EXT], see DESIGN.md); the file:line given is the
 * reference's own call site of that interface.
 *
 * Conventions
 *  - status: 0 = CG_OK, negative = error; cg_last_error() returns a thread-local message.
 *  - transforms: float[7] = {qw, qx, qy, qz, tx, ty, tz} (kindr::minimal::QuatTransformation,
 *    unit quaternion); points: float xyz triples; colours: uint8 r,g,b,a quadruples.
 *  - host pointers are caller-owned, may be pageable, and are only read during the call.
 *    `*_device` variants take pointers to device memory on the context's GPU.
 *  - calls return after the work has completed on the GPU unless stated otherwise.
 *  - handles are thread-compatible, not thread-safe (the reference drives this path from a
 *    single-threaded ros::spin(), coxgraph/src/tsdf_recover_node.cpp:23).
 *  - there is NO CPU fallback: without a CUDA device every compute call fails with
 *    CG_ERR_CUDA.
 */
#ifndef COXGRAPH_B200_H_
#define COXGRAPH_B200_H_

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define CG_VOXELS_PER_SIDE 16
#define CG_VOXELS_PER_BLOCK 4096
#define CG_VOXEL_BYTES 12
#define CG_BLOCK_BYTES (CG_VOXELS_PER_BLOCK * CG_VOXEL_BYTES) /* 49152 */

enum cg_status {
  CG_OK = 0,
  CG_ERR_INVALID_ARG = -1,
  CG_ERR_CUDA = -2,         /* CUDA runtime error (no device, OOM, launch failure) */
  CG_ERR_POOL_FULL = -3,    /* block pool exhausted (max_blocks of cg_layer_create) */
  CG_ERR_OUT_OF_RANGE = -4, /* a voxel index left the +-2^19 voxel addressable range */
  CG_ERR_UNSUPPORTED = -5   /* e.g. method FAST (order-dependent, see DESIGN.md) */
};

enum cg_method { CG_METHOD_SIMPLE = 0, CG_METHOD_MERGED = 1, CG_METHOD_FAST = 2 };
enum cg_order_mode { CG_ORDER_MIXED = 0, CG_ORDER_NATURAL = 1 };

/* The voxel record handed across the boundary: voxblox::TsdfVoxel
 * (consumed by the reference at coxgraph/include/coxgraph/utils/msg_converter.h:49-50 and
 * coxgraph/src/client/map_server.cpp:88-89 through serializeLayerAsMsg). */
typedef struct cg_tsdf_voxel {
  float distance;
  float weight;
  uint8_t r, g, b, a;
} cg_tsdf_voxel;

/* voxblox::TsdfIntegratorBase::Config — the parameter set the reference loads from
 * coxgraph/config/tsdf_server_*.yaml and coxgraph/config/tsdf_recover.yaml:2-11.
 * cg_integrator_config_default() fills the upstream defaults. */
typedef struct cg_integrator_config {
  float default_truncation_distance; /* truncation_distance */
  float max_weight;
  int32_t voxel_carving_enabled;
  float min_ray_length_m;
  float max_ray_length_m;
  int32_t use_const_weight;
  int32_t allow_clear;
  int32_t use_weight_dropoff;
  int32_t use_sparsity_compensation_factor;
  float sparsity_compensation_factor;
  int32_t enable_anti_grazing;
  int32_t method;                 /* cg_method; `method:` in the yaml files */
  int32_t integration_order_mode; /* cg_order_mode */
  float start_voxel_subsampling_factor;   /* FAST only */
  int32_t max_consecutive_ray_collisions; /* FAST only */
} cg_integrator_config;

typedef struct cg_context cg_context;
typedef struct cg_layer cg_layer;

/* Per-call statistics (the byte model of DESIGN.md / SURVEY.md §8d uses these). */
typedef struct cg_integrate_stats {
  uint64_t points_in;       /* N */
  uint64_t rays;            /* rays cast (bundles for MERGED) */
  uint64_t voxel_updates;   /* (ray, voxel) visits */
  uint64_t general_updates; /* visits replayed in order (voxels inside the truncation band) */
  uint64_t blocks_touched;  /* distinct blocks visited by any ray of the call */
  uint64_t blocks_allocated;/* new blocks */
  uint64_t points_beyond_reach; /* valid points more than 8191 voxels from the sensor (MERGED):
                                   dropped — the reference would integrate them as clearing rays
                                   cut at max_ray_length_m */
} cg_integrate_stats;

typedef struct cg_merge_stats {
  uint64_t blocks_in;        /* allocated blocks of the source layer(s) */
  uint64_t blocks_candidate; /* output blocks marked by the forward pass */
  uint64_t blocks_out;       /* output blocks that received data */
} cg_merge_stats;

const char* cg_last_error(void);
const char* cg_version(void);

/* --- context: one per GPU / per process rank --------------------------------------- */
/* `stream` is a cudaStream_t passed as void* (NULL = a stream owned by the context). */
int32_t cg_context_create(int32_t device, void* stream, cg_context** out);
int32_t cg_context_destroy(cg_context* ctx);
int32_t cg_context_synchronize(cg_context* ctx);
/* Orders the context's stream behind everything queued so far on `producer_stream` (a
 * cudaStream_t as void*; NULL = the legacy default stream).  The `*_device` entry points read the
 * caller's device buffers on the context's stream: call this first when another stream produced
 * them (no-op when it is the context's own stream). */
int32_t cg_context_wait_stream(cg_context* ctx, void* producer_stream);

/* Named stage timers (CUDA events on the context's stream) and launch counters — the
 * counterpart of the voxblox::timing::Timer scopes the reference wraps around this path
 * (coxgraph/include/coxgraph/map_comm/tsdf_recover.h:63,74-76,93). */
typedef struct cg_stage_profile {
  char name[32];
  double ms;         /* accumulated device time of the stage while profiling was enabled */
  uint64_t launches; /* kernels of this library launched in the stage (always counted) */
} cg_stage_profile;
int32_t cg_context_set_profiling(cg_context* ctx, int32_t enable);
int32_t cg_context_get_profile(cg_context* ctx, cg_stage_profile* out, size_t capacity,
                               size_t* num_out);
int32_t cg_context_reset_profile(cg_context* ctx);
/* Total number of this library's own kernels launched so far on the context. */
uint64_t cg_context_kernel_launches(const cg_context* ctx);

/* --- layer: replaces voxblox::Layer<TsdfVoxel> (block hash map keyed by BlockIndex) --- */
/* voxels_per_side must be 16 (the reference never overrides tsdf_voxels_per_side). */
int32_t cg_layer_create(cg_context* ctx, float voxel_size, int32_t voxels_per_side,
                        size_t max_blocks, cg_layer** out);
int32_t cg_layer_destroy(cg_layer* layer);
/* Layer::removeAllBlocks — coxgraph/include/coxgraph/map_comm/tsdf_recover.h:62,
 * coxgraph/src/client/map_server.cpp:65 */
int32_t cg_layer_clear(cg_layer* layer);
/* Layer::removeBlock for each listed block index (absent ones are ignored); *removed_out
 * (optional) = blocks actually removed.  The pool is compacted and the hash rebuilt. */
int32_t cg_layer_remove_blocks(cg_layer* layer, size_t num_blocks, const int32_t* block_idx_xyz,
                               uint64_t* removed_out);
/* Layer::getNumberOfAllocatedBlocks */
int64_t cg_layer_num_blocks(const cg_layer* layer);
float cg_layer_voxel_size(const cg_layer* layer);

/* Copy the layer out in voxblox's own layout: blocks sorted by (z, y, x) block index,
 * block_idx_xyz int32[B*3], voxels cg_tsdf_voxel[B*4096] (linear x + 16*(y + 16*z)),
 * flags uint8[B] (bit0 has_data, bit1 updated).  Any output may be NULL.  `capacity_blocks`
 * bounds B.  This is what serializeLayerAsMsg consumes
 * (coxgraph/include/coxgraph/map_comm/tsdf_recover.h:95). */
int32_t cg_layer_download(const cg_layer* layer, size_t capacity_blocks, int32_t* block_idx_xyz,
                          cg_tsdf_voxel* voxels, uint8_t* flags, size_t* num_blocks_out);
/* Only the blocks whose `updated` flag is set (Layer::getAllUpdatedBlocks), in (z, y, x) order —
 * what a consumer that keeps a host copy of the layer needs after integratePointCloud calls
 * (the adapter's syncLayerToHost, INTEGRATION.md §1); clear the flags with cg_layer_reset_updated.
 * Call with NULL arrays for the count. */
int32_t cg_layer_download_updated(const cg_layer* layer, size_t capacity_blocks,
                                  int32_t* block_idx_xyz, cg_tsdf_voxel* voxels, uint8_t* flags,
                                  size_t* num_blocks_out);
/* The listed blocks only (Layer::getBlockPtrByIndex for each index), in the order given:
 * voxels cg_tsdf_voxel[n*4096], flags uint8[n] (either may be NULL), found uint8[n] = 1 where the
 * block is allocated (the other outputs of a missing block are unspecified).  For layers too
 * large to copy out whole (config C4: ~2 M blocks = 98 GB) and for incremental consumers. */
int32_t cg_layer_download_blocks(const cg_layer* layer, size_t num_blocks,
                                 const int32_t* block_idx_xyz, cg_tsdf_voxel* voxels,
                                 uint8_t* flags, uint8_t* found);
/* Occupancy of the block hash (AnyIndexHash replacement): probe length = table entries visited
 * to find an allocated block, measured over all allocated blocks. */
typedef struct cg_hash_stats {
  uint64_t num_blocks;
  uint64_t max_blocks;
  uint64_t hash_capacity;
  double load_factor;
  double mean_probe_length;
  uint64_t max_probe_length;
} cg_hash_stats;
int32_t cg_layer_hash_stats(const cg_layer* layer, cg_hash_stats* out);
/* Insert / overwrite blocks (deserializeMsgToLayer hand-off,
 * coxgraph/include/coxgraph/utils/msg_converter.h:107-109). flags may be NULL (has_data). */
int32_t cg_layer_upload(cg_layer* layer, size_t num_blocks, const int32_t* block_idx_xyz,
                        const cg_tsdf_voxel* voxels, const uint8_t* flags);
/* The block payload of voxblox_msgs/Layer, produced / consumed on the device
 * (voxblox::serializeLayerAsMsg / deserializeMsgToLayer = Block::serializeToIntegers per block;
 * reference call sites coxgraph/include/coxgraph/utils/msg_converter.h:49-50 and :107-109,
 * coxgraph/src/client/map_server.cpp:88-89, coxgraph/include/coxgraph/map_comm/tsdf_recover.h:95).
 * Per block: x/y/z index (block_idx_xyz, int32[3]) and data = 4096 x 3 uint32 words {float bits
 * of distance, float bits of weight, colour a | b<<8 | g<<16 | r<<24}, blocks in (z, y, x) order.
 * only_updated != 0 keeps the blocks whose `updated` flag is set (serializeLayerAsMsg's
 * only_updated / getAllUpdatedBlocks).  Call with data == NULL to get the block count. */
int32_t cg_layer_serialize(const cg_layer* layer, int32_t only_updated, size_t capacity_blocks,
                           int32_t* block_idx_xyz, uint32_t* data, size_t* num_blocks_out);
/* Block::updated().reset() for every block (what a publisher does after sending the updated
 * blocks). */
int32_t cg_layer_reset_updated(cg_layer* layer);
/* Blocks are created or overwritten and marked has_data + updated (deserializeMsgToLayer with
 * action kUpdate; call cg_layer_clear first for kReset). */
int32_t cg_layer_deserialize(cg_layer* layer, size_t num_blocks, const int32_t* block_idx_xyz,
                             const uint32_t* data);
/* Block indices only (sorted), e.g. to compare allocation sets. */
int32_t cg_layer_block_indices(const cg_layer* layer, size_t capacity_blocks,
                               int32_t* block_idx_xyz, size_t* num_blocks_out);

/* --- integration: replaces voxblox::TsdfIntegratorBase::integratePointCloud(T_G_C,
 * points_C, colors, freespace_points) — called by the reference at
 * coxgraph/include/coxgraph/map_comm/tsdf_recover.h:75 and by voxblox_ros TsdfServer
 * (coxgraph/launch/firefly/tsdf_client.launch:24). */
void cg_integrator_config_default(cg_integrator_config* cfg);
int32_t cg_integrate_pointcloud(cg_layer* layer, const cg_integrator_config* cfg,
                                const float T_G_C[7], const float* points_xyz,
                                const uint8_t* colors_rgba, size_t num_points,
                                int32_t freespace_points, cg_integrate_stats* stats);
int32_t cg_integrate_pointcloud_device(cg_layer* layer, const cg_integrator_config* cfg,
                                       const float T_G_C[7], const float* d_points_xyz,
                                       const uint8_t* d_colors_rgba, size_t num_points,
                                       int32_t freespace_points, cg_integrate_stats* stats);
/* F consecutive integratePointCloud calls (the loop of tsdf_recover.h:71-86) submitted as
 * one job; identical result to F single calls in order.  frame_offsets has F+1 entries
 * (points of frame f are [frame_offsets[f], frame_offsets[f+1])); poses is F*7 floats. */
int32_t cg_integrate_batch(cg_layer* layer, const cg_integrator_config* cfg, size_t num_frames,
                           const float* T_G_C_poses, const float* points_xyz,
                           const uint8_t* colors_rgba, const uint64_t* frame_offsets,
                           int32_t freespace_points, cg_integrate_stats* stats);
int32_t cg_integrate_batch_device(cg_layer* layer, const cg_integrator_config* cfg,
                                  size_t num_frames, const float* T_G_C_poses,
                                  const float* d_points_xyz, const uint8_t* d_colors_rgba,
                                  const uint64_t* frame_offsets, int32_t freespace_points,
                                  cg_integrate_stats* stats);

/* Double-buffered input staging (slot 0 or 1): cg_stage_batch_async queues the host->device copy
 * of a later job's points / colours on the context's copy stream and returns at once (pinned host
 * memory; it must stay valid until the matching cg_integrate_batch_staged returns), so the
 * transfer of job k+1 overlaps the fusion of job k — the counterpart of the ROS subscriber queue
 * that holds the next PointCloud2 while the current one is integrated
 * (coxgraph/launch/firefly/tsdf_client.launch:24, voxblox_ros TsdfServer).  frame_offsets must
 * start at 0 and end at the staged point count. */
int32_t cg_stage_batch_async(cg_context* ctx, int32_t slot, const float* points_xyz,
                             const uint8_t* colors_rgba, size_t num_points);
int32_t cg_integrate_batch_staged(cg_layer* layer, const cg_integrator_config* cfg,
                                  size_t num_frames, const float* T_G_C_poses, int32_t slot,
                                  const uint64_t* frame_offsets, int32_t freespace_points,
                                  cg_integrate_stats* stats);

/* Pipelined jobs.  The first half of a job — validity, T_G_C * p, bundling, one ray per bundle —
 * never touches the layer, so it can run while the previous job is still being fused:
 * cg_prepare_batch_device / _staged queue that half of a LATER job on the context's second stream
 * (own scratch set per slot, 0 or 1) and return at once; cg_integrate_prepared(layer, slot) then
 * runs the rest on the context's stream and returns when the job is complete, with the same
 * result as cg_integrate_batch_device.  The counterpart, one level up, of the ROS subscriber queue
 * that already holds the next clouds (tsdf_recover.h:71-86 knows every frame of the mesh in
 * advance).  The input buffers (device memory, or the staged slot) must stay valid and unchanged
 * until cg_integrate_prepared has returned; a job the fast path cannot take (several groups, a
 * point outside the bundle-key box, an invalid config) is simply run the plain way there. */
int32_t cg_prepare_batch_device(cg_layer* layer, const cg_integrator_config* cfg,
                                size_t num_frames, const float* T_G_C_poses,
                                const float* d_points_xyz, const uint8_t* d_colors_rgba,
                                const uint64_t* frame_offsets, int32_t freespace_points,
                                int32_t slot);
int32_t cg_prepare_batch_staged(cg_layer* layer, const cg_integrator_config* cfg,
                                size_t num_frames, const float* T_G_C_poses, int32_t stage_slot,
                                const uint64_t* frame_offsets, int32_t freespace_points,
                                int32_t slot);
int32_t cg_integrate_prepared(cg_layer* layer, int32_t slot, cg_integrate_stats* stats);

/* --- integration of registered depth + colour images: replaces depth_image_proc
 * point_cloud_xyzrgb (depth_conversions.h convert<T>) followed by voxblox_ros TsdfServer's
 * insertion (convertPointcloud drops the points with a non-finite coordinate, then
 * integratePointCloud).  The result is bit-identical, stats included, to cg_integrate_batch_device
 * on that cloud: per pixel (u, v) in row-major order, a valid depth d (16UC1: d != 0, millimetres;
 * 32FC1: finite, metres) gives x = ((u - float(cx)) * d) * float(unit / fx), y likewise, z = d in
 * metres, colour (r, g, b, 255) from the encoding's byte offsets; invalid pixels and points with a
 * non-finite coordinate are dropped.  Lens distortion is ignored (as depth_image_proc does), the
 * colour image has the depth image's size and both are tightly packed.  stats.points_in counts
 * the kept points.  The entry points mirror the cloud family above one to one. */
enum cg_depth_encoding { CG_DEPTH_16UC1 = 0, CG_DEPTH_32FC1 = 1 };
enum cg_color_encoding {
  CG_COLOR_RGB8 = 0,  /* r, g, b offsets 0, 1, 2; 3 bytes a pixel */
  CG_COLOR_RGBA8 = 1, /* 0, 1, 2; 4 bytes */
  CG_COLOR_BGR8 = 2,  /* 2, 1, 0; 3 bytes */
  CG_COLOR_BGRA8 = 3, /* 2, 1, 0; 4 bytes */
  CG_COLOR_MONO8 = 4  /* 0, 0, 0; 1 byte */
};
/* sensor_msgs/CameraInfo as image_geometry::PinholeCameraModel reports it (fx = P[0], fy = P[5],
 * cx = P[2], cy = P[6]) plus the two image encodings. */
typedef struct cg_depth_camera {
  int32_t width, height;
  double fx, fy, cx, cy;
  int32_t depth_encoding; /* cg_depth_encoding */
  int32_t color_encoding; /* cg_color_encoding */
} cg_depth_camera;
/* F frames: depth [F][H][W] (uint16 or float), colour [F][H][W][pixel bytes]; host memory
 * (pageable or pinned) or, for _device, device memory on the context's GPU. */
int32_t cg_integrate_depth_batch(cg_layer* layer, const cg_integrator_config* cfg,
                                 size_t num_frames, const float* T_G_C_poses,
                                 const cg_depth_camera* camera, const void* depth,
                                 const uint8_t* color, cg_integrate_stats* stats);
int32_t cg_integrate_depth_batch_device(cg_layer* layer, const cg_integrator_config* cfg,
                                        size_t num_frames, const float* T_G_C_poses,
                                        const cg_depth_camera* camera, const void* d_depth,
                                        const uint8_t* d_color, cg_integrate_stats* stats);
/* Staging of images into slot 0 or 1 (pinned host memory; returns at once).  The slots are those
 * of cg_stage_batch_async: staging replaces what the slot held, and a slot that holds images is
 * only usable by the _depth_ calls (and one that holds a cloud only by the cloud calls);
 * otherwise CG_ERR_INVALID_ARG.  The camera and frame count must be those staged. */
int32_t cg_stage_depth_async(cg_context* ctx, int32_t slot, const cg_depth_camera* camera,
                             size_t num_frames, const void* depth, const uint8_t* color);
int32_t cg_integrate_depth_staged(cg_layer* layer, const cg_integrator_config* cfg,
                                  size_t num_frames, const float* T_G_C_poses,
                                  const cg_depth_camera* camera, int32_t slot,
                                  cg_integrate_stats* stats);
/* Pipelined depth jobs, completed by cg_integrate_prepared.  The unprojected points are kept in
 * the prepare slot, so a job the fast path cannot take runs the plain way from them. */
int32_t cg_prepare_depth_device(cg_layer* layer, const cg_integrator_config* cfg,
                                size_t num_frames, const float* T_G_C_poses,
                                const cg_depth_camera* camera, const void* d_depth,
                                const uint8_t* d_color, int32_t slot);
int32_t cg_prepare_depth_staged(cg_layer* layer, const cg_integrator_config* cfg,
                                size_t num_frames, const float* T_G_C_poses,
                                const cg_depth_camera* camera, int32_t stage_slot, int32_t slot);

/* --- mesh recovery: the recover node's front end (SURVEY §8f N3) ----------------------
 * voxblox_msgs/Mesh (the fork's "mesh with observation history") flattened into plain arrays:
 * block b owns vertices [vertex_begin[b], vertex_begin[b+1]) (triangles: multiples of 3), x/y/z
 * are the uint16 vertex offsets inside the block, r/g/b the vertex colours; triangle t (= vertex
 * index / 3) owns the entries [hist_begin[t], hist_begin[t+1]) of `hist`, read as (first stamp,
 * last stamp) pairs (voxblox_msgs/ObsHistory); block_has_history[b] = 0 means MeshBlock.history
 * was empty (the block is skipped, mesh_converter.h:87).  All pointers are host pointers. */
typedef struct cg_mesh {
  size_t num_blocks;
  const int32_t* block_index;        /* [B*3]  MeshBlock.index */
  const uint8_t* block_has_history;  /* [B] */
  const uint32_t* vertex_begin;      /* [B+1] */
  const uint16_t *x, *y, *z;         /* [V]    MeshBlock.x / y / z */
  const uint8_t *r, *g, *b;          /* [V]    MeshBlock.r / g / b */
  const uint32_t* hist_begin;        /* [V/3 + 1] */
  const uint32_t* hist;              /* (first, last) stamp pairs */
  float block_edge_length;           /* Mesh.block_edge_length */
} cg_mesh;
/* voxblox::MeshConverter::convertToPointCloud followed by getNextPointcloud for every trajectory
 * pose (coxgraph/include/coxgraph/map_comm/mesh_converter.h:74-172, :186-209, :211-265): the
 * point clouds, in the sensor frame, that TsdfRecover::processMesh integrates.  poses: F x 7,
 * stamps_sec: the trajectory's time stamps.  frame_offsets (F + 1) is always filled; points and
 * colours only when non-NULL and capacity_points suffices. */
int32_t cg_mesh_to_frames(cg_context* ctx, const cg_mesh* mesh, float interpolate_voxel_size,
                          size_t num_poses, const float* T_G_C_poses, const double* stamps_sec,
                          uint64_t* frame_offsets, float* points_xyz, uint8_t* colors_rgba,
                          size_t capacity_points);
/* TsdfRecover::processMesh without the ROS plumbing (coxgraph/include/coxgraph/map_comm/
 * tsdf_recover.h:59-99): removeAllBlocks, mesh -> per-pose clouds, integratePointCloud for every
 * pose with a non-empty cloud — all on the device; serialise the result with cg_layer_serialize
 * (:95). */
int32_t cg_recover_mesh(cg_layer* layer, const cg_integrator_config* cfg, const cg_mesh* mesh,
                        float interpolate_voxel_size, size_t num_poses, const float* T_G_C_poses,
                        const double* stamps_sec, cg_integrate_stats* stats);

/* --- merge: replaces voxblox::mergeLayerAintoLayerB(layer_A, T_B_A, layer_B) — called at
 * coxgraph/src/client/map_server.cpp:67-69 — and cblox SubmapCollection::getProjectedMap(),
 * the server's submap-to-global entry reached from
 * coxgraph/src/server/visualizer/server_visualizer.cpp:123-126. */
int32_t cg_merge_layer_into_layer(const cg_layer* layer_a, const float T_B_A[7],
                                  cg_layer* layer_b, cg_merge_stats* stats);
/* for s in 0..n-1: mergeLayerAintoLayerB(submaps[s], T_M_S[s], global), in that order. */
int32_t cg_project_submaps(const cg_layer* const* submaps, const float* T_M_S_poses,
                           size_t num_submaps, cg_layer* global_layer, cg_merge_stats* stats);

/* --- meshing on the device-resident layer (SURVEY.md §8f N4): replaces
 * voxblox::MeshIntegrator<TsdfVoxel>::generateMesh as run by
 * voxgraph::SubmapVisuals::saveAndPubCombinedMesh right after the merge
 * (coxgraph/src/server/visualizer/server_visualizer.cpp:123-126) and by generateSubmapMesh on the
 * client (coxgraph/src/client/map_server.cpp:126-130), so only triangles leave the GPU.
 * Blocks come in (z, y, x) order; block b owns vertices [vertex_begin[b], vertex_begin[b+1])
 * (num_blocks + 1 entries), in the reference's voxel loop order; three consecutive vertices are
 * one triangle (voxblox's per-block `indices` are 0..n-1), normals are per vertex, colours the
 * nearest voxel's (MeshIntegratorConfig: use_color, min_weight, default 1e-4).  With
 * only_updated, blocks whose `updated` flag is clear produce no vertices (clear the flags with
 * cg_layer_reset_updated).  Counts are always reported; host arrays (any may be NULL) are filled
 * when the capacities suffice, otherwise CG_ERR_INVALID_ARG.  The result also stays on the device
 * until the next cg_layer_mesh on the same context: call with NULL arrays to get the counts, then
 * cg_mesh_fetch to copy it out without meshing again. */
int32_t cg_layer_mesh(const cg_layer* layer, float min_weight, int32_t use_color,
                      int32_t only_updated, size_t capacity_blocks, size_t capacity_vertices,
                      int32_t* block_idx_xyz, uint32_t* vertex_begin, float* vertices_xyz,
                      float* normals_xyz, uint8_t* colors_rgba, size_t* num_blocks_out,
                      size_t* num_vertices_out);
int32_t cg_mesh_fetch(cg_context* ctx, size_t capacity_blocks, size_t capacity_vertices,
                      int32_t* block_idx_xyz, uint32_t* vertex_begin, float* vertices_xyz,
                      float* normals_xyz, uint8_t* colors_rgba);

/* MeshLayer::getConnectedMesh (voxblox::createConnectedMesh, [EXT] mesh/mesh_utils.h) of the mesh
 * the last cg_layer_mesh left in the context — the PLY step of saveAndPubCombinedMesh when a file
 * path is given (coxgraph/src/server/visualizer/server_visualizer.cpp:118-126 ->
 * io::outputMeshLayerAsPly).  Vertices that fall into the same cell of the 1e-10 m grid
 * (round(double(v) / double(1e-10f)) per axis) are merged into the first of them, block meshes
 * taken in (z, y, x) block order: vertices / normals / colours of the first occurrences in order
 * of first occurrence, indices[i] = new index of old vertex i (three per triangle).  Counts are
 * always reported; arrays (any may be NULL) are filled when the capacities suffice. */
int32_t cg_mesh_connect(cg_context* ctx, size_t capacity_vertices, size_t capacity_indices,
                        float* vertices_xyz, float* normals_xyz, uint8_t* colors_rgba,
                        uint32_t* indices, size_t* num_vertices_out, size_t* num_indices_out);

/* --- ESDF of the device-resident layer (SURVEY.md §8f N4, second half): replaces
 * voxblox::EsdfIntegrator::updateFromTsdfLayerBatch() as the client's MapServer runs it after the
 * merge (coxgraph/include/coxgraph/client/map_server.h:141-145, from
 * coxgraph/src/client/map_server.cpp:99) and voxblox::createFreePointcloudFromEsdfLayer
 * (coxgraph/src/client/map_server.cpp:112-113).  Mirrors voxblox::EsdfIntegrator::Config (upstream
 * defaults in comments; coxgraph/config/coxgraph_client.yaml:68-69 sets esdf_max/min_distance).
 * The ESDF gets one block per allocated TSDF block; a voxel with tsdf weight >= min_weight is
 * observed; |tsdf distance| < min_distance_m copies the distance and fixes the voxel; every other
 * observed voxel starts at +-default_distance_m and takes the quasi-Euclidean 26-neighbour
 * wavefront distance from voxels of equal sign with |distance| < max_distance_m (processOpenSet).
 * The device computes the FIXED POINT of that relaxation, i.e. upstream's result for
 * min_diff_m = 0 (unique, order-independent, bit-identical to a sequential run); with upstream's
 * min_diff_m > 0 the sequential queue may stop above it by less than min_diff_m per hop.
 * min_diff_m, num_buckets and multi_queue are therefore accepted and ignored;
 * full_euclidean_distance != 0 returns CG_ERR_UNSUPPORTED; default_distance_m must be >=
 * max_distance_m (what voxblox_ros' parameter loader enforces). */
typedef struct cg_esdf_config {
  float max_distance_m;             /* 2.0 */
  float default_distance_m;         /* 2.0 */
  float min_distance_m;             /* 0.2 */
  float min_diff_m;                 /* 0.001 (ignored: see above) */
  float min_weight;                 /* 1e-6 */
  int32_t num_buckets;              /* 20 (ignored) */
  int32_t multi_queue;              /* 0 (ignored) */
  int32_t add_occupied_crust;       /* 0 */
  int32_t full_euclidean_distance;  /* 0 */
} cg_esdf_config;
typedef struct cg_esdf_stats {
  uint64_t blocks;           /* ESDF blocks = allocated TSDF blocks */
  uint64_t observed_voxels;
  uint64_t fixed_voxels;
  uint64_t sweeps;           /* rounds over the dirty blocks until none was left */
  uint64_t block_passes;     /* blocks relaxed, summed over the sweeps */
} cg_esdf_stats;
void cg_esdf_config_default(cg_esdf_config* cfg);
/* Rebuilds the ESDF of `tsdf_layer` on the device; the result (8 bytes per voxel: 32 KB per block)
 * stays in the layer's context until the next call. */
int32_t cg_layer_esdf_batch(const cg_layer* tsdf_layer, const cg_esdf_config* cfg,
                            cg_esdf_stats* stats);
/* voxblox::EsdfIntegrator::updateFromTsdfLayer(), the incremental form: brings the ESDF retained in
 * the context up to date with `tsdf_layer`, re-solving only the blocks within reach of what
 * changed.  On return the retained ESDF is bit-identical to what cg_layer_esdf_batch(tsdf_layer,
 * cfg) leaves (block list and order, distances, packed words).  Changes are found by comparing the
 * layer's content with the retained result, so the layer's `updated` flags are neither read nor
 * cleared and any writer of the layer is covered.  When there is nothing to start from — no ESDF
 * retained (or an empty one), one of another layer, one computed under other max_distance_m,
 * default_distance_m, min_distance_m, min_weight or add_occupied_crust, or a layer without
 * blocks — the call runs the batch and sets full_rebuild.  Config rules and errors are the batch's; a rejected call leaves the
 * retained ESDF untouched.  `stats`: blocks / observed_voxels / fixed_voxels are whole-map totals,
 * sweeps / block_passes this call's.  Either stats pointer may be NULL. */
typedef struct cg_esdf_update_stats {
  uint64_t blocks_changed;   /* current blocks whose init state changed, new blocks included */
  uint64_t blocks_removed;   /* retained blocks the layer no longer has */
  uint64_t blocks_region;    /* blocks re-solved: those within reach of a changed or removed one */
  int32_t full_rebuild;      /* 1: ran as the batch (all blocks changed and re-solved) */
  int32_t reserved;
} cg_esdf_update_stats;
int32_t cg_layer_esdf_update(const cg_layer* tsdf_layer, const cg_esdf_config* cfg,
                             cg_esdf_stats* stats, cg_esdf_update_stats* update_stats);
/* Copies the retained ESDF out: blocks in (z, y, x) order, distance float[B*4096] and
 * packed uint32[B*4096] by linear voxel index — the two words Block<EsdfVoxel>::serializeToIntegers
 * emits per voxel: packed = parent.x << 24 | parent.y << 16 | parent.z << 8 | flags (int8 parent
 * components; flags: 1 observed, 2 hallucinated, 4 in_queue (always 0), 8 fixed).  `parent` points
 * to the first neighbour (faces, edges, corners; dz, dy, dx ascending) that attains the distance
 * (upstream: whichever the queue order met).  Any pointer may be NULL. */
int32_t cg_esdf_fetch(cg_context* ctx, size_t capacity_blocks, int32_t* block_idx_xyz,
                      float* distance, uint32_t* packed, size_t* num_blocks_out);
/* createFreePointcloudFromEsdfLayer(esdf, min_distance): (x, y, z, intensity = distance) of every
 * observed voxel with distance >= min_distance, blocks in (z, y, x) order, voxels by linear index.
 * *num_points_out is always set; xyzi (float[4*capacity_points], may be NULL) is filled when the
 * capacity suffices.  Uses the scratch of cg_layer_mesh: a mesh retained for cg_mesh_fetch /
 * cg_mesh_connect is gone afterwards. */
int32_t cg_esdf_free_points(cg_context* ctx, float min_distance, size_t capacity_points,
                            float* xyzi, size_t* num_points_out);

/* --- incremental re-projection (SURVEY.md §8f N1).  The reference rebuilds the whole global map
 * on every trigger (coxgraph/include/coxgraph/server/coxgraph_server.h:275-283 ->
 * coxgraph/src/server/visualizer/server_visualizer.cpp:123-126) although it knows which submap
 * poses the optimisation moved (coxgraph/src/client/coxgraph_client.cpp:135-153,
 * coxgraph/src/server/client_handler.cpp:106-129).  Precondition: `global_layer` holds the
 * projection of `submaps` under `poses_old` (cg_project_submaps into an empty layer, or an earlier
 * cg_reproject_submaps).  Submap i counts as moved when its translation changed by more than
 * eps_translation [m] or its rotation by more than eps_rotation [rad] (bit-identical poses never
 * count).  On return the layer is bit-identical to clearing it and projecting every submap with
 * pose_eff[i] = moved ? poses_new[i] : poses_old[i]; changed_out[i] (optional) tells which. */
typedef struct cg_reproject_stats {
  uint64_t submaps_moved;
  uint64_t blocks_dirty;    /* destination blocks a moved submap reaches under either pose */
  uint64_t candidates;      /* (dirty block, submap) pairs resampled */
  uint64_t blocks_folded;   /* pairs that carried data */
  uint64_t blocks_removed;  /* dirty blocks left without data: removed from the layer */
  uint64_t full_rebuild;    /* 1: more than 30 % of the map was dirty, the whole map was rebuilt
                               (same result, cheaper than rebuilding block by block) */
} cg_reproject_stats;
int32_t cg_reproject_submaps(const cg_layer* const* submaps, const float* poses_old,
                             const float* poses_new, size_t num_submaps, float eps_translation,
                             float eps_rotation, cg_layer* global_layer, uint8_t* changed_out,
                             cg_reproject_stats* stats);

/* --- multi-GPU exchange of partial global layers (DESIGN.md "Multi-GPU") -------------
 * Ownership of a global block is owner = cg_block_owner(idx, nranks).  Each rank packs the
 * blocks of its partial layer destined to every peer into one device buffer of records
 * {int32 x,y,z,flags; 3 x 4096 x 4 B planes} grouped by owner; the host exchanges them
 * (NCCL all-to-all through torch.distributed or ncclSend/Recv) and the owner folds the
 * received records in ascending source-rank order with mergeVoxelAIntoVoxelB. */
#define CG_PACKED_BLOCK_BYTES (16 + CG_BLOCK_BYTES)
int32_t cg_block_owner(int32_t bx, int32_t by, int32_t bz, int32_t nranks);
/* counts_out[nranks]: number of blocks per owner; d_packed must hold num_blocks records. */
int32_t cg_layer_pack_by_owner(const cg_layer* layer, int32_t nranks, void* d_packed,
                               size_t capacity_blocks, uint64_t* counts_out);
/* Fold `num_blocks` packed records (device memory) into `layer` in record order. */
int32_t cg_layer_merge_packed(cg_layer* layer, const void* d_packed, size_t num_blocks);

/* --- the same exchange without the host in the data path (SURVEY.md §8b cg_comm_init /
 * cg_gather_global): one process per GPU of one box.  Rank 0 makes a unique id
 * (cg_comm_get_unique_id = ncclGetUniqueId) and the host hands it to every rank (MPI, a TCP store,
 * a ROS parameter ...); cg_comm_init builds the NCCL communicator on the context's GPU.
 * cg_gather_global is collective: every rank passes ITS partial global layer (all created with
 * the same voxel size and max_blocks) and the layer it owns.  Every block of every partial layer
 * ends up in exactly one rank's `owned` layer: the owner is one of the ranks that HOLD the block,
 * picked by a hash of its index (a block only one rank holds never leaves that GPU), and it folds
 * the holders' copies in ascending rank order (2-argument mergeLayerAintoLayerB semantics,
 * coxgraph/src/server/submap_collection.cpp:31-33) — the union of the owned layers is bit-identical
 * to the packed exchange above.  The fold kernel reads the peers' copies straight from their block
 * pools over NVLink (CUDA IPC peer mappings, opened the first time a partial layer is used); NCCL
 * is the bootstrap and the stream-ordered barrier.  The partial layer may be cleared or refilled as
 * soon as the call returns.  cg_project_submaps_sharded = cg_layer_clear(partial) +
 * cg_project_submaps(this rank's submaps -> partial) + cg_gather_global: cblox getProjectedMap()
 * (coxgraph/src/server/visualizer/server_visualizer.cpp:123-126) over all ranks. */
#define CG_COMM_ID_BYTES 128
int32_t cg_comm_get_unique_id(uint8_t id[CG_COMM_ID_BYTES]);
int32_t cg_comm_init(cg_context* ctx, const uint8_t id[CG_COMM_ID_BYTES], int32_t rank,
                     int32_t nranks);
int32_t cg_comm_destroy(cg_context* ctx);
int32_t cg_gather_global(const cg_layer* partial_layer, cg_layer* owned_layer,
                         uint64_t* blocks_folded);
int32_t cg_project_submaps_sharded(const cg_layer* const* submaps, const float* T_M_S_poses,
                                   size_t num_submaps, cg_layer* partial_layer,
                                   cg_layer* owned_layer, cg_merge_stats* stats);

/* MeshIntegrator::generateMesh over the sharded global map, where it lies (the mesh half of
 * saveAndPubCombinedMesh on several GPUs).  Collective: every rank of the context's communicator
 * passes its owned layer (cg_gather_global's `owned`; all ranks' owned layers have the same voxel
 * size and max_blocks) and gets the block meshes of the blocks that layer holds, in (z, y, x)
 * order, with cg_layer_mesh's conventions and arguments; the result stays in the context for
 * cg_mesh_fetch and the NULL-array count query.  Every block lookup of the mesher — the +x/+y/+z
 * neighbours a block's border cubes read, and the block of a vertex's colour — is resolved across
 * the ranks (the peer's block is read over NVLink), so for every block the rank holding it produces
 * byte for byte what cg_layer_mesh produces for that block on ONE layer holding the union of all
 * ranks' owned layers (voxels and `updated` flags).  A block no rank holds is missing, as in
 * cg_layer_mesh.
 * Errors: no communicator (cg_comm_init) -> CG_ERR_INVALID_ARG; owned layers of different voxel
 * size or max_blocks, or a block key held by more than one rank (two cg_gather_global calls into
 * owned layers not cleared in between can leave one) -> CG_ERR_INVALID_ARG on every rank, the
 * message names the rank or the key.  The call ends with a barrier: a rank may clear or refill its
 * owned layer as soon as it returns.  The owned layer's buffers are mapped into the peers the first
 * time it is used and stay mapped until every rank has passed another owned layer or destroyed its
 * communicator; destroy an owned layer only after that.  cg_mesh_connect stays rank-local (the
 * first-occurrence order over the global block order would need a gather). */
int32_t cg_layer_mesh_sharded(const cg_layer* owned_layer, float min_weight, int32_t use_color,
                              int32_t only_updated, size_t capacity_blocks, size_t capacity_vertices,
                              int32_t* block_idx_xyz, uint32_t* vertex_begin, float* vertices_xyz,
                              float* normals_xyz, uint8_t* colors_rgba,
                              size_t* num_blocks_out, size_t* num_vertices_out);
/* Peer mappings (cudaIpcOpenMemHandle) of the context's communicator: opened since cg_comm_init,
 * and open now.  A layer is mapped once per role (partial, owned), not once per call. */
int32_t cg_comm_peer_mappings(const cg_context* ctx, uint64_t* opened_total, uint64_t* open_now);

/* --- self checks of device arithmetic shortcuts (which: 0 = exact division through a
 * precomputed reciprocal, 1 = round-half-away, 2 = RayCaster state at block entries computed
 * without walking, `samples` random rays); *mismatches must come back 0.  which = 3 runs the same
 * rays as 2 and returns the number of block entries it compared instead. */
int32_t cg_debug_selftest(cg_context* ctx, int32_t which, uint64_t samples, uint64_t* mismatches);

#ifdef __cplusplus
}
#endif
#endif /* COXGRAPH_B200_H_ */
