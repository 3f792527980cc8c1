/*
 * tsdf_oracle.h — C interface of the CPU ORACLE for the coxgraph TSDF hot path.
 *
 * TEST INFRASTRUCTURE ONLY.  Nothing under oracle/ is part of the product: only
 * tests/, __graft_entry__.smoke() and bench.py's cpu_baseline / --impl reference
 * legs may load this library, and there only as the checker / CPU baseline.
 *
 * PARITY UNPINNED: the reference tree (/root/reference) holds no source of the
 * arithmetic on this path (it lives in the un-vendored forks LXYYY/voxblox,
 * LXYYY/cblox, LXYYY/voxgraph, branch names only, coxgraph_ssh.rosinstall:1-8,55-58),
 * no tests and no golden vectors.  This oracle restates the published upstream
 * voxblox algorithm (integrator/tsdf_integrator.cc, integrator/integrator_utils.cc,
 * integrator/merge_integration.h, interpolator/interpolator_inl.h, core/voxel.cc,
 * core/color.h, core/common.h) and is anchored on the reference's call sites:
 *   coxgraph/include/coxgraph/map_comm/tsdf_recover.h:59-99 (integratePointCloud :75)
 *   coxgraph/src/client/map_server.cpp:59-73            (mergeLayerAintoLayerB :67-69)
 *   coxgraph/src/server/visualizer/server_visualizer.cpp:123-126 (getProjectedMap)
 * It is pinned by analytic / algebraic known-answer tests (tests/test_oracle_*.py)
 * and by frozen digests under tests/golden/.
 * One part IS pinned to reference source: the MeshConverter section (orc_mesh_to_frames) restates
 * coxgraph/include/coxgraph/map_comm/mesh_converter.h, which is in the reference tree, line by
 * line (tests/test_mesh_recover.py checks it against hand-evaluated values of those formulas).
 */
#ifndef TSDF_ORACLE_H_
#define TSDF_ORACLE_H_

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

typedef struct orc_layer orc_layer;

/* Mirrors voxblox::TsdfIntegratorBase::Config (upstream defaults in comments). */
typedef struct orc_integrator_config {
  float default_truncation_distance;  /* 0.1 */
  float max_weight;                   /* 10000 */
  int32_t voxel_carving_enabled;      /* 1 */
  float min_ray_length_m;             /* 0.1 */
  float max_ray_length_m;             /* 5.0 */
  int32_t use_const_weight;           /* 0 */
  int32_t allow_clear;                /* 1 */
  int32_t use_weight_dropoff;         /* 1 */
  int32_t use_sparsity_compensation_factor; /* 0 */
  float sparsity_compensation_factor; /* 1.0 */
  int32_t enable_anti_grazing;        /* 0 */
  int32_t method;                     /* 0 simple, 1 merged, 2 fast */
  int32_t integration_order_mode;     /* 0 mixed (default), 1 natural index order */
  float start_voxel_subsampling_factor;     /* 2.0 (fast) */
  int32_t max_consecutive_ray_collisions;   /* 2   (fast) */
} orc_integrator_config;

void orc_default_config(orc_integrator_config* cfg);

orc_layer* orc_layer_create(float voxel_size, int32_t voxels_per_side);
void orc_layer_destroy(orc_layer* layer);
void orc_layer_clear(orc_layer* layer); /* Layer::removeAllBlocks */
size_t orc_layer_num_blocks(const orc_layer* layer);

/* Blocks are returned sorted by (z, y, x) block index.  voxels: B*4096 records of
 * {float distance; float weight; uint8 r,g,b,a} (voxblox TsdfVoxel AoS, linear index
 * x + 16*(y + 16*z)).  flags: bit0 has_data, bit1 updated.  Any pointer may be NULL. */
void orc_layer_download(const orc_layer* layer, int32_t* block_idx_xyz, void* voxels,
                        uint8_t* flags);
void orc_layer_upload(orc_layer* layer, const int32_t* block_idx_xyz, const void* voxels,
                      const uint8_t* flags, size_t num_blocks);

/* TsdfIntegratorBase::integratePointCloud(T_G_C, points_C, colors, freespace_points).
 * T = {qw,qx,qy,qz,tx,ty,tz}.  Single thread, canonical deterministic order.
 * Returns 0, or <0 on error.  *blocks_touched (optional) = distinct blocks visited. */
int32_t orc_integrate_pointcloud(orc_layer* layer, const orc_integrator_config* cfg,
                                 const float T_G_C[7], const float* points_xyz,
                                 const uint8_t* colors_rgba, size_t n,
                                 int32_t freespace_points, uint64_t* blocks_touched);

/* One call of updateTsdfVoxel: the global voxel index, the signed distance, the weight after
 * drop-off and sparsity compensation, and the ray colour. */
typedef struct orc_visit {
  int32_t x, y, z;
  float sdf;
  float weight;
  uint8_t rgba[4];
} orc_visit;

/* orc_integrate_pointcloud that also records every voxel update, in call order (anti-grazing
 * skips are not updates).  The arithmetic is the same.  On success *trace is a malloc'd array of
 * *num_visits records (free it with orc_trace_free). */
int32_t orc_integrate_pointcloud_traced(orc_layer* layer, const orc_integrator_config* cfg,
                                        const float T_G_C[7], const float* points_xyz,
                                        const uint8_t* colors_rgba, size_t n,
                                        int32_t freespace_points, uint64_t* blocks_touched,
                                        orc_visit** trace, size_t* num_visits);
void orc_trace_free(orc_visit* trace);

/* Timing variant: voxblox-style threading (striped voxel mutexes, allocation mutex).
 * Result is order-nondeterministic like the real thing; used only as CPU baseline. */
int32_t orc_integrate_pointcloud_mt(orc_layer* layer, const orc_integrator_config* cfg,
                                    const float T_G_C[7], const float* points_xyz,
                                    const uint8_t* colors_rgba, size_t n,
                                    int32_t freespace_points, int32_t threads);

/* voxblox::mergeLayerAintoLayerB(layer_A, T_B_A, layer_B) = transformLayer + merge.
 * *blocks_out (optional) = blocks of the transformed layer that carried data. */
int32_t orc_merge_layer_into_layer(const orc_layer* layer_a, const float T_B_A[7],
                                   orc_layer* layer_b, uint64_t* blocks_out);
/* Same, candidate blocks resampled by `threads` workers (block-parallel; deterministic). */
int32_t orc_merge_layer_into_layer_mt(const orc_layer* layer_a, const float T_B_A[7],
                                      orc_layer* layer_b, int32_t threads,
                                      uint64_t* blocks_out);

/* 2-argument voxblox::mergeLayerAintoLayerB(layer_A, layer_B) for layers on the same grid
 * (call site coxgraph/src/server/submap_collection.cpp:31-33): Block::mergeBlock per block,
 * blocks of A without data are skipped. */
int32_t orc_merge_layer_aligned(const orc_layer* layer_a, orc_layer* layer_b);

/* Small pieces exposed for known-answer tests. */
void orc_transform_point(const float T[7], const float p[3], float out[3]);
void orc_inverse_transform(const float T[7], float Tinv[7]);
/* Ray-cast; writes up to cap voxel indices (int64 xyz), returns number produced. */
size_t orc_cast_ray(const float origin[3], const float point_G[3], int32_t clearing,
                    int32_t carving, float max_ray, float voxel_size_inv, float trunc,
                    int32_t cast_from_origin, int64_t* out_xyz, size_t cap);
/* Interpolator<TsdfVoxel>::getVoxel(pos, &voxel, interpolate). returns 1 on success. */
int32_t orc_interp_voxel(const orc_layer* layer, const float pos[3], int32_t interpolate,
                         float* distance, float* weight, uint8_t rgba[4]);

/* ---- MeshConverter (coxgraph/include/coxgraph/map_comm/mesh_converter.h, IN the reference tree:
 * this part of the oracle is pinned to the reference's own source lines).
 * voxblox_msgs/Mesh flattened: block b owns vertices [vertex_begin[b], vertex_begin[b+1]) (a
 * multiple of 3 each: triangles), x/y/z are the uint16 offsets inside the block, r/g/b the vertex
 * colours; triangle t (= vertex index / 3) owns the history entries [hist_begin[t],
 * hist_begin[t+1]) of `hist`, read as (first stamp, last stamp) pairs; block_has_history[b] = 0
 * means MeshBlock.history was empty (the block is skipped, mesh_converter.h:87). */
typedef struct orc_mesh {
  size_t num_blocks;
  const int32_t* block_index;
  const uint8_t* block_has_history;
  const uint32_t* vertex_begin;
  const uint16_t *x, *y, *z;
  const uint8_t *r, *g, *b;
  const uint32_t* hist_begin;
  const uint32_t* hist;
  float block_edge_length;
} orc_mesh;
size_t orc_mesh_to_frames(const orc_mesh* mesh, float interpolate_voxel_size, size_t num_poses,
                          const float* poses, const double* stamps_sec, uint64_t* frame_offsets,
                          float* points_xyz, uint8_t* colors_rgba, size_t capacity_points);

/* ---- MeshIntegrator<TsdfVoxel>::generateMesh (marching cubes per block, [EXT] voxblox
 * mesh/mesh_integrator.h + mesh/marching_cubes.h; parity unpinned).  Blocks in (z, y, x) order;
 * block b owns vertices [vertex_begin[b], vertex_begin[b+1]) (B + 1 entries), in the reference's
 * voxel loop order; three consecutive vertices = one triangle (indices are 0..n-1 per block);
 * normals per vertex (the triangle's), colours nearest-voxel.  With only_updated, blocks whose
 * `updated` flag is clear produce nothing.  Returns the vertex count; arrays are filled only if
 * capacity_vertices suffices.  Any pointer may be NULL. */
size_t orc_layer_mesh(const orc_layer* layer, float min_weight, int32_t use_color,
                      int32_t only_updated, uint32_t* vertex_begin, float* vertices, float* normals,
                      uint8_t* colors, size_t capacity_vertices);
/* voxblox::createConnectedMesh ([EXT] mesh/mesh_utils.h; MeshLayer::getConnectedMesh, the PLY step
 * of saveAndPubCombinedMesh, coxgraph/src/server/visualizer/server_visualizer.cpp:118-126) of a
 * flat triangle list (n vertices in block order): a hash map from round(double(v) / double(1e-10f))
 * per axis to the first vertex of that cell.  out_indices[n]; the unique vertices' old indices go to
 * first_old_index (capacity n).  Returns the number of unique vertices. */
size_t orc_connect_mesh(const float* vertices, size_t n, uint32_t* out_indices,
                        uint32_t* first_old_index);
/* kTriangleTable[256][16] */
const int* orc_triangle_table(void);

/* ---- EsdfIntegrator::updateFromTsdfLayerBatch ([EXT] voxblox integrator/esdf_integrator.cc,
 * utils/bucket_queue.h, utils/neighbor_tools.h; parity unpinned), the call of
 * coxgraph/include/coxgraph/client/map_server.h:141-145: the ESDF layer is rebuilt from every
 * allocated TSDF block — voxels inside |distance| < min_distance_m are copied and fixed, the others
 * start at +-default_distance_m and are lowered by the quasi-Euclidean 26-neighbour wavefront of
 * processOpenSet (bucketed open queue, an update is taken when it improves by more than
 * min_diff_m).  Sequential; blocks in (z, y, x) order.  Mirrors voxblox::EsdfIntegrator::Config
 * (upstream defaults in comments); full_euclidean_distance is not restated. */
typedef struct orc_esdf_config {
  float max_distance_m;      /* 2.0 */
  float default_distance_m;  /* 2.0 */
  float min_distance_m;      /* 0.2 */
  float min_diff_m;          /* 0.001 */
  float min_weight;          /* 1e-6 */
  int32_t num_buckets;       /* 20 */
  int32_t multi_queue;       /* 0 */
  int32_t add_occupied_crust; /* 0 */
} orc_esdf_config;
typedef struct orc_esdf orc_esdf;
void orc_esdf_default_config(orc_esdf_config* cfg);
orc_esdf* orc_esdf_batch(const orc_layer* tsdf, const orc_esdf_config* cfg);
void orc_esdf_destroy(orc_esdf* esdf);
size_t orc_esdf_num_blocks(const orc_esdf* esdf);
uint64_t orc_esdf_updates(const orc_esdf* esdf); /* neighbour updates taken by processOpenSet */
/* blocks in (z, y, x) order; distance float[B*4096]; flags uint8[B*4096]: bit0 observed,
 * bit1 hallucinated, bit2 in_queue, bit3 fixed; parent int8[B*4096*3].  Any pointer may be NULL. */
void orc_esdf_download(const orc_esdf* esdf, int32_t* block_idx_xyz, float* distance,
                       uint8_t* flags, int8_t* parent);
/* voxblox::createFreePointcloudFromEsdfLayer (coxgraph/src/client/map_server.cpp:112-113):
 * (x, y, z, intensity = distance) of every observed voxel with distance >= min_distance, blocks in
 * (z, y, x) order, voxels by linear index.  Returns the count; fills up to `capacity` points. */
size_t orc_esdf_free_points(const orc_esdf* esdf, float min_distance, float* xyzi, size_t capacity);

#ifdef __cplusplus
}
#endif
#endif /* TSDF_ORACLE_H_ */
