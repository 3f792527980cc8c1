// coxgraph_b200.hpp — C++ host-side mirror of the reference-facing interface of the hot path,
// header-only, on top of the C ABI (include/coxgraph_b200.h, libcoxgraph_b200.so).
//
// The reference (mfkiwl/coxgraph) is C++ and reaches this path through voxblox's classes; this
// header keeps their names, argument order and meaning so that the call sites read the same:
//   tsdf_integrator_->integratePointCloud(T_G_C, *points_C, *colors, false)
//       coxgraph/include/coxgraph/map_comm/tsdf_recover.h:75
//   tsdf_map_->getTsdfLayerPtr()->removeAllBlocks()                    tsdf_recover.h:62
//   voxblox::mergeLayerAintoLayerB(layer, submap->getPose(), combined) coxgraph/src/client/map_server.cpp:67-69
//   SubmapCollection::getProjectedMap()   via coxgraph/src/server/visualizer/server_visualizer.cpp:123-126
// Types are layout-compatible with the ones the reference passes (Eigen::Vector3f = 3 floats,
// voxblox::Color = 4 x uint8, kindr QuatTransformation = unit quaternion w,x,y,z + translation),
// so an adapter inside a voxblox build is a reinterpret of the containers' data pointers
// (INTEGRATION.md shows it).
//
// Error behaviour: the reference aborts through glog CHECK / LOG(FATAL) on this path
// (e.g. coxgraph/include/coxgraph/utils/msg_converter.h:110-111).  Here every failed C-ABI call
// goes through fatal(), which prints cg_last_error() and aborts; set_fatal_handler() lets a host
// turn that into an exception instead.  There is no CPU fallback anywhere.
#ifndef COXGRAPH_B200_HPP_
#define COXGRAPH_B200_HPP_

#include <cstdint>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <functional>
#include <memory>
#include <stdexcept>
#include <string>
#include <vector>

#include "../../include/coxgraph_b200.h"

namespace coxgraph_b200 {

using FloatingPoint = float;
struct Point {  // Eigen::Matrix<float, 3, 1>
  FloatingPoint x, y, z;
};
struct Color {  // voxblox::Color
  uint8_t r = 0, g = 0, b = 0, a = 255;
};
using Pointcloud = std::vector<Point>;  // voxblox::AlignedVector<Point>
using Colors = std::vector<Color>;
struct BlockIndex {  // voxblox::BlockIndex (Eigen::Vector3i)
  int32_t x, y, z;
};
using BlockIndexList = std::vector<BlockIndex>;
using TsdfVoxel = cg_tsdf_voxel;  // {float distance; float weight; Color color}
static_assert(sizeof(Point) == 12 && sizeof(Color) == 4 && sizeof(TsdfVoxel) == 12 &&
                  sizeof(BlockIndex) == 12,
              "layouts must match the reference's types");

// kindr::minimal::QuatTransformationTemplate<float>: p_G = q * p_C + t
struct Transformation {
  FloatingPoint qw = 1, qx = 0, qy = 0, qz = 0, tx = 0, ty = 0, tz = 0;
  const float* data() const { return &qw; }
};

// ---- error handling -------------------------------------------------------------------
using FatalHandler = std::function<void(int32_t status, const char* message)>;
inline FatalHandler& fatal_handler() {
  static FatalHandler h = [](int32_t status, const char* message) {
    std::fprintf(stderr, "coxgraph_b200: fatal error %d: %s\n", static_cast<int>(status), message);
    std::abort();  // what glog CHECK does in the reference
  };
  return h;
}
inline void set_fatal_handler(FatalHandler h) { fatal_handler() = std::move(h); }
struct Error : std::runtime_error {
  int32_t status;
  Error(int32_t s, const char* m) : std::runtime_error(m), status(s) {}
};
inline void throw_on_error() {
  set_fatal_handler([](int32_t s, const char* m) { throw Error(s, m); });
}
inline void check(int32_t status) {
  if (status != CG_OK) fatal_handler()(status, cg_last_error());
}

// ---- context: one per GPU / process rank ----------------------------------------------
class Context {
 public:
  explicit Context(int device = 0, void* cuda_stream = nullptr) {
    check(cg_context_create(device, cuda_stream, &ctx_));
  }
  ~Context() {
    if (ctx_) cg_context_destroy(ctx_);
  }
  Context(const Context&) = delete;
  Context& operator=(const Context&) = delete;
  cg_context* handle() const { return ctx_; }
  void synchronize() const { check(cg_context_synchronize(ctx_)); }
  uint64_t kernelLaunches() const { return cg_context_kernel_launches(ctx_); }
  // queue the host->device copy of a LATER job's clouds into staging slot 0 / 1 and return at
  // once; the vectors must stay alive and unchanged until that job has been integrated
  void stageBatchAsync(int stage_slot, const Pointcloud& points_C, const Colors& colors) const {
    if (points_C.size() != colors.size())
      fatal_handler()(CG_ERR_INVALID_ARG, "stageBatchAsync: points_C.size() != colors.size()");
    check(cg_stage_batch_async(ctx_, stage_slot, points_C.empty() ? nullptr : &points_C[0].x,
                               colors.empty() ? nullptr : &colors[0].r, points_C.size()));
  }

 private:
  cg_context* ctx_ = nullptr;
};

// ---- voxblox::Block<TsdfVoxel> as handed across the boundary ---------------------------
struct TsdfBlock {
  BlockIndex block_index;
  bool has_data = false, updated = false;
  std::vector<TsdfVoxel> voxels;  // 4096, linear index x + 16 (y + 16 z)
};

// ---- voxblox::Layer<TsdfVoxel> ----------------------------------------------------------
class TsdfLayer {
 public:
  // Layer(voxel_size, voxels_per_side); max_blocks sizes the block pool in HBM
  TsdfLayer(const Context& ctx, FloatingPoint voxel_size, size_t voxels_per_side = 16,
            size_t max_blocks = 4096) {
    check(cg_layer_create(ctx.handle(), voxel_size, static_cast<int32_t>(voxels_per_side),
                          max_blocks, &layer_));
    ctx_ = ctx.handle();
  }
  ~TsdfLayer() {
    if (layer_) cg_layer_destroy(layer_);
  }
  TsdfLayer(const TsdfLayer&) = delete;
  TsdfLayer& operator=(const TsdfLayer&) = delete;

  cg_layer* handle() const { return layer_; }
  cg_context* context() const { return ctx_; }
  FloatingPoint voxel_size() const { return cg_layer_voxel_size(layer_); }
  size_t voxels_per_side() const { return CG_VOXELS_PER_SIDE; }
  FloatingPoint block_size() const { return voxel_size() * CG_VOXELS_PER_SIDE; }
  size_t getNumberOfAllocatedBlocks() const {
    return static_cast<size_t>(cg_layer_num_blocks(layer_));
  }
  size_t getMemorySize() const { return getNumberOfAllocatedBlocks() * CG_BLOCK_BYTES; }
  void removeAllBlocks() { check(cg_layer_clear(layer_)); }
  // Layer::removeBlock(index); returns whether the block existed
  bool removeBlock(const BlockIndex& index) {
    uint64_t removed = 0;
    check(cg_layer_remove_blocks(layer_, 1, &index.x, &removed));
    return removed != 0;
  }
  void getAllAllocatedBlocks(BlockIndexList* blocks) const {
    const size_t n = getNumberOfAllocatedBlocks();
    blocks->resize(n);
    size_t got = 0;
    check(cg_layer_block_indices(layer_, n, n ? &(*blocks)[0].x : nullptr, &got));
  }
  // copy the layer out in voxblox's own block layout (what serializeLayerAsMsg walks,
  // coxgraph/include/coxgraph/map_comm/tsdf_recover.h:95)
  void download(BlockIndexList* indices, std::vector<TsdfVoxel>* voxels,
                std::vector<uint8_t>* flags = nullptr) const {
    const size_t n = getNumberOfAllocatedBlocks();
    indices->resize(n);
    voxels->resize(n * CG_VOXELS_PER_BLOCK);
    if (flags) flags->resize(n);
    size_t got = 0;
    check(cg_layer_download(layer_, n, n ? &(*indices)[0].x : nullptr, voxels->data(),
                            flags ? flags->data() : nullptr, &got));
  }
  // voxblox::serializeLayerAsMsg block payload (Block::serializeToIntegers per block: 3 words per
  // voxel, colour a | b<<8 | g<<16 | r<<24), produced on the device
  void serializeLayerAsMsg(bool only_updated, BlockIndexList* indices,
                           std::vector<uint32_t>* data) const {
    size_t n = 0;
    check(cg_layer_serialize(layer_, only_updated ? 1 : 0, 0, nullptr, nullptr, &n));
    indices->resize(n);
    data->resize(n * 3 * CG_VOXELS_PER_BLOCK);
    if (n)
      check(cg_layer_serialize(layer_, only_updated ? 1 : 0, n, &(*indices)[0].x, data->data(), &n));
  }
  void deserializeMsgToLayer(const BlockIndexList& indices, const std::vector<uint32_t>& data) {
    if (data.size() != indices.size() * 3 * CG_VOXELS_PER_BLOCK)
      fatal_handler()(CG_ERR_INVALID_ARG, "deserializeMsgToLayer: data size does not match");
    check(cg_layer_deserialize(layer_, indices.size(), indices.empty() ? nullptr : &indices[0].x,
                               data.data()));
  }
  // Layer::getBlockPtrByIndex for the listed blocks only: found[i] tells whether block i is
  // allocated (for layers too large to copy out whole)
  void downloadBlocks(const BlockIndexList& indices, std::vector<TsdfVoxel>* voxels,
                      std::vector<uint8_t>* found, std::vector<uint8_t>* flags = nullptr) const {
    voxels->resize(indices.size() * CG_VOXELS_PER_BLOCK);
    found->resize(indices.size());
    if (flags) flags->resize(indices.size());
    check(cg_layer_download_blocks(layer_, indices.size(), indices.empty() ? nullptr : &indices[0].x,
                                   voxels->data(), flags ? flags->data() : nullptr, found->data()));
  }
  cg_hash_stats hashStats() const {
    cg_hash_stats st;
    check(cg_layer_hash_stats(layer_, &st));
    return st;
  }
  // insert / overwrite blocks (deserializeMsgToLayer hand-off,
  // coxgraph/include/coxgraph/utils/msg_converter.h:107-109)
  void upload(const BlockIndexList& indices, const std::vector<TsdfVoxel>& voxels,
              const std::vector<uint8_t>* flags = nullptr) {
    if (voxels.size() != indices.size() * CG_VOXELS_PER_BLOCK)
      fatal_handler()(CG_ERR_INVALID_ARG, "TsdfLayer::upload: voxel count does not match");
    check(cg_layer_upload(layer_, indices.size(), indices.empty() ? nullptr : &indices[0].x,
                          voxels.data(), flags ? flags->data() : nullptr));
  }

 private:
  cg_layer* layer_ = nullptr;
  cg_context* ctx_ = nullptr;
};

// ---- voxblox::TsdfIntegratorBase and its concrete integrators ---------------------------
class TsdfIntegratorBase {
 public:
  using Ptr = std::shared_ptr<TsdfIntegratorBase>;
  struct Config : cg_integrator_config {
    Config() { cg_integrator_config_default(this); }
  };
  TsdfIntegratorBase(const Config& config, TsdfLayer* layer) : config_(config), layer_(layer) {}
  virtual ~TsdfIntegratorBase() = default;

  // Integrates the point cloud into the TSDF layer (same contract as voxblox: points in the
  // sensor frame C, T_G_C the sensor pose, one colour per point).
  virtual void integratePointCloud(const Transformation& T_G_C, const Pointcloud& points_C,
                                   const Colors& colors, const bool freespace_points = false) {
    if (points_C.size() != colors.size())
      fatal_handler()(CG_ERR_INVALID_ARG, "integratePointCloud: points_C.size() != colors.size()");
    check(cg_integrate_pointcloud(layer_->handle(), &config_, T_G_C.data(),
                                  points_C.empty() ? nullptr : &points_C[0].x,
                                  colors.empty() ? nullptr : &colors[0].r, points_C.size(),
                                  freespace_points ? 1 : 0, &stats_));
  }
  // The frame loop of TsdfRecover::processMesh (tsdf_recover.h:71-86) as one job: identical
  // result to calling integratePointCloud once per frame, in order.
  void integratePointClouds(const std::vector<Transformation>& T_G_C,
                            const std::vector<const Pointcloud*>& points_C,
                            const std::vector<const Colors*>& colors,
                            const bool freespace_points = false) {
    const size_t F = T_G_C.size();
    if (points_C.size() != F || colors.size() != F)
      fatal_handler()(CG_ERR_INVALID_ARG, "integratePointClouds: one cloud per pose expected");
    std::vector<uint64_t> offs(F + 1, 0);
    for (size_t f = 0; f < F; ++f) offs[f + 1] = offs[f] + points_C[f]->size();
    std::vector<Point> pts(offs[F]);
    std::vector<Color> cols(offs[F]);
    std::vector<float> poses(7 * F);
    for (size_t f = 0; f < F; ++f) {
      std::copy(points_C[f]->begin(), points_C[f]->end(), pts.begin() + offs[f]);
      std::copy(colors[f]->begin(), colors[f]->end(), cols.begin() + offs[f]);
      std::copy(T_G_C[f].data(), T_G_C[f].data() + 7, poses.begin() + 7 * f);
    }
    check(cg_integrate_batch(layer_->handle(), &config_, F, poses.data(),
                             pts.empty() ? nullptr : &pts[0].x, cols.empty() ? nullptr : &cols[0].r,
                             offs.data(), freespace_points ? 1 : 0, &stats_));
  }
  // Registered depth + colour images (sensor_msgs/Image pairs of one CameraInfo): the same
  // layer as depth_image_proc point_cloud_xyzrgb followed by TsdfServer's insertion of that cloud
  // (its non-finite points dropped).  depth: W*H uint16 (16UC1) or float (32FC1) per frame,
  // tightly packed; colour: W*H pixels of the camera's colour encoding.
  struct DepthImage {
    const void* data;
  };
  struct ColorImage {
    const uint8_t* data;
  };
  void integrateDepthImage(const Transformation& T_G_C, const DepthImage& depth,
                           const ColorImage& color, const cg_depth_camera& camera) {
    check(cg_integrate_depth_batch(layer_->handle(), &config_, 1, T_G_C.data(), &camera, depth.data,
                                   color.data, &stats_));
  }
  // F frames as one job: depth / colour of frame f at depth[f] / color[f]
  void integrateDepthImages(const std::vector<Transformation>& T_G_C,
                            const std::vector<DepthImage>& depth,
                            const std::vector<ColorImage>& color, const cg_depth_camera& camera) {
    const size_t F = T_G_C.size();
    if (depth.size() != F || color.size() != F)
      fatal_handler()(CG_ERR_INVALID_ARG, "integrateDepthImages: one image pair per pose expected");
    if (camera.width <= 0 || camera.height <= 0)
      fatal_handler()(CG_ERR_INVALID_ARG, "integrateDepthImages: invalid image size");
    const size_t px = static_cast<size_t>(camera.width) * static_cast<size_t>(camera.height);
    const size_t dsize = camera.depth_encoding == CG_DEPTH_16UC1 ? 2 : 4;
    const size_t csize = camera.color_encoding == CG_COLOR_MONO8 ? 1
                         : (camera.color_encoding == CG_COLOR_RGBA8 ||
                            camera.color_encoding == CG_COLOR_BGRA8) ? 4 : 3;
    std::vector<uint8_t> d(F * px * dsize), c(F * px * csize);
    std::vector<float> poses(7 * F);
    for (size_t f = 0; f < F; ++f) {
      std::memcpy(&d[f * px * dsize], depth[f].data, px * dsize);
      std::memcpy(&c[f * px * csize], color[f].data, px * csize);
      std::copy(T_G_C[f].data(), T_G_C[f].data() + 7, poses.begin() + 7 * f);
    }
    check(cg_integrate_depth_batch(layer_->handle(), &config_, F, poses.data(), &camera,
                                   d.empty() ? nullptr : d.data(), c.empty() ? nullptr : c.data(),
                                   &stats_));
  }
  // Pipelined jobs for a host that knows its next job (the recover loop does: tsdf_recover.h:
  // 71-86): prepareDevice queues the layer-independent first half of a LATER job — points already
  // on the device, or staged with cg_stage_batch_async — into slot 0 / 1 and returns at once;
  // integratePrepared completes it.  Same result as integratePointClouds.
  void prepareDevice(int slot, const std::vector<Transformation>& T_G_C, const float* d_points_xyz,
                     const uint8_t* d_colors_rgba, const std::vector<uint64_t>& frame_offsets,
                     const bool freespace_points = false) {
    if (frame_offsets.size() != T_G_C.size() + 1)
      fatal_handler()(CG_ERR_INVALID_ARG, "prepareDevice: F + 1 frame offsets expected");
    std::vector<float> poses(7 * T_G_C.size());
    for (size_t f = 0; f < T_G_C.size(); ++f)
      std::copy(T_G_C[f].data(), T_G_C[f].data() + 7, poses.begin() + 7 * f);
    check(cg_prepare_batch_device(layer_->handle(), &config_, T_G_C.size(), poses.data(),
                                  d_points_xyz, d_colors_rgba, frame_offsets.data(),
                                  freespace_points ? 1 : 0, slot));
  }
  // the same for clouds staged with Context::stageBatchAsync(stage_slot, ...)
  void prepareStaged(int slot, const std::vector<Transformation>& T_G_C, int stage_slot,
                     const std::vector<uint64_t>& frame_offsets,
                     const bool freespace_points = false) {
    if (frame_offsets.size() != T_G_C.size() + 1)
      fatal_handler()(CG_ERR_INVALID_ARG, "prepareStaged: F + 1 frame offsets expected");
    std::vector<float> poses(7 * T_G_C.size());
    for (size_t f = 0; f < T_G_C.size(); ++f)
      std::copy(T_G_C[f].data(), T_G_C[f].data() + 7, poses.begin() + 7 * f);
    check(cg_prepare_batch_staged(layer_->handle(), &config_, T_G_C.size(), poses.data(),
                                  stage_slot, frame_offsets.data(), freespace_points ? 1 : 0, slot));
  }
  void integratePrepared(int slot) { check(cg_integrate_prepared(layer_->handle(), slot, &stats_)); }
  void setLayer(TsdfLayer* layer) { layer_ = layer; }
  const Config& getConfig() const { return config_; }
  const cg_integrate_stats& lastStats() const { return stats_; }

 protected:
  Config config_;
  TsdfLayer* layer_;
  cg_integrate_stats stats_{};
};

class SimpleTsdfIntegrator : public TsdfIntegratorBase {
 public:
  SimpleTsdfIntegrator(const Config& config, TsdfLayer* layer) : TsdfIntegratorBase(config, layer) {
    config_.method = CG_METHOD_SIMPLE;
  }
};
class MergedTsdfIntegrator : public TsdfIntegratorBase {
 public:
  MergedTsdfIntegrator(const Config& config, TsdfLayer* layer) : TsdfIntegratorBase(config, layer) {
    config_.method = CG_METHOD_MERGED;
  }
};

// voxblox::TsdfIntegratorFactory::create(integrator_type_name, config, layer).  The reference's
// yaml files ask for "fast" (tsdf_server_euroc.yaml:6, tsdf_recover.yaml:6): FastTsdfIntegrator
// is an approximation of the merged integrator whose result depends on thread timing, so "fast"
// maps to the deterministic merged integrator here (DESIGN.md "Integrator methods").
struct TsdfIntegratorFactory {
  static TsdfIntegratorBase::Ptr create(const std::string& integrator_type_name,
                                        const TsdfIntegratorBase::Config& config, TsdfLayer* layer) {
    if (integrator_type_name == "simple")
      return std::make_shared<SimpleTsdfIntegrator>(config, layer);
    if (integrator_type_name == "merged" || integrator_type_name == "fast")
      return std::make_shared<MergedTsdfIntegrator>(config, layer);
    fatal_handler()(CG_ERR_UNSUPPORTED, ("unknown TSDF integrator type: " + integrator_type_name).c_str());
    return nullptr;
  }
};

// ---- TsdfRecover::processMesh (coxgraph/include/coxgraph/map_comm/tsdf_recover.h:59-99): mesh
// with observation history -> per-pose clouds (voxblox::MeshConverter) -> fused layer ----------
inline void recoverMesh(TsdfLayer* layer, const TsdfIntegratorBase::Config& config,
                        const cg_mesh& mesh, FloatingPoint interpolate_voxel_size,
                        const std::vector<Transformation>& T_G_C, const std::vector<double>& stamps_sec,
                        cg_integrate_stats* stats = nullptr) {
  if (T_G_C.size() != stamps_sec.size())
    fatal_handler()(CG_ERR_INVALID_ARG, "recoverMesh: one time stamp per pose expected");
  std::vector<float> poses(7 * T_G_C.size());
  for (size_t i = 0; i < T_G_C.size(); ++i)
    std::copy(T_G_C[i].data(), T_G_C[i].data() + 7, poses.begin() + 7 * i);
  check(cg_recover_mesh(layer->handle(), &config, &mesh, interpolate_voxel_size, T_G_C.size(),
                        poses.data(), stamps_sec.data(), stats));
}

// ---- voxblox::mergeLayerAintoLayerB(layer_A, T_B_A, layer_B) ---------------------------
inline void mergeLayerAintoLayerB(const TsdfLayer& layer_A, const Transformation& T_B_A,
                                  TsdfLayer* layer_B, cg_merge_stats* stats = nullptr) {
  check(cg_merge_layer_into_layer(layer_A.handle(), T_B_A.data(), layer_B->handle(), stats));
}

// ---- cblox::SubmapCollection::getProjectedMap(): every submap merged into one layer, in
// order, with its pose T_M_S (the server's submap-to-global entry point) ---------------------
inline void getProjectedMap(const std::vector<const TsdfLayer*>& submap_layers,
                            const std::vector<Transformation>& T_M_S, TsdfLayer* projected_layer,
                            cg_merge_stats* stats = nullptr) {
  if (submap_layers.size() != T_M_S.size())
    fatal_handler()(CG_ERR_INVALID_ARG, "getProjectedMap: one pose per submap expected");
  std::vector<const cg_layer*> handles(submap_layers.size());
  std::vector<float> poses(7 * T_M_S.size());
  for (size_t i = 0; i < submap_layers.size(); ++i) {
    handles[i] = submap_layers[i]->handle();
    std::copy(T_M_S[i].data(), T_M_S[i].data() + 7, poses.begin() + 7 * i);
  }
  check(cg_project_submaps(handles.data(), poses.data(), handles.size(), projected_layer->handle(),
                           stats));
}

// ---- the same over the GPUs of one box, one process per GPU: every rank passes ITS submaps, a
// scratch partial layer and the layer it owns (all ranks: same voxel size and max_blocks for the
// partial layers).  commInit once per context with the 128-byte id rank 0 made (commUniqueId)
// and the host handed round.
inline std::vector<uint8_t> commUniqueId() {
  std::vector<uint8_t> id(CG_COMM_ID_BYTES);
  check(cg_comm_get_unique_id(id.data()));
  return id;
}
inline void commInit(const Context& ctx, const std::vector<uint8_t>& id, int rank, int nranks) {
  if (id.size() != CG_COMM_ID_BYTES) fatal_handler()(CG_ERR_INVALID_ARG, "commInit: 128-byte id expected");
  check(cg_comm_init(ctx.handle(), id.data(), rank, nranks));
}
inline void getProjectedMapSharded(const std::vector<const TsdfLayer*>& my_submap_layers,
                                   const std::vector<Transformation>& T_M_S, TsdfLayer* partial_layer,
                                   TsdfLayer* owned_layer, cg_merge_stats* stats = nullptr) {
  if (my_submap_layers.size() != T_M_S.size())
    fatal_handler()(CG_ERR_INVALID_ARG, "getProjectedMapSharded: one pose per submap expected");
  std::vector<const cg_layer*> handles(my_submap_layers.size());
  std::vector<float> poses(7 * T_M_S.size());
  for (size_t i = 0; i < my_submap_layers.size(); ++i) {
    handles[i] = my_submap_layers[i]->handle();
    std::copy(T_M_S[i].data(), T_M_S[i].data() + 7, poses.begin() + 7 * i);
  }
  check(cg_project_submaps_sharded(handles.data(), poses.data(), handles.size(),
                                   partial_layer->handle(), owned_layer->handle(), stats));
}

// ---- voxblox::MeshIntegrator<TsdfVoxel>::generateMesh over a device-resident layer (what
// saveAndPubCombinedMesh runs on the projected map, server_visualizer.cpp:123-126): per-block
// marching cubes; block b owns vertices [vertex_begin[b], vertex_begin[b + 1]), three per triangle
struct MeshIntegratorConfig {  // voxblox::MeshIntegratorConfig
  bool use_color = true;
  float min_weight = 1e-4f;
};
struct LayerMesh {
  BlockIndexList block_indices;        // (z, y, x) order
  std::vector<uint32_t> vertex_begin;  // block_indices.size() + 1
  std::vector<Point> vertices, normals;
  std::vector<Color> colors;
};
namespace detail {
// cg_layer_mesh or cg_layer_mesh_sharded (same arguments), then cg_mesh_fetch
template <class MeshEntry>
inline void meshAndFetch(MeshEntry entry, const TsdfLayer& layer, LayerMesh* mesh,
                         const MeshIntegratorConfig& config, bool only_mesh_updated_blocks) {
  size_t nb = 0, nv = 0;
  check(entry(layer.handle(), config.min_weight, config.use_color ? 1 : 0,
              only_mesh_updated_blocks ? 1 : 0, 0, 0, nullptr, nullptr, nullptr, nullptr, nullptr,
              &nb, &nv));
  mesh->block_indices.resize(nb);
  mesh->vertex_begin.assign(nb + 1, 0);
  mesh->vertices.resize(nv);
  mesh->normals.resize(nv);
  mesh->colors.resize(nv);
  if (nb == 0) return;
  check(cg_mesh_fetch(layer.context(), nb, nv, &mesh->block_indices[0].x, mesh->vertex_begin.data(),
                      nv ? &mesh->vertices[0].x : nullptr, nv ? &mesh->normals[0].x : nullptr,
                      nv ? &mesh->colors[0].r : nullptr));
}
}  // namespace detail
inline void generateMesh(const TsdfLayer& layer, LayerMesh* mesh,
                         const MeshIntegratorConfig& config = MeshIntegratorConfig(),
                         bool only_mesh_updated_blocks = false) {
  detail::meshAndFetch(cg_layer_mesh, layer, mesh, config, only_mesh_updated_blocks);
}
// The same over the sharded global map that getProjectedMapSharded leaves, every rank with its
// owned layer (collective): each rank gets the meshes of its own blocks, byte for byte what
// generateMesh gives for them on the gathered map; the halo blocks are read from the peers.
inline void generateMeshSharded(const TsdfLayer& owned_layer, LayerMesh* mesh,
                                const MeshIntegratorConfig& config = MeshIntegratorConfig(),
                                bool only_mesh_updated_blocks = false) {
  detail::meshAndFetch(cg_layer_mesh_sharded, owned_layer, mesh, config, only_mesh_updated_blocks);
}

// ---- MeshLayer::getConnectedMesh + io::outputMeshAsPly: what saveAndPubCombinedMesh does with a
// file path (server_visualizer.cpp:118-126).  Operates on the mesh the last generateMesh of this
// layer's context left on the device.
struct ConnectedMesh {  // voxblox::Mesh with shared vertices
  std::vector<Point> vertices, normals;
  std::vector<Color> colors;
  std::vector<uint32_t> indices;  // three per triangle
};
inline void getConnectedMesh(const TsdfLayer& layer, ConnectedMesh* mesh) {
  size_t nu = 0, ni = 0;
  check(cg_mesh_connect(layer.context(), 0, 0, nullptr, nullptr, nullptr, nullptr, &nu, &ni));
  mesh->vertices.resize(nu);
  mesh->normals.resize(nu);
  mesh->colors.resize(nu);
  mesh->indices.resize(ni);
  if (ni == 0) return;
  check(cg_mesh_connect(layer.context(), nu, ni, &mesh->vertices[0].x, &mesh->normals[0].x,
                        &mesh->colors[0].r, mesh->indices.data(), &nu, &ni));
}
// voxblox::outputMeshAsPly (io/mesh_ply.h): ascii PLY with vertex colours and triangle faces
inline bool outputMeshAsPly(const std::string& filename, const ConnectedMesh& mesh) {
  FILE* f = std::fopen(filename.c_str(), "w");
  if (!f) return false;
  std::fprintf(f, "ply\nformat ascii 1.0\nelement vertex %zu\nproperty float x\nproperty float y\n"
                  "property float z\nproperty uchar red\nproperty uchar green\nproperty uchar blue\n"
                  "property uchar alpha\nelement face %zu\nproperty list uchar int vertex_indices\n"
                  "end_header\n", mesh.vertices.size(), mesh.indices.size() / 3);
  for (size_t i = 0; i < mesh.vertices.size(); ++i)
    std::fprintf(f, "%f %f %f %d %d %d %d\n", mesh.vertices[i].x, mesh.vertices[i].y,
                 mesh.vertices[i].z, mesh.colors[i].r, mesh.colors[i].g, mesh.colors[i].b,
                 mesh.colors[i].a);
  for (size_t t = 0; t + 2 < mesh.indices.size(); t += 3)
    std::fprintf(f, "3 %u %u %u\n", mesh.indices[t], mesh.indices[t + 1], mesh.indices[t + 2]);
  return std::fclose(f) == 0;
}

// ---- voxblox::EsdfIntegrator / EsdfMap over a device-resident TSDF layer: the client's
// MapServer::updateEsdfBatch (coxgraph/include/coxgraph/client/map_server.h:141-145) and
// publishTraversable's createFreePointcloudFromEsdfLayer (src/client/map_server.cpp:112-113).
// The ESDF stays on the device (in the layer's context) between updateFromTsdfLayerBatch and the
// getters.
struct EsdfVoxel {  // voxblox::EsdfVoxel
  float distance = 0.0f;
  bool observed = false, hallucinated = false, in_queue = false, fixed = false;
  int8_t parent[3] = {0, 0, 0};
};
struct PointXYZI {  // pcl::PointXYZI
  float x, y, z, intensity;
};
class EsdfIntegrator {
 public:
  struct Config : cg_esdf_config {
    Config() { cg_esdf_config_default(this); }
  };
  // EsdfIntegrator(config, tsdf_layer, esdf_layer): the ESDF layer lives on the device
  EsdfIntegrator(const Config& config, const TsdfLayer* tsdf_layer)
      : config_(config), tsdf_layer_(tsdf_layer) {}
  void updateFromTsdfLayerBatch(cg_esdf_stats* stats = nullptr) {
    check(cg_layer_esdf_batch(tsdf_layer_->handle(), &config_, stats));
  }
  // updateFromTsdfLayer: re-solves only the blocks within reach of what changed in the TSDF layer
  // since the ESDF retained in the context was computed; bit-identical to the batch.  Changes are
  // found by content, so `clear_updated_flag` is accepted and ignored (the layer's updated flags
  // belong to the mesher and the serialiser), as min_diff_m is.
  void updateFromTsdfLayer(bool clear_updated_flag = false, cg_esdf_stats* stats = nullptr,
                           cg_esdf_update_stats* update_stats = nullptr) {
    (void)clear_updated_flag;
    check(cg_layer_esdf_update(tsdf_layer_->handle(), &config_, stats, update_stats));
  }
  // Layer<EsdfVoxel>: blocks in (z, y, x) order, 4096 voxels each
  void getEsdfLayer(BlockIndexList* block_indices, std::vector<EsdfVoxel>* voxels) const {
    size_t nb = 0;
    check(cg_esdf_fetch(tsdf_layer_->context(), 0, nullptr, nullptr, nullptr, &nb));
    block_indices->resize(nb);
    voxels->assign(nb * 4096, EsdfVoxel());
    if (nb == 0) return;
    std::vector<float> dist(nb * 4096);
    std::vector<uint32_t> packed(nb * 4096);
    check(cg_esdf_fetch(tsdf_layer_->context(), nb, &(*block_indices)[0].x, dist.data(),
                        packed.data(), nullptr));
    for (size_t i = 0; i < dist.size(); ++i) {
      EsdfVoxel& v = (*voxels)[i];
      const uint32_t w = packed[i];
      v.distance = dist[i];
      v.observed = w & 1u;
      v.hallucinated = w & 2u;
      v.in_queue = w & 4u;
      v.fixed = w & 8u;
      v.parent[0] = static_cast<int8_t>(w >> 24);
      v.parent[1] = static_cast<int8_t>((w >> 16) & 0xFF);
      v.parent[2] = static_cast<int8_t>((w >> 8) & 0xFF);
    }
  }
  // voxblox::createFreePointcloudFromEsdfLayer(esdf_layer, min_distance, &pointcloud)
  void createFreePointcloud(float min_distance, std::vector<PointXYZI>* pointcloud) const {
    size_t n = 0;
    check(cg_esdf_free_points(tsdf_layer_->context(), min_distance, 0, nullptr, &n));
    pointcloud->resize(n);
    if (n) check(cg_esdf_free_points(tsdf_layer_->context(), min_distance, n, &(*pointcloud)[0].x, &n));
  }

 private:
  Config config_;
  const TsdfLayer* tsdf_layer_;
};

// ---- the same map after a pose-graph update, rebuilt only where a moved submap reaches
// (SURVEY §8f N1; the reference re-projects everything, coxgraph_server.h:275-283).  The layer must
// hold getProjectedMap(submap_layers, T_M_S_old); afterwards it is bit-identical to
// getProjectedMap with the moved submaps at T_M_S_new.  Returns which submaps counted as moved.
inline std::vector<uint8_t> reprojectSubmaps(const std::vector<const TsdfLayer*>& submap_layers,
                                             const std::vector<Transformation>& T_M_S_old,
                                             const std::vector<Transformation>& T_M_S_new,
                                             TsdfLayer* projected_layer, float eps_translation = 0.0f,
                                             float eps_rotation = 0.0f,
                                             cg_reproject_stats* stats = nullptr) {
  const size_t n = submap_layers.size();
  if (T_M_S_old.size() != n || T_M_S_new.size() != n)
    fatal_handler()(CG_ERR_INVALID_ARG, "reprojectSubmaps: one old and one new pose per submap expected");
  std::vector<const cg_layer*> handles(n);
  std::vector<float> po(7 * n), pn(7 * n);
  for (size_t i = 0; i < n; ++i) {
    handles[i] = submap_layers[i]->handle();
    std::copy(T_M_S_old[i].data(), T_M_S_old[i].data() + 7, po.begin() + 7 * i);
    std::copy(T_M_S_new[i].data(), T_M_S_new[i].data() + 7, pn.begin() + 7 * i);
  }
  std::vector<uint8_t> changed(n, 0);
  check(cg_reproject_submaps(handles.data(), po.data(), pn.data(), n, eps_translation, eps_rotation,
                             projected_layer->handle(), changed.data(), stats));
  return changed;
}

}  // namespace coxgraph_b200
#endif  // COXGRAPH_B200_HPP_
