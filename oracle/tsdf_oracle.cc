// tsdf_oracle.cc — CPU ORACLE for the coxgraph TSDF hot path.  TEST INFRASTRUCTURE ONLY
// (see tsdf_oracle.h).  PARITY UNPINNED: restates upstream voxblox semantics (the forks the
// reference depends on are not vendored, coxgraph_ssh.rosinstall:1-8,55-58).
//
// Everything here is written against the *published* voxblox algorithm, independently of
// the CUDA implementation under coxgraph_b200/csrc (no shared headers), with the float
// operation order of voxblox/Eigen/minkindr spelled out.  Compile without FMA contraction
// (-ffp-contract=off) so that every rounding step is the IEEE single-precision one.
//
// Section tags R1..R10 follow SURVEY.md §8(a).  Reference call sites:
//   integratePointCloud  : coxgraph/include/coxgraph/map_comm/tsdf_recover.h:75
//   mergeLayerAintoLayerB: coxgraph/src/client/map_server.cpp:67-69,
//                          coxgraph/src/server/visualizer/server_visualizer.cpp:123-126
#include "tsdf_oracle.h"

#include <algorithm>
#include <atomic>
#include <cmath>
#include <cstdlib>
#include <cstring>
#include <deque>
#include <memory>
#include <mutex>
#include <thread>
#include <unordered_map>
#include <unordered_set>
#include <limits>
#include <vector>

namespace {

constexpr float kEps = 1e-6f;  // voxblox kEpsilon == kFloatEpsilon == kCoordinateEpsilon
constexpr int kVps = 16;
constexpr int kVoxelsPerBlock = kVps * kVps * kVps;

// ---------------------------------------------------------------- small vector algebra
struct V3 {
  float x, y, z;
};
inline V3 operator+(V3 a, V3 b) { return {a.x + b.x, a.y + b.y, a.z + b.z}; }
inline V3 operator-(V3 a, V3 b) { return {a.x - b.x, a.y - b.y, a.z - b.z}; }
inline V3 operator*(V3 a, float s) { return {a.x * s, a.y * s, a.z * s}; }
inline V3 operator/(V3 a, float s) { return {a.x / s, a.y / s, a.z / s}; }
// Eigen fixed-size-3 reduction unrolls as a0 + (a1 + a2) (redux_novec_unroller halves).
inline float dot(V3 a, V3 b) { return a.x * b.x + (a.y * b.y + a.z * b.z); }
inline float norm(V3 a) { return std::sqrt(dot(a, a)); }
inline V3 cross(V3 a, V3 b) {
  return {a.y * b.z - a.z * b.y, a.z * b.x - a.x * b.z, a.x * b.y - a.y * b.x};
}
inline V3 normalized(V3 a) {  // Eigen MatrixBase::normalized()
  float z = dot(a, a);
  if (z > 0.0f) return a / std::sqrt(z);
  return a;
}

struct Xform {  // kindr::minimal::QuatTransformationTemplate<float>
  float w;
  V3 v;  // quaternion (w, vec)
  V3 t;
};
inline Xform load_xform(const float T[7]) { return {T[0], {T[1], T[2], T[3]}, {T[4], T[5], T[6]}}; }
// Eigen QuaternionBase::_transformVector
inline V3 rotate(float w, V3 qv, V3 p) {
  V3 uv = cross(qv, p);
  uv = uv + uv;
  V3 c = cross(qv, uv);
  return {(p.x + w * uv.x) + c.x, (p.y + w * uv.y) + c.y, (p.z + w * uv.z) + c.z};
}
inline V3 apply(const Xform& T, V3 p) { return rotate(T.w, T.v, p) + T.t; }  // R2
inline Xform inverse(const Xform& T) {  // (q*, -(q* (x) t))
  V3 cv = {-T.v.x, -T.v.y, -T.v.z};
  V3 r = rotate(T.w, cv, T.t);
  return {T.w, cv, {-r.x, -r.y, -r.z}};
}

// ---------------------------------------------------------------- voxel / colour
// Alpha of a default-constructed voxblox::Color.  Upstream core/color.h is not in the reference
// tree; this restatement takes (0, 0, 0, 255).  A fork whose Color() zeroes the alpha too is matched
// by building with -DORC_DEFAULT_ALPHA=0 (and the library with CG_DEFAULT_ALPHA=0, see the
// Makefiles): only alpha bytes change (voxels that
// were carved before they were coloured, and the vertices taking their colour).
#ifndef ORC_DEFAULT_ALPHA
#define ORC_DEFAULT_ALPHA 255
#endif
struct Color {
  uint8_t r = 0, g = 0, b = 0, a = ORC_DEFAULT_ALPHA;
};
struct Voxel {  // voxblox::TsdfVoxel, 12 bytes
  float distance = 0.0f;
  float weight = 0.0f;
  Color color;
};
static_assert(sizeof(Voxel) == 12, "TsdfVoxel layout");

inline uint8_t round_u8(float v) { return static_cast<uint8_t>(std::round(v)); }
// Color::blendTwoColors
inline Color blend(Color c1, float w1, Color c2, float w2) {
  float total = w1 + w2;
  w1 /= total;
  w2 /= total;
  Color o;
  o.r = round_u8(c1.r * w1 + c2.r * w2);
  o.g = round_u8(c1.g * w1 + c2.g * w2);
  o.b = round_u8(c1.b * w1 + c2.b * w2);
  o.a = round_u8(c1.a * w1 + c2.a * w2);
  return o;
}

// ---------------------------------------------------------------- indices
struct I3 {
  int32_t x, y, z;
  bool operator==(const I3& o) const { return x == o.x && y == o.y && z == o.z; }
  bool operator!=(const I3& o) const { return !(*this == o); }
};
struct L3 {
  int64_t x, y, z;
  bool operator==(const L3& o) const { return x == o.x && y == o.y && z == o.z; }
  bool operator!=(const L3& o) const { return !(*this == o); }
};
struct I3Hash {  // voxblox AnyIndexHash
  size_t operator()(const I3& i) const {
    constexpr size_t sl = 17191, sl2 = sl * sl;
    return static_cast<unsigned int>(i.x + i.y * sl + i.z * sl2);
  }
};
struct L3Hash {  // voxblox LongIndexHash
  size_t operator()(const L3& i) const {
    constexpr size_t sl = 17191, sl2 = sl * sl;
    return static_cast<unsigned int>(i.x + i.y * sl + i.z * sl2);
  }
};
inline bool zyx_less(const L3& a, const L3& b) {
  if (a.z != b.z) return a.z < b.z;
  if (a.y != b.y) return a.y < b.y;
  return a.x < b.x;
}
inline bool zyx_less_i(const I3& a, const I3& b) {
  if (a.z != b.z) return a.z < b.z;
  if (a.y != b.y) return a.y < b.y;
  return a.x < b.x;
}

// getGridIndexFromPoint(point, inv): floor(p*inv + 1e-6)
inline L3 grid_index_long(V3 p, float inv) {
  return {static_cast<int64_t>(std::floor(p.x * inv + kEps)),
          static_cast<int64_t>(std::floor(p.y * inv + kEps)),
          static_cast<int64_t>(std::floor(p.z * inv + kEps))};
}
inline L3 grid_index_long(V3 scaled) {
  return {static_cast<int64_t>(std::floor(scaled.x + kEps)),
          static_cast<int64_t>(std::floor(scaled.y + kEps)),
          static_cast<int64_t>(std::floor(scaled.z + kEps))};
}
inline I3 grid_index_int(V3 p, float inv) {
  return {static_cast<int32_t>(std::floor(p.x * inv + kEps)),
          static_cast<int32_t>(std::floor(p.y * inv + kEps)),
          static_cast<int32_t>(std::floor(p.z * inv + kEps))};
}
// getCenterPointFromGridIndex: (float(idx) + 0.5) * grid_size, evaluated in double and
// rounded once to float (the 0.5 literal is a double in the upstream source).
inline float center_coord(int64_t idx, float grid) {
  return static_cast<float>((static_cast<double>(static_cast<float>(idx)) + 0.5) *
                            static_cast<double>(grid));
}
inline V3 center_point(L3 i, float grid) {
  return {center_coord(i.x, grid), center_coord(i.y, grid), center_coord(i.z, grid)};
}
inline V3 origin_point(I3 i, float grid) {  // getOriginPointFromGridIndex
  return {static_cast<float>(i.x) * grid, static_cast<float>(i.y) * grid,
          static_cast<float>(i.z) * grid};
}
// R4: getBlockIndexFromGlobalVoxelIndex / getLocalFromGlobalVoxelIndex
inline I3 block_of_voxel(L3 v, float vps_inv) {
  return {static_cast<int32_t>(std::floor(static_cast<float>(v.x) * vps_inv)),
          static_cast<int32_t>(std::floor(static_cast<float>(v.y) * vps_inv)),
          static_cast<int32_t>(std::floor(static_cast<float>(v.z) * vps_inv))};
}
inline int local_linear(L3 v) {
  constexpr int64_t offset = int64_t(1) << 31;
  int lx = static_cast<int>((v.x + offset) & (kVps - 1));
  int ly = static_cast<int>((v.y + offset) & (kVps - 1));
  int lz = static_cast<int>((v.z + offset) & (kVps - 1));
  return lx + kVps * (ly + kVps * lz);
}

// ---------------------------------------------------------------- layer
struct Block {
  Voxel voxels[kVoxelsPerBlock];
  bool has_data = false;
  bool updated = false;
};
using BlockMap = std::unordered_map<I3, std::unique_ptr<Block>, I3Hash>;

}  // namespace

struct orc_layer {
  float voxel_size;
  float voxel_size_inv;
  float block_size;
  float block_size_inv;
  float vps_inv;
  BlockMap blocks;
  const Block* find(I3 idx) const {
    auto it = blocks.find(idx);
    return it == blocks.end() ? nullptr : it->second.get();
  }
  Block* find(I3 idx) {
    auto it = blocks.find(idx);
    return it == blocks.end() ? nullptr : it->second.get();
  }
  Block* get_or_create(I3 idx) {
    auto& p = blocks[idx];
    if (!p) p.reset(new Block());
    return p.get();
  }
};

namespace {

// ---------------------------------------------------------------- R3 RayCaster
struct RayCaster {
  L3 curr;
  uint32_t steps = 0;
  uint32_t current_step = 0;
  int sign[3];
  float t_next[3];
  float t_step[3];
  bool valid = true;

  RayCaster(V3 origin, V3 point_G, bool clearing, bool carving, float max_ray,
            float voxel_size_inv, float trunc, bool cast_from_origin = true) {
    const V3 unit_ray = normalized(point_G - origin);
    V3 ray_start, ray_end;
    if (clearing) {
      float ray_length = norm(point_G - origin);
      ray_length = std::min(std::max(ray_length - trunc, 0.0f), max_ray);
      ray_end = origin + unit_ray * ray_length;
      ray_start = carving ? origin : ray_end;
    } else {
      ray_end = point_G + unit_ray * trunc;
      ray_start = carving ? origin : (point_G - unit_ray * trunc);
    }
    const V3 s = ray_start * voxel_size_inv;
    const V3 e = ray_end * voxel_size_inv;
    if (cast_from_origin)
      setup(s, e);
    else
      setup(e, s);
  }

  static int signum(float v) { return (v == 0.0f) ? 0 : (v < 0.0f ? -1 : 1); }

  void setup(V3 start, V3 end) {
    if (std::isnan(start.x) || std::isnan(start.y) || std::isnan(start.z) ||
        std::isnan(end.x) || std::isnan(end.y) || std::isnan(end.z)) {
      valid = false;  // upstream leaves the caster unusable; we emit nothing
      return;
    }
    curr = grid_index_long(start);
    const L3 e = grid_index_long(end);
    const int64_t dx = e.x - curr.x, dy = e.y - curr.y, dz = e.z - curr.z;
    steps = static_cast<uint32_t>(std::llabs(dx) + std::llabs(dy) + std::llabs(dz));
    const float ray[3] = {end.x - start.x, end.y - start.y, end.z - start.z};
    const float shifted[3] = {start.x - static_cast<float>(curr.x),
                              start.y - static_cast<float>(curr.y),
                              start.z - static_cast<float>(curr.z)};
    for (int a = 0; a < 3; ++a) {
      sign[a] = signum(ray[a]);
      const float corrected = static_cast<float>(std::max(0, sign[a]));
      const float dist_to_boundary = corrected - shifted[a];
      // upstream guards with (abs(ray) < 0.0), which is never true: plain IEEE division,
      // inf / NaN included.
      t_next[a] = dist_to_boundary / ray[a];
      t_step[a] = static_cast<float>(sign[a]) / ray[a];
    }
  }

  bool next(L3* out) {
    if (!valid) return false;
    if (current_step++ > steps) return false;
    *out = curr;
    // Eigen minCoeff visitor: res = coeff(0); later coeffs replace it only if (value < res).
    int m = 0;
    float best = t_next[0];
    if (t_next[1] < best) {
      best = t_next[1];
      m = 1;
    }
    if (t_next[2] < best) {
      best = t_next[2];
      m = 2;
    }
    if (m == 0)
      curr.x += sign[0];
    else if (m == 1)
      curr.y += sign[1];
    else
      curr.z += sign[2];
    t_next[m] += t_step[m];
    return true;
  }
};

// ---------------------------------------------------------------- integrator core
struct Cfg {
  orc_integrator_config c;
  float voxel_size, voxel_size_inv, vps_inv;
  std::vector<orc_visit>* trace = nullptr;  // every update_voxel call, in order (single thread)
};

// R1 isPointValid (+ non-finite points are dropped, as voxblox_ros TsdfServer does before
// the integrator ever sees them).
inline bool point_valid(const Cfg& cfg, V3 p, bool freespace, bool* clearing) {
  if (!std::isfinite(p.x) || !std::isfinite(p.y) || !std::isfinite(p.z)) return false;
  const float d = norm(p);
  if (d < cfg.c.min_ray_length_m) return false;
  if (d > cfg.c.max_ray_length_m) {
    if (cfg.c.allow_clear || freespace) {
      *clearing = true;
      return true;
    }
    return false;
  }
  *clearing = freespace;
  return true;
}

inline float voxel_weight(const Cfg& cfg, V3 p_C) {  // getVoxelWeight
  if (cfg.c.use_const_weight) return 1.0f;
  const float dz = std::fabs(p_C.z);
  if (dz > kEps) return 1.0f / (dz * dz);
  return 0.0f;
}

inline float compute_distance(V3 origin, V3 point_G, V3 voxel_center) {
  const V3 v_voxel_origin = voxel_center - origin;
  const V3 v_point_origin = point_G - origin;
  const float dist_G = norm(v_point_origin);
  const float dist_G_V = dot(v_voxel_origin, v_point_origin) / dist_G;
  return dist_G - dist_G_V;
}

// R5 updateTsdfVoxel (the voxel lock is the caller's business)
template <class Lock>
inline void update_voxel(const Cfg& cfg, V3 origin, V3 point_G, L3 gvi, Color color,
                         float weight, Voxel* voxel, Lock&& lock) {
  const V3 center = center_point(gvi, cfg.voxel_size);
  const float sdf = compute_distance(origin, point_G, center);
  const float trunc = cfg.c.default_truncation_distance;
  float updated_weight = weight;
  const float dropoff_epsilon = cfg.voxel_size;
  if (cfg.c.use_weight_dropoff && sdf < -dropoff_epsilon) {
    updated_weight = weight * (trunc + sdf) / (trunc - dropoff_epsilon);
    updated_weight = std::max(updated_weight, 0.0f);
  }
  if (cfg.c.use_sparsity_compensation_factor) {
    if (std::fabs(sdf) < trunc) updated_weight *= cfg.c.sparsity_compensation_factor;
  }
  if (cfg.trace)
    cfg.trace->push_back(orc_visit{static_cast<int32_t>(gvi.x), static_cast<int32_t>(gvi.y),
                                   static_cast<int32_t>(gvi.z), sdf, updated_weight,
                                   {color.r, color.g, color.b, color.a}});
  auto guard = lock(gvi);
  (void)guard;
  const float new_weight = voxel->weight + updated_weight;
  if (new_weight < kEps) return;
  const float new_sdf = (sdf * updated_weight + voxel->distance * voxel->weight) / new_weight;
  if (std::fabs(sdf) < trunc)
    voxel->color = blend(voxel->color, voxel->weight, color, updated_weight);
  voxel->distance = (new_sdf > 0.0f) ? std::min(trunc, new_sdf) : std::max(-trunc, new_sdf);
  voxel->weight = std::min(cfg.c.max_weight, new_weight);
}

struct NoLock {
  int operator()(const L3&) const { return 0; }
};

// MixedThreadSafeIndex: sequential counter k -> point index
struct IndexOrder {
  size_t n, groups;
  int mode;
  IndexOrder(size_t n_, int mode_) : n(n_), groups(n_ / 1024), mode(mode_) {}
  size_t at(size_t k) const {
    if (mode != 0) return k;
    if (groups * 1024 <= k) return k;
    return (k % groups) * 1024 + (k / groups);
  }
};

// Block storage during one integratePointCloud call: existing layer blocks are used in
// place, new ones are collected and committed at the end (updateLayerWithStoredBlocks).
struct CallStorage {
  orc_layer* layer;
  BlockMap temp;
  std::unordered_set<I3, I3Hash> touched;
  explicit CallStorage(orc_layer* l) : layer(l) {}
  Voxel* voxel_ptr(const Cfg& cfg, L3 gvi) {  // allocateStorageAndGetVoxelPtr
    const I3 bi = block_of_voxel(gvi, cfg.vps_inv);
    touched.insert(bi);
    Block* b = layer->find(bi);
    if (!b) {
      auto& p = temp[bi];
      if (!p) p.reset(new Block());
      b = p.get();
    }
    b->updated = true;
    return &b->voxels[local_linear(gvi)];
  }
  void commit() {
    for (auto& kv : temp) layer->blocks[kv.first] = std::move(kv.second);
    temp.clear();
  }
};

struct Bundle {
  L3 key;
  std::vector<size_t> pts;
};

// R6 bundleRays: single-threaded, points visited in index-getter order (as upstream)
void bundle_rays(const Cfg& cfg, const Xform& T, const float* pts, size_t n, bool freespace,
                 std::vector<Bundle>* normal, std::vector<Bundle>* clear) {
  std::unordered_map<L3, size_t, L3Hash> nmap, cmap;
  IndexOrder order(n, cfg.c.integration_order_mode);
  for (size_t k = 0; k < n; ++k) {
    const size_t i = order.at(k);
    const V3 p_C = {pts[3 * i], pts[3 * i + 1], pts[3 * i + 2]};
    bool clearing = false;
    if (!point_valid(cfg, p_C, freespace, &clearing)) continue;
    const V3 p_G = apply(T, p_C);
    const L3 key = grid_index_long(p_G, cfg.voxel_size_inv);
    auto& map = clearing ? cmap : nmap;
    auto* vec = clearing ? clear : normal;
    auto it = map.find(key);
    if (it == map.end()) {
      map.emplace(key, vec->size());
      vec->push_back(Bundle{key, {i}});
    } else {
      (*vec)[it->second].pts.push_back(i);
    }
  }
  // canonical order over bundles (upstream: unordered_map order x thread interleaving)
  auto by_key = [](const Bundle& a, const Bundle& b) { return zyx_less(a.key, b.key); };
  std::sort(normal->begin(), normal->end(), by_key);
  std::sort(clear->begin(), clear->end(), by_key);
}

struct MergedRay {
  V3 point_G;
  Color color;
  float weight;
};

// MergedTsdfIntegrator::integrateVoxel, first half
MergedRay fold_bundle(const Cfg& cfg, const Xform& T, const float* pts, const uint8_t* cols,
                      const Bundle& b, bool clearing) {
  Color merged_color;
  V3 merged_point_C = {0.0f, 0.0f, 0.0f};
  float merged_weight = 0.0f;
  for (size_t i : b.pts) {
    const V3 p_C = {pts[3 * i], pts[3 * i + 1], pts[3 * i + 2]};
    Color c;
    c.r = cols[4 * i];
    c.g = cols[4 * i + 1];
    c.b = cols[4 * i + 2];
    c.a = cols[4 * i + 3];
    const float w = voxel_weight(cfg, p_C);
    if (w < kEps) continue;
    merged_point_C = (merged_point_C * merged_weight + p_C * w) / (merged_weight + w);
    merged_color = blend(merged_color, merged_weight, c, w);
    merged_weight += w;
    if (clearing) break;  // only take first point when clearing
  }
  return {apply(T, merged_point_C), merged_color, merged_weight};
}

template <class Storage, class Lock>
void integrate_bundle(const Cfg& cfg, const Xform& T, const float* pts, const uint8_t* cols,
                      const Bundle& b, bool clearing,
                      const std::unordered_set<L3, L3Hash>* grazing_set, Storage& st,
                      Lock&& lock) {
  if (b.pts.empty()) return;
  const V3 origin = T.t;
  const MergedRay r = fold_bundle(cfg, T, pts, cols, b, clearing);
  RayCaster rc(origin, r.point_G, clearing, cfg.c.voxel_carving_enabled != 0,
               cfg.c.max_ray_length_m, cfg.voxel_size_inv, cfg.c.default_truncation_distance);
  L3 gvi;
  while (rc.next(&gvi)) {
    if (grazing_set) {
      if ((clearing || gvi != b.key) && grazing_set->count(gvi)) continue;
    }
    Voxel* v = st.voxel_ptr(cfg, gvi);
    update_voxel(cfg, origin, r.point_G, gvi, r.color, r.weight, v, lock);
  }
}

int integrate_merged(orc_layer* layer, const Cfg& cfg, const Xform& T, const float* pts,
                     const uint8_t* cols, size_t n, bool freespace, uint64_t* touched) {
  std::vector<Bundle> normal, clear;
  bundle_rays(cfg, T, pts, n, freespace, &normal, &clear);
  std::unordered_set<L3, L3Hash> grazing;
  if (cfg.c.enable_anti_grazing)
    for (const auto& b : normal) grazing.insert(b.key);
  const auto* gs = cfg.c.enable_anti_grazing ? &grazing : nullptr;
  CallStorage st(layer);
  for (const auto& b : normal) integrate_bundle(cfg, T, pts, cols, b, false, gs, st, NoLock());
  st.commit();
  for (const auto& b : clear) integrate_bundle(cfg, T, pts, cols, b, true, gs, st, NoLock());
  st.commit();
  if (touched) *touched = st.touched.size();
  return 0;
}

int integrate_simple(orc_layer* layer, const Cfg& cfg, const Xform& T, const float* pts,
                     const uint8_t* cols, size_t n, bool freespace, uint64_t* touched) {
  CallStorage st(layer);
  IndexOrder order(n, cfg.c.integration_order_mode);
  const V3 origin = T.t;
  for (size_t k = 0; k < n; ++k) {
    const size_t i = order.at(k);
    const V3 p_C = {pts[3 * i], pts[3 * i + 1], pts[3 * i + 2]};
    bool clearing = false;
    if (!point_valid(cfg, p_C, freespace, &clearing)) continue;
    const V3 p_G = apply(T, p_C);
    Color c;
    c.r = cols[4 * i];
    c.g = cols[4 * i + 1];
    c.b = cols[4 * i + 2];
    c.a = cols[4 * i + 3];
    RayCaster rc(origin, p_G, clearing, cfg.c.voxel_carving_enabled != 0,
                 cfg.c.max_ray_length_m, cfg.voxel_size_inv, cfg.c.default_truncation_distance);
    L3 gvi;
    while (rc.next(&gvi)) {
      Voxel* v = st.voxel_ptr(cfg, gvi);
      const float w = voxel_weight(cfg, p_C);
      update_voxel(cfg, origin, p_G, gvi, c, w, v, NoLock());
    }
  }
  st.commit();
  if (touched) *touched = st.touched.size();
  return 0;
}

// FastTsdfIntegrator, one thread, approximate hash sets reset every call
// (clear_checks_every_n_frames = 1).
struct ApproxSet {
  static constexpr size_t kBits = 20;
  std::vector<size_t> slots;
  ApproxSet() : slots(size_t(1) << kBits, ~size_t(0)) {}
  bool replace(const L3& idx) {
    const size_t h = L3Hash()(idx);
    size_t& s = slots[h & ((size_t(1) << kBits) - 1)];
    if (s == h) return false;
    s = h;
    return true;
  }
};

int integrate_fast(orc_layer* layer, const Cfg& cfg, const Xform& T, const float* pts,
                   const uint8_t* cols, size_t n, bool freespace, uint64_t* touched) {
  CallStorage st(layer);
  IndexOrder order(n, cfg.c.integration_order_mode);
  ApproxSet start_set, observed_set;
  const V3 origin = T.t;
  for (size_t k = 0; k < n; ++k) {
    const size_t i = order.at(k);
    const V3 p_C = {pts[3 * i], pts[3 * i + 1], pts[3 * i + 2]};
    bool clearing = false;
    if (!point_valid(cfg, p_C, freespace, &clearing)) continue;
    const V3 p_G = apply(T, p_C);
    Color c;
    c.r = cols[4 * i];
    c.g = cols[4 * i + 1];
    c.b = cols[4 * i + 2];
    c.a = cols[4 * i + 3];
    L3 gvi = grid_index_long(p_G, cfg.c.start_voxel_subsampling_factor * cfg.voxel_size_inv);
    if (!start_set.replace(gvi)) continue;
    RayCaster rc(origin, p_G, clearing, cfg.c.voxel_carving_enabled != 0,
                 cfg.c.max_ray_length_m, cfg.voxel_size_inv, cfg.c.default_truncation_distance,
                 /*cast_from_origin=*/false);
    int64_t collisions = 0;
    while (rc.next(&gvi)) {
      if (!observed_set.replace(gvi))
        ++collisions;
      else
        collisions = 0;
      if (collisions > cfg.c.max_consecutive_ray_collisions) break;
      Voxel* v = st.voxel_ptr(cfg, gvi);
      const float w = voxel_weight(cfg, p_C);
      update_voxel(cfg, origin, p_G, gvi, c, w, v, NoLock());
    }
  }
  st.commit();
  if (touched) *touched = st.touched.size();
  return 0;
}

// ---------------------------------------------------------------- threaded timing variant
struct MtStorage {
  orc_layer* layer;
  BlockMap temp;
  std::mutex temp_mutex;
  explicit MtStorage(orc_layer* l) : layer(l) {}
  Voxel* voxel_ptr(const Cfg& cfg, L3 gvi) {
    const I3 bi = block_of_voxel(gvi, cfg.vps_inv);
    Block* b = layer->find(bi);
    if (!b) {
      std::lock_guard<std::mutex> g(temp_mutex);
      auto& p = temp[bi];
      if (!p) p.reset(new Block());
      b = p.get();
    }
    b->updated = true;
    return &b->voxels[local_linear(gvi)];
  }
  void commit() {
    for (auto& kv : temp) layer->blocks[kv.first] = std::move(kv.second);
    temp.clear();
  }
};
struct StripedLocks {  // voxblox ApproxHashArray<12, std::mutex, ...>
  std::mutex m[4096];
  std::unique_lock<std::mutex> operator()(const L3& i) {
    return std::unique_lock<std::mutex>(m[L3Hash()(i) & 4095]);
  }
};

int integrate_mt(orc_layer* layer, const Cfg& cfg, const Xform& T, const float* pts,
                 const uint8_t* cols, size_t n, bool freespace, int threads) {
  if (threads < 1) threads = 1;
  static StripedLocks locks;
  MtStorage st(layer);
  const V3 origin = T.t;
  if (cfg.c.method == 1) {
    std::vector<Bundle> normal, clear;
    bundle_rays(cfg, T, pts, n, freespace, &normal, &clear);
    for (int pass = 0; pass < 2; ++pass) {
      const auto& list = pass == 0 ? normal : clear;
      std::vector<std::thread> pool;
      for (int t = 0; t < threads; ++t)
        pool.emplace_back([&, t, pass]() {
          for (size_t i = t; i < list.size(); i += threads)
            integrate_bundle(cfg, T, pts, cols, list[i], pass == 1, nullptr, st, locks);
        });
      for (auto& th : pool) th.join();
      st.commit();
    }
    return 0;
  }
  if (cfg.c.method != 0) return -2;  // fast: single thread only in this oracle
  std::atomic<size_t> counter{0};
  IndexOrder order(n, cfg.c.integration_order_mode);
  std::vector<std::thread> pool;
  for (int t = 0; t < threads; ++t)
    pool.emplace_back([&]() {
      size_t k;
      while ((k = counter.fetch_add(1)) < n) {
        const size_t i = order.at(k);
        const V3 p_C = {pts[3 * i], pts[3 * i + 1], pts[3 * i + 2]};
        bool clearing = false;
        if (!point_valid(cfg, p_C, freespace, &clearing)) continue;
        const V3 p_G = apply(T, p_C);
        Color c;
        c.r = cols[4 * i];
        c.g = cols[4 * i + 1];
        c.b = cols[4 * i + 2];
        c.a = cols[4 * i + 3];
        RayCaster rc(origin, p_G, clearing, cfg.c.voxel_carving_enabled != 0,
                     cfg.c.max_ray_length_m, cfg.voxel_size_inv,
                     cfg.c.default_truncation_distance);
        L3 gvi;
        while (rc.next(&gvi)) {
          Voxel* v = st.voxel_ptr(cfg, gvi);
          update_voxel(cfg, origin, p_G, gvi, c, voxel_weight(cfg, p_C), v, locks);
        }
      }
    });
  for (auto& th : pool) th.join();
  st.commit();
  return 0;
}

// ---------------------------------------------------------------- R8/R9 Interpolator
inline I3 block_index_from_coords(const orc_layer& L, V3 p) {
  return grid_index_int(p, L.block_size_inv);
}
inline V3 block_origin(const orc_layer& L, I3 bi) { return origin_point(bi, L.block_size); }
inline V3 voxel_coords(const orc_layer& L, I3 bi, I3 vi) {  // computeCoordinatesFromVoxelIndex
  const V3 o = block_origin(L, bi);
  const V3 c = center_point(L3{vi.x, vi.y, vi.z}, L.voxel_size);
  return o + c;
}
inline int linear_of(I3 v) { return v.x + kVps * (v.y + kVps * v.z); }

// 8x8 table from the SPIE PM159 trilinear formulation used by voxblox
const int kInterpTable[8][8] = {
    {1, 0, 0, 0, 0, 0, 0, 0},   {-1, 0, 0, 0, 1, 0, 0, 0},  {-1, 0, 1, 0, 0, 0, 0, 0},
    {-1, 1, 0, 0, 0, 0, 0, 0},  {1, 0, -1, 0, -1, 0, 1, 0}, {1, -1, -1, 1, 0, 0, 0, 0},
    {1, -1, 0, 0, -1, 1, 0, 0}, {-1, 1, 1, -1, 1, -1, -1, 1}};

inline float interp_member(const float q[8], const float data[8]) {
  // q . (M . data); rows accumulated left to right over the non-zero entries, then the
  // dot product accumulated left to right (order fixed by this oracle, SURVEY R8).
  float acc = 0.0f;
  for (int r = 0; r < 8; ++r) {
    float row = 0.0f;
    bool first = true;
    for (int c = 0; c < 8; ++c) {
      const int m = kInterpTable[r][c];
      if (m == 0) continue;
      const float term = (m > 0) ? data[c] : -data[c];
      row = first ? term : row + term;
      first = false;
    }
    const float prod = q[r] * row;
    acc = (r == 0) ? prod : acc + prod;
  }
  return acc;
}
inline uint8_t trunc_u8(float v) {  // static_cast<uint8_t>(float): truncation; clamped here
  if (!(v > 0.0f)) return 0;
  if (v >= 255.0f) return 255;
  return static_cast<uint8_t>(static_cast<int>(v));
}

bool interp_trilinear(const orc_layer& L, V3 pos, Voxel* out) {
  // setIndexes
  I3 bi = block_index_from_coords(L, pos);
  if (!L.find(bi)) return false;
  const V3 rel = pos - block_origin(L, bi);
  I3 vi = grid_index_int(rel, L.voxel_size_inv);  // un-clamped
  const V3 off = pos - voxel_coords(L, bi, vi);
  int* vip[3] = {&vi.x, &vi.y, &vi.z};
  int* bip[3] = {&bi.x, &bi.y, &bi.z};
  const float offs[3] = {off.x, off.y, off.z};
  for (int a = 0; a < 3; ++a) {
    if (offs[a] < 0.0f) {
      (*vip[a])--;
      if (*vip[a] < 0) {
        (*bip[a])--;
        *vip[a] += kVps;
      }
    }
  }
  static const int kOff[8][3] = {{0, 0, 0}, {0, 0, 1}, {0, 1, 0}, {0, 1, 1},
                                 {1, 0, 0}, {1, 0, 1}, {1, 1, 0}, {1, 1, 1}};
  const Voxel* vox[8];
  float q[8];
  for (int i = 0; i < 8; ++i) {
    // getVoxelsAndQVector: the base block must exist for every neighbour
    const Block* blk = L.find(bi);
    if (!blk) return false;
    I3 nvi = {vi.x + kOff[i][0], vi.y + kOff[i][1], vi.z + kOff[i][2]};
    I3 nbi = bi;
    if (nvi.x >= kVps || nvi.y >= kVps || nvi.z >= kVps) {
      if (nvi.x >= kVps) {
        nbi.x++;
        nvi.x -= kVps;
      }
      if (nvi.y >= kVps) {
        nbi.y++;
        nvi.y -= kVps;
      }
      if (nvi.z >= kVps) {
        nbi.z++;
        nvi.z -= kVps;
      }
      blk = L.find(nbi);
      if (!blk) return false;
    }
    if (i == 0) {  // getQVector
      const V3 vpos = voxel_coords(L, nbi, nvi);
      const V3 o = (pos - vpos) * L.voxel_size_inv;
      q[0] = 1.0f;
      q[1] = o.x;
      q[2] = o.y;
      q[3] = o.z;
      q[4] = o.x * o.y;
      q[5] = o.y * o.z;
      q[6] = o.z * o.x;
      q[7] = o.x * o.y * o.z;
    }
    // The epsilon of getGridIndexFromPoint can leave a voxel index of -1 that the shift above does
    // not touch (pos within 1e-6 of a block face, centre offset >= 0).  Upstream then indexes
    // voxels_[x + 16 (y + 16 z)] with it: inside the array that is a definite (if unintended)
    // voxel and is kept; outside the array it is undefined behaviour — defined here as
    // "not observed", i.e. the trilinear attempt fails and the nearest-neighbour fallback decides.
    const int lin = linear_of(nvi);
    if (lin < 0 || lin >= kVoxelsPerBlock) return false;
    const Voxel& v = blk->voxels[lin];
    vox[i] = &v;
    if (!(v.weight > kEps)) return false;  // utils::isObservedVoxel
  }
  float d[8];
  for (int i = 0; i < 8; ++i) d[i] = vox[i]->distance;
  out->distance = interp_member(q, d);
  for (int i = 0; i < 8; ++i) d[i] = vox[i]->weight;
  out->weight = interp_member(q, d);
  for (int i = 0; i < 8; ++i) d[i] = static_cast<float>(vox[i]->color.r);
  out->color.r = trunc_u8(interp_member(q, d));
  for (int i = 0; i < 8; ++i) d[i] = static_cast<float>(vox[i]->color.g);
  out->color.g = trunc_u8(interp_member(q, d));
  for (int i = 0; i < 8; ++i) d[i] = static_cast<float>(vox[i]->color.b);
  out->color.b = trunc_u8(interp_member(q, d));
  for (int i = 0; i < 8; ++i) d[i] = static_cast<float>(vox[i]->color.a);
  out->color.a = trunc_u8(interp_member(q, d));
  return true;
}

bool interp_nearest(const orc_layer& L, V3 pos, Voxel* out) {  // R9
  const I3 bi = block_index_from_coords(L, pos);
  const Block* blk = L.find(bi);
  if (!blk) return false;
  const V3 rel = pos - block_origin(L, bi);
  I3 vi = grid_index_int(rel, L.voxel_size_inv);
  vi.x = std::max(std::min(vi.x, kVps - 1), 0);
  vi.y = std::max(std::min(vi.y, kVps - 1), 0);
  vi.z = std::max(std::min(vi.z, kVps - 1), 0);
  *out = blk->voxels[linear_of(vi)];
  return out->weight > kEps;
}

// ---------------------------------------------------------------- R7 transformLayer, R10 merge
void candidate_blocks(const orc_layer& in, const Xform& T, float block_size_out,
                      std::vector<I3>* out) {
  std::unordered_set<I3, I3Hash> set;
  const float inv_out = 1.0f / block_size_out;
  const float kDiag = static_cast<float>(std::sqrt(3.0));
  for (const auto& kv : in.blocks) {
    const I3 bi = kv.first;
    const V3 c_in = center_point(L3{bi.x, bi.y, bi.z}, in.block_size);
    const V3 c_out = apply(T, c_in);
    const float offset = kDiag * in.block_size * 0.5f;
    for (float x = c_out.x - offset; x < c_out.x + offset; x += block_size_out)
      for (float y = c_out.y - offset; y < c_out.y + offset; y += block_size_out)
        for (float z = c_out.z - offset; z < c_out.z + offset; z += block_size_out)
          set.insert(grid_index_int(V3{x, y, z}, inv_out));
  }
  out->assign(set.begin(), set.end());
  std::sort(out->begin(), out->end(), zyx_less_i);
}

// resample one candidate block of the output grid; returns has_data
bool resample_block(const orc_layer& in, const orc_layer& grid_out, const Xform& T_in_out, I3 bi,
                    Block* blk) {
  bool has = false;
  for (int lin = 0; lin < kVoxelsPerBlock; ++lin) {
    const I3 vi = {lin % kVps, (lin / kVps) % kVps, lin / (kVps * kVps)};
    const V3 center_out = voxel_coords(grid_out, bi, vi);
    const V3 p = apply(T_in_out, center_out);
    Voxel v;
    if (interp_trilinear(in, p, &v)) {
      blk->voxels[lin] = v;
      has = true;
    } else if (interp_nearest(in, p, &v)) {
      blk->voxels[lin] = v;
      has = true;
    } else {
      // upstream passes the destination voxel itself into getVoxel; a failed nearest
      // lookup that found a block still overwrites it with the unobserved source voxel
      // (v stays default-constructed when no block was found).
      blk->voxels[lin] = v;
    }
  }
  return has;
}

inline void merge_voxel(const Voxel& a, Voxel* b) {  // mergeVoxelAIntoVoxelB
  const float cw = a.weight + b->weight;
  if (cw > 0.0f) {
    b->distance = (a.distance * a.weight + b->distance * b->weight) / cw;
    b->color = blend(a.color, a.weight, b->color, b->weight);
    b->weight = cw;
  }
}

int merge_layers(const orc_layer* A, const Xform& T_B_A, orc_layer* B, int threads,
                 uint64_t* blocks_out) {
  std::vector<I3> cand;
  candidate_blocks(*A, T_B_A, B->block_size, &cand);
  const Xform T_A_B = inverse(T_B_A);
  std::vector<std::unique_ptr<Block>> temp(cand.size());
  std::vector<char> has(cand.size(), 0);
  auto work = [&](size_t lo, size_t hi) {
    for (size_t i = lo; i < hi; ++i) {
      temp[i].reset(new Block());
      has[i] = resample_block(*A, *B, T_A_B, cand[i], temp[i].get()) ? 1 : 0;
    }
  };
  if (threads <= 1) {
    work(0, cand.size());
  } else {
    std::atomic<size_t> next{0};
    std::vector<std::thread> pool;
    for (int t = 0; t < threads; ++t)
      pool.emplace_back([&]() {
        size_t i;
        while ((i = next.fetch_add(8)) < cand.size()) work(i, std::min(cand.size(), i + 8));
      });
    for (auto& th : pool) th.join();
  }
  uint64_t nout = 0;
  for (size_t i = 0; i < cand.size(); ++i) {
    if (!has[i]) continue;  // block removed from the transformed layer
    ++nout;
    Block* dst = B->get_or_create(cand[i]);
    dst->has_data = true;
    dst->updated = true;
    for (int lin = 0; lin < kVoxelsPerBlock; ++lin)
      merge_voxel(temp[i]->voxels[lin], &dst->voxels[lin]);
  }
  if (blocks_out) *blocks_out = nout;
  return 0;
}

Cfg make_cfg(const orc_layer* layer, const orc_integrator_config* c) {
  Cfg cfg;
  cfg.c = *c;
  cfg.voxel_size = layer->voxel_size;
  cfg.voxel_size_inv = layer->voxel_size_inv;
  cfg.vps_inv = layer->vps_inv;
  return cfg;
}

}  // namespace

// ================================================================== C interface
extern "C" {

void orc_default_config(orc_integrator_config* c) {
  c->default_truncation_distance = 0.1f;
  c->max_weight = 10000.0f;
  c->voxel_carving_enabled = 1;
  c->min_ray_length_m = 0.1f;
  c->max_ray_length_m = 5.0f;
  c->use_const_weight = 0;
  c->allow_clear = 1;
  c->use_weight_dropoff = 1;
  c->use_sparsity_compensation_factor = 0;
  c->sparsity_compensation_factor = 1.0f;
  c->enable_anti_grazing = 0;
  c->method = 1;
  c->integration_order_mode = 0;
  c->start_voxel_subsampling_factor = 2.0f;
  c->max_consecutive_ray_collisions = 2;
}

orc_layer* orc_layer_create(float voxel_size, int32_t vps) {
  if (vps != kVps || !(voxel_size > 0.0f)) return nullptr;
  orc_layer* l = new orc_layer();
  l->voxel_size = voxel_size;
  l->voxel_size_inv = 1.0f / voxel_size;
  l->block_size = voxel_size * static_cast<float>(vps);
  l->block_size_inv = 1.0f / l->block_size;
  l->vps_inv = 1.0f / static_cast<float>(vps);
  return l;
}
void orc_layer_destroy(orc_layer* l) { delete l; }
void orc_layer_clear(orc_layer* l) { l->blocks.clear(); }
size_t orc_layer_num_blocks(const orc_layer* l) { return l->blocks.size(); }

void orc_layer_download(const orc_layer* l, int32_t* idx, void* voxels, uint8_t* flags) {
  std::vector<I3> keys;
  keys.reserve(l->blocks.size());
  for (const auto& kv : l->blocks) keys.push_back(kv.first);
  std::sort(keys.begin(), keys.end(), zyx_less_i);
  for (size_t i = 0; i < keys.size(); ++i) {
    const Block* b = l->find(keys[i]);
    if (idx) {
      idx[3 * i] = keys[i].x;
      idx[3 * i + 1] = keys[i].y;
      idx[3 * i + 2] = keys[i].z;
    }
    if (voxels)
      std::memcpy(static_cast<char*>(voxels) + i * sizeof(Voxel) * kVoxelsPerBlock, b->voxels,
                  sizeof(Voxel) * kVoxelsPerBlock);
    if (flags) flags[i] = (b->has_data ? 1 : 0) | (b->updated ? 2 : 0);
  }
}

void orc_layer_upload(orc_layer* l, const int32_t* idx, const void* voxels, const uint8_t* flags,
                      size_t n) {
  for (size_t i = 0; i < n; ++i) {
    Block* b = l->get_or_create(I3{idx[3 * i], idx[3 * i + 1], idx[3 * i + 2]});
    std::memcpy(b->voxels, static_cast<const char*>(voxels) + i * sizeof(Voxel) * kVoxelsPerBlock,
                sizeof(Voxel) * kVoxelsPerBlock);
    b->has_data = flags ? (flags[i] & 1) != 0 : true;
    b->updated = flags ? (flags[i] & 2) != 0 : false;
  }
}

static int32_t integrate_single(orc_layer* layer, const orc_integrator_config* c,
                                const float T[7], const float* pts, const uint8_t* cols,
                                size_t n, int32_t freespace, uint64_t* touched,
                                std::vector<orc_visit>* trace) {
  if (!layer || !c || !T || (n && (!pts || !cols))) return -1;
  Cfg cfg = make_cfg(layer, c);
  cfg.trace = trace;
  const Xform X = load_xform(T);
  switch (c->method) {
    case 0:
      return integrate_simple(layer, cfg, X, pts, cols, n, freespace != 0, touched);
    case 1:
      return integrate_merged(layer, cfg, X, pts, cols, n, freespace != 0, touched);
    case 2:
      return integrate_fast(layer, cfg, X, pts, cols, n, freespace != 0, touched);
  }
  return -2;
}

int32_t orc_integrate_pointcloud(orc_layer* layer, const orc_integrator_config* c,
                                 const float T[7], const float* pts, const uint8_t* cols,
                                 size_t n, int32_t freespace, uint64_t* touched) {
  return integrate_single(layer, c, T, pts, cols, n, freespace, touched, nullptr);
}

int32_t orc_integrate_pointcloud_traced(orc_layer* layer, const orc_integrator_config* c,
                                        const float T[7], const float* pts, const uint8_t* cols,
                                        size_t n, int32_t freespace, uint64_t* touched,
                                        orc_visit** trace, size_t* num_visits) {
  if (!trace || !num_visits) return -1;
  *trace = nullptr;
  *num_visits = 0;
  std::vector<orc_visit> rec;
  const int32_t rc = integrate_single(layer, c, T, pts, cols, n, freespace, touched, &rec);
  if (rc != 0 || rec.empty()) return rc;
  *trace = static_cast<orc_visit*>(std::malloc(rec.size() * sizeof(orc_visit)));
  if (!*trace) return -3;
  std::memcpy(*trace, rec.data(), rec.size() * sizeof(orc_visit));
  *num_visits = rec.size();
  return 0;
}

void orc_trace_free(orc_visit* trace) { std::free(trace); }

int32_t orc_integrate_pointcloud_mt(orc_layer* layer, const orc_integrator_config* c,
                                    const float T[7], const float* pts, const uint8_t* cols,
                                    size_t n, int32_t freespace, int32_t threads) {
  if (!layer || !c || !T || (n && (!pts || !cols))) return -1;
  return integrate_mt(layer, make_cfg(layer, c), load_xform(T), pts, cols, n, freespace != 0,
                      threads);
}

int32_t orc_merge_layer_into_layer(const orc_layer* a, const float T[7], orc_layer* b,
                                   uint64_t* blocks_out) {
  if (!a || !b || !T) return -1;
  return merge_layers(a, load_xform(T), b, 1, blocks_out);
}
int32_t orc_merge_layer_into_layer_mt(const orc_layer* a, const float T[7], orc_layer* b,
                                      int32_t threads, uint64_t* blocks_out) {
  if (!a || !b || !T) return -1;
  return merge_layers(a, load_xform(T), b, threads, blocks_out);
}

int32_t orc_merge_layer_aligned(const orc_layer* a, orc_layer* b) {
  if (!a || !b || a->voxel_size != b->voxel_size) return -1;
  std::vector<I3> keys;
  for (const auto& kv : a->blocks) keys.push_back(kv.first);
  std::sort(keys.begin(), keys.end(), zyx_less_i);
  for (const I3& k : keys) {
    const Block* src = a->find(k);
    Block* dst = b->get_or_create(k);  // allocated even when the source carries no data
    if (!src->has_data) continue;      // Block::mergeBlock
    dst->has_data = true;
    dst->updated = true;
    for (int lin = 0; lin < kVoxelsPerBlock; ++lin) merge_voxel(src->voxels[lin], &dst->voxels[lin]);
  }
  return 0;
}

void orc_transform_point(const float T[7], const float p[3], float out[3]) {
  const V3 r = apply(load_xform(T), V3{p[0], p[1], p[2]});
  out[0] = r.x;
  out[1] = r.y;
  out[2] = r.z;
}
void orc_inverse_transform(const float T[7], float Ti[7]) {
  const Xform i = inverse(load_xform(T));
  Ti[0] = i.w;
  Ti[1] = i.v.x;
  Ti[2] = i.v.y;
  Ti[3] = i.v.z;
  Ti[4] = i.t.x;
  Ti[5] = i.t.y;
  Ti[6] = i.t.z;
}
size_t orc_cast_ray(const float o[3], const float p[3], int32_t clearing, int32_t carving,
                    float max_ray, float vinv, float trunc, int32_t from_origin, int64_t* out,
                    size_t cap) {
  RayCaster rc(V3{o[0], o[1], o[2]}, V3{p[0], p[1], p[2]}, clearing != 0, carving != 0, max_ray,
               vinv, trunc, from_origin != 0);
  size_t n = 0;
  L3 g;
  while (rc.next(&g)) {
    if (n < cap) {
      out[3 * n] = g.x;
      out[3 * n + 1] = g.y;
      out[3 * n + 2] = g.z;
    }
    ++n;
  }
  return n;
}
int32_t orc_interp_voxel(const orc_layer* l, const float pos[3], int32_t interpolate, float* d,
                         float* w, uint8_t rgba[4]) {
  Voxel v;
  const V3 p = {pos[0], pos[1], pos[2]};
  const bool ok = interpolate ? interp_trilinear(*l, p, &v) : interp_nearest(*l, p, &v);
  if (d) *d = v.distance;
  if (w) *w = v.weight;
  if (rgba) {
    rgba[0] = v.color.r;
    rgba[1] = v.color.g;
    rgba[2] = v.color.b;
    rgba[3] = v.color.a;
  }
  return ok ? 1 : 0;
}

}  // extern "C"

// ================================================================== MeshConverter (in-repo code)
// Unlike the voxblox arithmetic above, this part of the path IS in the reference tree:
// coxgraph/include/coxgraph/map_comm/mesh_converter.h.  The restatement follows it line by line,
// including its quirks (edge p0-p2 blends colors[0] with colors[1], :235-236; the observation
// map is keyed by uint8_t, :274).
namespace {

// MeshConverter::interpolateTriangle — mesh_converter.h:211-265
void interpolate_triangle(const V3 tri[3], const Color col[3], float voxel_size,
                          std::vector<V3>* out_pts, std::vector<Color>* out_cols) {
  const V3 p0 = tri[0], p1 = tri[1], p2 = tri[2];
  const V3 t01 = p1 - p0, t02 = p2 - p0, t12 = p2 - p1;
  std::vector<V3> e01, e02, e12;
  std::vector<Color> c01, c02, c12;
  for (float dist = voxel_size; dist < norm(t01); dist += voxel_size) {  // :224-230
    e01.push_back(p0 + (t01 / norm(t01)) * dist);
    c01.push_back(blend(col[0], 1 - dist / norm(t01), col[1], dist / norm(t01)));
  }
  for (float dist = voxel_size; dist < norm(t02); dist += voxel_size) {  // :231-237 (colors[1]: sic)
    e02.push_back(p0 + (t02 / norm(t02)) * dist);
    c02.push_back(blend(col[0], 1 - dist / norm(t02), col[1], dist / norm(t02)));
  }
  for (float dist = voxel_size; dist < norm(t12); dist += voxel_size) {  // :238-244
    e12.push_back(p1 + (t12 / norm(t12)) * dist);
    c12.push_back(blend(col[1], 1 - dist / norm(t12), col[2], dist / norm(t12)));
  }
  e01.push_back(((p0 + p1) + p2) / 3.0f);  // :246
  c01.push_back(blend(col[2], static_cast<float>(1 / 3.0), blend(col[0], 0.5f, col[1], 0.5f),
                      static_cast<float>(2 / 3.0)));  // :247-249
  out_pts->clear();
  out_cols->clear();
  for (const auto* v : {&e01, &e02, &e12}) out_pts->insert(out_pts->end(), v->begin(), v->end());
  for (const auto* v : {&c01, &c02, &c12}) out_cols->insert(out_cols->end(), v->begin(), v->end());
}

}  // namespace

extern "C" {

// MeshConverter::convertToPointCloud (mesh_converter.h:74-172) followed, for every trajectory
// pose, by getNextPointcloud (:186-209): the per-frame clouds TsdfRecover::processMesh
// (tsdf_recover.h:59-99) hands to integratePointCloud.  Returns the total number of points;
// points / colours are written only if capacity_points is large enough.
size_t orc_mesh_to_frames(const orc_mesh* m, float interp_voxel_size, size_t F, const float* poses,
                          const double* stamps, uint64_t* frame_offsets, float* pts_out,
                          uint8_t* cols_out, size_t capacity_points) {
  std::vector<std::vector<V3>> bucket_pts(256);
  std::vector<std::vector<Color>> bucket_cols(256);
  for (size_t b = 0; b < m->num_blocks; ++b) {
    if (!m->block_has_history[b]) continue;  // :87
    const int32_t* index = m->block_index + 3 * b;
    V3 tri[3];
    Color col[3];
    int nt = 0;
    for (uint32_t i = m->vertex_begin[b]; i < m->vertex_begin[b + 1]; ++i) {
      constexpr float point_conv_factor = 2.0f / std::numeric_limits<uint16_t>::max();  // :97-98
      const float mx = (static_cast<float>(m->x[i]) * point_conv_factor +
                        static_cast<float>(index[0])) * m->block_edge_length;
      const float my = (static_cast<float>(m->y[i]) * point_conv_factor +
                        static_cast<float>(index[1])) * m->block_edge_length;
      const float mz = (static_cast<float>(m->z[i]) * point_conv_factor +
                        static_cast<float>(index[2])) * m->block_edge_length;
      tri[nt] = V3{mx, my, mz};
      col[nt] = Color{m->r[i], m->g[i], m->b[i], 255};  // Color(r, g, b): alpha 255
      if (++nt < 3) continue;
      nt = 0;
      std::vector<V3> ipts;
      std::vector<Color> icols;
      interpolate_triangle(tri, col, interp_voxel_size, &ipts, &icols);  // :133-135
      const uint32_t t = i / 3;  // history of the triangle: the one of its last vertex (:112)
      for (uint32_t h = m->hist_begin[t]; h + 1 < m->hist_begin[t + 1]; h += 2)  // :138-142
        for (size_t j = m->hist[h]; j <= m->hist[h + 1]; ++j) {
          const uint8_t key = static_cast<uint8_t>(j);  // std::map<uint8_t, ...>, :274
          auto& bp = bucket_pts[key];
          auto& bc = bucket_cols[key];
          bp.insert(bp.end(), tri, tri + 3);  // :148-160
          bp.insert(bp.end(), ipts.begin(), ipts.end());
          bc.insert(bc.end(), col, col + 3);
          bc.insert(bc.end(), icols.begin(), icols.end());
        }
    }
  }
  size_t total = 0;
  std::vector<int> frame_bucket(F);
  for (size_t i = 0; i < F; ++i) {  // getNextPointcloud, :195-200
    const double id = stamps[i] == stamps[0] ? 0 : std::round((stamps[i] - stamps[0]) / 0.05);
    frame_bucket[i] = static_cast<uint8_t>(static_cast<long long>(id));
    if (frame_offsets) frame_offsets[i] = total;
    total += bucket_pts[frame_bucket[i]].size();
  }
  if (frame_offsets) frame_offsets[F] = total;
  if (!pts_out || !cols_out || capacity_points < total) return total;
  size_t o = 0;
  for (size_t i = 0; i < F; ++i) {
    // T_Submap_C = T_odom_submap_.inverse() * T_G_C with T_odom_submap_ = identity (:50,:202),
    // exact; the cloud is moved into the sensor frame with its inverse (:203-204)
    const Xform Ti = inverse(load_xform(poses + 7 * i));
    const auto& bp = bucket_pts[frame_bucket[i]];
    const auto& bc = bucket_cols[frame_bucket[i]];
    for (size_t k = 0; k < bp.size(); ++k, ++o) {
      const V3 pc = apply(Ti, bp[k]);
      pts_out[3 * o] = pc.x;
      pts_out[3 * o + 1] = pc.y;
      pts_out[3 * o + 2] = pc.z;
      cols_out[4 * o] = bc[k].r;
      cols_out[4 * o + 1] = bc[k].g;
      cols_out[4 * o + 2] = bc[k].b;
      cols_out[4 * o + 3] = bc[k].a;
    }
  }
  return total;
}

}  // extern "C"

// ================================================================== MeshIntegrator / MarchingCubes
// SURVEY §8f N4: what the caller does right after the merge (saveAndPubCombinedMesh ->
// voxblox::MeshIntegrator<TsdfVoxel>::generateMesh, coxgraph/src/server/visualizer/
// server_visualizer.cpp:123-126; client side coxgraph/src/client/map_server.cpp:126-130).
// [EXT] restatement of upstream voxblox mesh/mesh_integrator.h (extractBlockMesh,
// extractMeshInsideBlock, extractMeshOnBorder, updateMeshColor) and mesh/marching_cubes.h
// (meshCube, interpolateEdgeVertices, interpolateVertex, kTriangleTable = the classic marching
// cubes table, kEdgeIndexPairs).  Parity unpinned like the rest of the [EXT] path; pinned by the
// table's own consistency (tests/test_oracle_mesh.py) and analytic plane / sphere cases.
namespace {

const int kTriangleTable[256][16] = {
    {-1, -1, -1, -1, -1, -1, -1, -1, -1, -1, -1, -1, -1, -1, -1, -1},
    {0, 8, 3, -1, -1, -1, -1, -1, -1, -1, -1, -1, -1, -1, -1, -1},
    {0, 1, 9, -1, -1, -1, -1, -1, -1, -1, -1, -1, -1, -1, -1, -1},
    {1, 8, 3, 9, 8, 1, -1, -1, -1, -1, -1, -1, -1, -1, -1, -1},
    {1, 2, 10, -1, -1, -1, -1, -1, -1, -1, -1, -1, -1, -1, -1, -1},
    {0, 8, 3, 1, 2, 10, -1, -1, -1, -1, -1, -1, -1, -1, -1, -1},
    {9, 2, 10, 0, 2, 9, -1, -1, -1, -1, -1, -1, -1, -1, -1, -1},
    {2, 8, 3, 2, 10, 8, 10, 9, 8, -1, -1, -1, -1, -1, -1, -1},
    {3, 11, 2, -1, -1, -1, -1, -1, -1, -1, -1, -1, -1, -1, -1, -1},
    {0, 11, 2, 8, 11, 0, -1, -1, -1, -1, -1, -1, -1, -1, -1, -1},
    {1, 9, 0, 2, 3, 11, -1, -1, -1, -1, -1, -1, -1, -1, -1, -1},
    {1, 11, 2, 1, 9, 11, 9, 8, 11, -1, -1, -1, -1, -1, -1, -1},
    {3, 10, 1, 11, 10, 3, -1, -1, -1, -1, -1, -1, -1, -1, -1, -1},
    {0, 10, 1, 0, 8, 10, 8, 11, 10, -1, -1, -1, -1, -1, -1, -1},
    {3, 9, 0, 3, 11, 9, 11, 10, 9, -1, -1, -1, -1, -1, -1, -1},
    {9, 8, 10, 10, 8, 11, -1, -1, -1, -1, -1, -1, -1, -1, -1, -1},
    {4, 7, 8, -1, -1, -1, -1, -1, -1, -1, -1, -1, -1, -1, -1, -1},
    {4, 3, 0, 7, 3, 4, -1, -1, -1, -1, -1, -1, -1, -1, -1, -1},
    {0, 1, 9, 8, 4, 7, -1, -1, -1, -1, -1, -1, -1, -1, -1, -1},
    {4, 1, 9, 4, 7, 1, 7, 3, 1, -1, -1, -1, -1, -1, -1, -1},
    {1, 2, 10, 8, 4, 7, -1, -1, -1, -1, -1, -1, -1, -1, -1, -1},
    {3, 4, 7, 3, 0, 4, 1, 2, 10, -1, -1, -1, -1, -1, -1, -1},
    {9, 2, 10, 9, 0, 2, 8, 4, 7, -1, -1, -1, -1, -1, -1, -1},
    {2, 10, 9, 2, 9, 7, 2, 7, 3, 7, 9, 4, -1, -1, -1, -1},
    {8, 4, 7, 3, 11, 2, -1, -1, -1, -1, -1, -1, -1, -1, -1, -1},
    {11, 4, 7, 11, 2, 4, 2, 0, 4, -1, -1, -1, -1, -1, -1, -1},
    {9, 0, 1, 8, 4, 7, 2, 3, 11, -1, -1, -1, -1, -1, -1, -1},
    {4, 7, 11, 9, 4, 11, 9, 11, 2, 9, 2, 1, -1, -1, -1, -1},
    {3, 10, 1, 3, 11, 10, 7, 8, 4, -1, -1, -1, -1, -1, -1, -1},
    {1, 11, 10, 1, 4, 11, 1, 0, 4, 7, 11, 4, -1, -1, -1, -1},
    {4, 7, 8, 9, 0, 11, 9, 11, 10, 11, 0, 3, -1, -1, -1, -1},
    {4, 7, 11, 4, 11, 9, 9, 11, 10, -1, -1, -1, -1, -1, -1, -1},
    {9, 5, 4, -1, -1, -1, -1, -1, -1, -1, -1, -1, -1, -1, -1, -1},
    {9, 5, 4, 0, 8, 3, -1, -1, -1, -1, -1, -1, -1, -1, -1, -1},
    {0, 5, 4, 1, 5, 0, -1, -1, -1, -1, -1, -1, -1, -1, -1, -1},
    {8, 5, 4, 8, 3, 5, 3, 1, 5, -1, -1, -1, -1, -1, -1, -1},
    {1, 2, 10, 9, 5, 4, -1, -1, -1, -1, -1, -1, -1, -1, -1, -1},
    {3, 0, 8, 1, 2, 10, 4, 9, 5, -1, -1, -1, -1, -1, -1, -1},
    {5, 2, 10, 5, 4, 2, 4, 0, 2, -1, -1, -1, -1, -1, -1, -1},
    {2, 10, 5, 3, 2, 5, 3, 5, 4, 3, 4, 8, -1, -1, -1, -1},
    {9, 5, 4, 2, 3, 11, -1, -1, -1, -1, -1, -1, -1, -1, -1, -1},
    {0, 11, 2, 0, 8, 11, 4, 9, 5, -1, -1, -1, -1, -1, -1, -1},
    {0, 5, 4, 0, 1, 5, 2, 3, 11, -1, -1, -1, -1, -1, -1, -1},
    {2, 1, 5, 2, 5, 8, 2, 8, 11, 4, 8, 5, -1, -1, -1, -1},
    {10, 3, 11, 10, 1, 3, 9, 5, 4, -1, -1, -1, -1, -1, -1, -1},
    {4, 9, 5, 0, 8, 1, 8, 10, 1, 8, 11, 10, -1, -1, -1, -1},
    {5, 4, 0, 5, 0, 11, 5, 11, 10, 11, 0, 3, -1, -1, -1, -1},
    {5, 4, 8, 5, 8, 10, 10, 8, 11, -1, -1, -1, -1, -1, -1, -1},
    {9, 7, 8, 5, 7, 9, -1, -1, -1, -1, -1, -1, -1, -1, -1, -1},
    {9, 3, 0, 9, 5, 3, 5, 7, 3, -1, -1, -1, -1, -1, -1, -1},
    {0, 7, 8, 0, 1, 7, 1, 5, 7, -1, -1, -1, -1, -1, -1, -1},
    {1, 5, 3, 3, 5, 7, -1, -1, -1, -1, -1, -1, -1, -1, -1, -1},
    {9, 7, 8, 9, 5, 7, 10, 1, 2, -1, -1, -1, -1, -1, -1, -1},
    {10, 1, 2, 9, 5, 0, 5, 3, 0, 5, 7, 3, -1, -1, -1, -1},
    {8, 0, 2, 8, 2, 5, 8, 5, 7, 10, 5, 2, -1, -1, -1, -1},
    {2, 10, 5, 2, 5, 3, 3, 5, 7, -1, -1, -1, -1, -1, -1, -1},
    {7, 9, 5, 7, 8, 9, 3, 11, 2, -1, -1, -1, -1, -1, -1, -1},
    {9, 5, 7, 9, 7, 2, 9, 2, 0, 2, 7, 11, -1, -1, -1, -1},
    {2, 3, 11, 0, 1, 8, 1, 7, 8, 1, 5, 7, -1, -1, -1, -1},
    {11, 2, 1, 11, 1, 7, 7, 1, 5, -1, -1, -1, -1, -1, -1, -1},
    {9, 5, 8, 8, 5, 7, 10, 1, 3, 10, 3, 11, -1, -1, -1, -1},
    {5, 7, 0, 5, 0, 9, 7, 11, 0, 1, 0, 10, 11, 10, 0, -1},
    {11, 10, 0, 11, 0, 3, 10, 5, 0, 8, 0, 7, 5, 7, 0, -1},
    {11, 10, 5, 7, 11, 5, -1, -1, -1, -1, -1, -1, -1, -1, -1, -1},
    {10, 6, 5, -1, -1, -1, -1, -1, -1, -1, -1, -1, -1, -1, -1, -1},
    {0, 8, 3, 5, 10, 6, -1, -1, -1, -1, -1, -1, -1, -1, -1, -1},
    {9, 0, 1, 5, 10, 6, -1, -1, -1, -1, -1, -1, -1, -1, -1, -1},
    {1, 8, 3, 1, 9, 8, 5, 10, 6, -1, -1, -1, -1, -1, -1, -1},
    {1, 6, 5, 2, 6, 1, -1, -1, -1, -1, -1, -1, -1, -1, -1, -1},
    {1, 6, 5, 1, 2, 6, 3, 0, 8, -1, -1, -1, -1, -1, -1, -1},
    {9, 6, 5, 9, 0, 6, 0, 2, 6, -1, -1, -1, -1, -1, -1, -1},
    {5, 9, 8, 5, 8, 2, 5, 2, 6, 3, 2, 8, -1, -1, -1, -1},
    {2, 3, 11, 10, 6, 5, -1, -1, -1, -1, -1, -1, -1, -1, -1, -1},
    {11, 0, 8, 11, 2, 0, 10, 6, 5, -1, -1, -1, -1, -1, -1, -1},
    {0, 1, 9, 2, 3, 11, 5, 10, 6, -1, -1, -1, -1, -1, -1, -1},
    {5, 10, 6, 1, 9, 2, 9, 11, 2, 9, 8, 11, -1, -1, -1, -1},
    {6, 3, 11, 6, 5, 3, 5, 1, 3, -1, -1, -1, -1, -1, -1, -1},
    {0, 8, 11, 0, 11, 5, 0, 5, 1, 5, 11, 6, -1, -1, -1, -1},
    {3, 11, 6, 0, 3, 6, 0, 6, 5, 0, 5, 9, -1, -1, -1, -1},
    {6, 5, 9, 6, 9, 11, 11, 9, 8, -1, -1, -1, -1, -1, -1, -1},
    {5, 10, 6, 4, 7, 8, -1, -1, -1, -1, -1, -1, -1, -1, -1, -1},
    {4, 3, 0, 4, 7, 3, 6, 5, 10, -1, -1, -1, -1, -1, -1, -1},
    {1, 9, 0, 5, 10, 6, 8, 4, 7, -1, -1, -1, -1, -1, -1, -1},
    {10, 6, 5, 1, 9, 7, 1, 7, 3, 7, 9, 4, -1, -1, -1, -1},
    {6, 1, 2, 6, 5, 1, 4, 7, 8, -1, -1, -1, -1, -1, -1, -1},
    {1, 2, 5, 5, 2, 6, 3, 0, 4, 3, 4, 7, -1, -1, -1, -1},
    {8, 4, 7, 9, 0, 5, 0, 6, 5, 0, 2, 6, -1, -1, -1, -1},
    {7, 3, 9, 7, 9, 4, 3, 2, 9, 5, 9, 6, 2, 6, 9, -1},
    {3, 11, 2, 7, 8, 4, 10, 6, 5, -1, -1, -1, -1, -1, -1, -1},
    {5, 10, 6, 4, 7, 2, 4, 2, 0, 2, 7, 11, -1, -1, -1, -1},
    {0, 1, 9, 4, 7, 8, 2, 3, 11, 5, 10, 6, -1, -1, -1, -1},
    {9, 2, 1, 9, 11, 2, 9, 4, 11, 7, 11, 4, 5, 10, 6, -1},
    {8, 4, 7, 3, 11, 5, 3, 5, 1, 5, 11, 6, -1, -1, -1, -1},
    {5, 1, 11, 5, 11, 6, 1, 0, 11, 7, 11, 4, 0, 4, 11, -1},
    {0, 5, 9, 0, 6, 5, 0, 3, 6, 11, 6, 3, 8, 4, 7, -1},
    {6, 5, 9, 6, 9, 11, 4, 7, 9, 7, 11, 9, -1, -1, -1, -1},
    {10, 4, 9, 6, 4, 10, -1, -1, -1, -1, -1, -1, -1, -1, -1, -1},
    {4, 10, 6, 4, 9, 10, 0, 8, 3, -1, -1, -1, -1, -1, -1, -1},
    {10, 0, 1, 10, 6, 0, 6, 4, 0, -1, -1, -1, -1, -1, -1, -1},
    {8, 3, 1, 8, 1, 6, 8, 6, 4, 6, 1, 10, -1, -1, -1, -1},
    {1, 4, 9, 1, 2, 4, 2, 6, 4, -1, -1, -1, -1, -1, -1, -1},
    {3, 0, 8, 1, 2, 9, 2, 4, 9, 2, 6, 4, -1, -1, -1, -1},
    {0, 2, 4, 4, 2, 6, -1, -1, -1, -1, -1, -1, -1, -1, -1, -1},
    {8, 3, 2, 8, 2, 4, 4, 2, 6, -1, -1, -1, -1, -1, -1, -1},
    {10, 4, 9, 10, 6, 4, 11, 2, 3, -1, -1, -1, -1, -1, -1, -1},
    {0, 8, 2, 2, 8, 11, 4, 9, 10, 4, 10, 6, -1, -1, -1, -1},
    {3, 11, 2, 0, 1, 6, 0, 6, 4, 6, 1, 10, -1, -1, -1, -1},
    {6, 4, 1, 6, 1, 10, 4, 8, 1, 2, 1, 11, 8, 11, 1, -1},
    {9, 6, 4, 9, 3, 6, 9, 1, 3, 11, 6, 3, -1, -1, -1, -1},
    {8, 11, 1, 8, 1, 0, 11, 6, 1, 9, 1, 4, 6, 4, 1, -1},
    {3, 11, 6, 3, 6, 0, 0, 6, 4, -1, -1, -1, -1, -1, -1, -1},
    {6, 4, 8, 11, 6, 8, -1, -1, -1, -1, -1, -1, -1, -1, -1, -1},
    {7, 10, 6, 7, 8, 10, 8, 9, 10, -1, -1, -1, -1, -1, -1, -1},
    {0, 7, 3, 0, 10, 7, 0, 9, 10, 6, 7, 10, -1, -1, -1, -1},
    {10, 6, 7, 1, 10, 7, 1, 7, 8, 1, 8, 0, -1, -1, -1, -1},
    {10, 6, 7, 10, 7, 1, 1, 7, 3, -1, -1, -1, -1, -1, -1, -1},
    {1, 2, 6, 1, 6, 8, 1, 8, 9, 8, 6, 7, -1, -1, -1, -1},
    {2, 6, 9, 2, 9, 1, 6, 7, 9, 0, 9, 3, 7, 3, 9, -1},
    {7, 8, 0, 7, 0, 6, 6, 0, 2, -1, -1, -1, -1, -1, -1, -1},
    {7, 3, 2, 6, 7, 2, -1, -1, -1, -1, -1, -1, -1, -1, -1, -1},
    {2, 3, 11, 10, 6, 8, 10, 8, 9, 8, 6, 7, -1, -1, -1, -1},
    {2, 0, 7, 2, 7, 11, 0, 9, 7, 6, 7, 10, 9, 10, 7, -1},
    {1, 8, 0, 1, 7, 8, 1, 10, 7, 6, 7, 10, 2, 3, 11, -1},
    {11, 2, 1, 11, 1, 7, 10, 6, 1, 6, 7, 1, -1, -1, -1, -1},
    {8, 9, 6, 8, 6, 7, 9, 1, 6, 11, 6, 3, 1, 3, 6, -1},
    {0, 9, 1, 11, 6, 7, -1, -1, -1, -1, -1, -1, -1, -1, -1, -1},
    {7, 8, 0, 7, 0, 6, 3, 11, 0, 11, 6, 0, -1, -1, -1, -1},
    {7, 11, 6, -1, -1, -1, -1, -1, -1, -1, -1, -1, -1, -1, -1, -1},
    {7, 6, 11, -1, -1, -1, -1, -1, -1, -1, -1, -1, -1, -1, -1, -1},
    {3, 0, 8, 11, 7, 6, -1, -1, -1, -1, -1, -1, -1, -1, -1, -1},
    {0, 1, 9, 11, 7, 6, -1, -1, -1, -1, -1, -1, -1, -1, -1, -1},
    {8, 1, 9, 8, 3, 1, 11, 7, 6, -1, -1, -1, -1, -1, -1, -1},
    {10, 1, 2, 6, 11, 7, -1, -1, -1, -1, -1, -1, -1, -1, -1, -1},
    {1, 2, 10, 3, 0, 8, 6, 11, 7, -1, -1, -1, -1, -1, -1, -1},
    {2, 9, 0, 2, 10, 9, 6, 11, 7, -1, -1, -1, -1, -1, -1, -1},
    {6, 11, 7, 2, 10, 3, 10, 8, 3, 10, 9, 8, -1, -1, -1, -1},
    {7, 2, 3, 6, 2, 7, -1, -1, -1, -1, -1, -1, -1, -1, -1, -1},
    {7, 0, 8, 7, 6, 0, 6, 2, 0, -1, -1, -1, -1, -1, -1, -1},
    {2, 7, 6, 2, 3, 7, 0, 1, 9, -1, -1, -1, -1, -1, -1, -1},
    {1, 6, 2, 1, 8, 6, 1, 9, 8, 8, 7, 6, -1, -1, -1, -1},
    {10, 7, 6, 10, 1, 7, 1, 3, 7, -1, -1, -1, -1, -1, -1, -1},
    {10, 7, 6, 1, 7, 10, 1, 8, 7, 1, 0, 8, -1, -1, -1, -1},
    {0, 3, 7, 0, 7, 10, 0, 10, 9, 6, 10, 7, -1, -1, -1, -1},
    {7, 6, 10, 7, 10, 8, 8, 10, 9, -1, -1, -1, -1, -1, -1, -1},
    {6, 8, 4, 11, 8, 6, -1, -1, -1, -1, -1, -1, -1, -1, -1, -1},
    {3, 6, 11, 3, 0, 6, 0, 4, 6, -1, -1, -1, -1, -1, -1, -1},
    {8, 6, 11, 8, 4, 6, 9, 0, 1, -1, -1, -1, -1, -1, -1, -1},
    {9, 4, 6, 9, 6, 3, 9, 3, 1, 11, 3, 6, -1, -1, -1, -1},
    {6, 8, 4, 6, 11, 8, 2, 10, 1, -1, -1, -1, -1, -1, -1, -1},
    {1, 2, 10, 3, 0, 11, 0, 6, 11, 0, 4, 6, -1, -1, -1, -1},
    {4, 11, 8, 4, 6, 11, 0, 2, 9, 2, 10, 9, -1, -1, -1, -1},
    {10, 9, 3, 10, 3, 2, 9, 4, 3, 11, 3, 6, 4, 6, 3, -1},
    {8, 2, 3, 8, 4, 2, 4, 6, 2, -1, -1, -1, -1, -1, -1, -1},
    {0, 4, 2, 4, 6, 2, -1, -1, -1, -1, -1, -1, -1, -1, -1, -1},
    {1, 9, 0, 2, 3, 4, 2, 4, 6, 4, 3, 8, -1, -1, -1, -1},
    {1, 9, 4, 1, 4, 2, 2, 4, 6, -1, -1, -1, -1, -1, -1, -1},
    {8, 1, 3, 8, 6, 1, 8, 4, 6, 6, 10, 1, -1, -1, -1, -1},
    {10, 1, 0, 10, 0, 6, 6, 0, 4, -1, -1, -1, -1, -1, -1, -1},
    {4, 6, 3, 4, 3, 8, 6, 10, 3, 0, 3, 9, 10, 9, 3, -1},
    {10, 9, 4, 6, 10, 4, -1, -1, -1, -1, -1, -1, -1, -1, -1, -1},
    {4, 9, 5, 7, 6, 11, -1, -1, -1, -1, -1, -1, -1, -1, -1, -1},
    {0, 8, 3, 4, 9, 5, 11, 7, 6, -1, -1, -1, -1, -1, -1, -1},
    {5, 0, 1, 5, 4, 0, 7, 6, 11, -1, -1, -1, -1, -1, -1, -1},
    {11, 7, 6, 8, 3, 4, 3, 5, 4, 3, 1, 5, -1, -1, -1, -1},
    {9, 5, 4, 10, 1, 2, 7, 6, 11, -1, -1, -1, -1, -1, -1, -1},
    {6, 11, 7, 1, 2, 10, 0, 8, 3, 4, 9, 5, -1, -1, -1, -1},
    {7, 6, 11, 5, 4, 10, 4, 2, 10, 4, 0, 2, -1, -1, -1, -1},
    {3, 4, 8, 3, 5, 4, 3, 2, 5, 10, 5, 2, 11, 7, 6, -1},
    {7, 2, 3, 7, 6, 2, 5, 4, 9, -1, -1, -1, -1, -1, -1, -1},
    {9, 5, 4, 0, 8, 6, 0, 6, 2, 6, 8, 7, -1, -1, -1, -1},
    {3, 6, 2, 3, 7, 6, 1, 5, 0, 5, 4, 0, -1, -1, -1, -1},
    {6, 2, 8, 6, 8, 7, 2, 1, 8, 4, 8, 5, 1, 5, 8, -1},
    {9, 5, 4, 10, 1, 6, 1, 7, 6, 1, 3, 7, -1, -1, -1, -1},
    {1, 6, 10, 1, 7, 6, 1, 0, 7, 8, 7, 0, 9, 5, 4, -1},
    {4, 0, 10, 4, 10, 5, 0, 3, 10, 6, 10, 7, 3, 7, 10, -1},
    {7, 6, 10, 7, 10, 8, 5, 4, 10, 4, 8, 10, -1, -1, -1, -1},
    {6, 9, 5, 6, 11, 9, 11, 8, 9, -1, -1, -1, -1, -1, -1, -1},
    {3, 6, 11, 0, 6, 3, 0, 5, 6, 0, 9, 5, -1, -1, -1, -1},
    {0, 11, 8, 0, 5, 11, 0, 1, 5, 5, 6, 11, -1, -1, -1, -1},
    {6, 11, 3, 6, 3, 5, 5, 3, 1, -1, -1, -1, -1, -1, -1, -1},
    {1, 2, 10, 9, 5, 11, 9, 11, 8, 11, 5, 6, -1, -1, -1, -1},
    {0, 11, 3, 0, 6, 11, 0, 9, 6, 5, 6, 9, 1, 2, 10, -1},
    {11, 8, 5, 11, 5, 6, 8, 0, 5, 10, 5, 2, 0, 2, 5, -1},
    {6, 11, 3, 6, 3, 5, 2, 10, 3, 10, 5, 3, -1, -1, -1, -1},
    {5, 8, 9, 5, 2, 8, 5, 6, 2, 3, 8, 2, -1, -1, -1, -1},
    {9, 5, 6, 9, 6, 0, 0, 6, 2, -1, -1, -1, -1, -1, -1, -1},
    {1, 5, 8, 1, 8, 0, 5, 6, 8, 3, 8, 2, 6, 2, 8, -1},
    {1, 5, 6, 2, 1, 6, -1, -1, -1, -1, -1, -1, -1, -1, -1, -1},
    {1, 3, 6, 1, 6, 10, 3, 8, 6, 5, 6, 9, 8, 9, 6, -1},
    {10, 1, 0, 10, 0, 6, 9, 5, 0, 5, 6, 0, -1, -1, -1, -1},
    {0, 3, 8, 5, 6, 10, -1, -1, -1, -1, -1, -1, -1, -1, -1, -1},
    {10, 5, 6, -1, -1, -1, -1, -1, -1, -1, -1, -1, -1, -1, -1, -1},
    {11, 5, 10, 7, 5, 11, -1, -1, -1, -1, -1, -1, -1, -1, -1, -1},
    {11, 5, 10, 11, 7, 5, 8, 3, 0, -1, -1, -1, -1, -1, -1, -1},
    {5, 11, 7, 5, 10, 11, 1, 9, 0, -1, -1, -1, -1, -1, -1, -1},
    {10, 7, 5, 10, 11, 7, 9, 8, 1, 8, 3, 1, -1, -1, -1, -1},
    {11, 1, 2, 11, 7, 1, 7, 5, 1, -1, -1, -1, -1, -1, -1, -1},
    {0, 8, 3, 1, 2, 7, 1, 7, 5, 7, 2, 11, -1, -1, -1, -1},
    {9, 7, 5, 9, 2, 7, 9, 0, 2, 2, 11, 7, -1, -1, -1, -1},
    {7, 5, 2, 7, 2, 11, 5, 9, 2, 3, 2, 8, 9, 8, 2, -1},
    {2, 5, 10, 2, 3, 5, 3, 7, 5, -1, -1, -1, -1, -1, -1, -1},
    {8, 2, 0, 8, 5, 2, 8, 7, 5, 10, 2, 5, -1, -1, -1, -1},
    {9, 0, 1, 5, 10, 3, 5, 3, 7, 3, 10, 2, -1, -1, -1, -1},
    {9, 8, 2, 9, 2, 1, 8, 7, 2, 10, 2, 5, 7, 5, 2, -1},
    {1, 3, 5, 3, 7, 5, -1, -1, -1, -1, -1, -1, -1, -1, -1, -1},
    {0, 8, 7, 0, 7, 1, 1, 7, 5, -1, -1, -1, -1, -1, -1, -1},
    {9, 0, 3, 9, 3, 5, 5, 3, 7, -1, -1, -1, -1, -1, -1, -1},
    {9, 8, 7, 5, 9, 7, -1, -1, -1, -1, -1, -1, -1, -1, -1, -1},
    {5, 8, 4, 5, 10, 8, 10, 11, 8, -1, -1, -1, -1, -1, -1, -1},
    {5, 0, 4, 5, 11, 0, 5, 10, 11, 11, 3, 0, -1, -1, -1, -1},
    {0, 1, 9, 8, 4, 10, 8, 10, 11, 10, 4, 5, -1, -1, -1, -1},
    {10, 11, 4, 10, 4, 5, 11, 3, 4, 9, 4, 1, 3, 1, 4, -1},
    {2, 5, 1, 2, 8, 5, 2, 11, 8, 4, 5, 8, -1, -1, -1, -1},
    {0, 4, 11, 0, 11, 3, 4, 5, 11, 2, 11, 1, 5, 1, 11, -1},
    {0, 2, 5, 0, 5, 9, 2, 11, 5, 4, 5, 8, 11, 8, 5, -1},
    {9, 4, 5, 2, 11, 3, -1, -1, -1, -1, -1, -1, -1, -1, -1, -1},
    {2, 5, 10, 3, 5, 2, 3, 4, 5, 3, 8, 4, -1, -1, -1, -1},
    {5, 10, 2, 5, 2, 4, 4, 2, 0, -1, -1, -1, -1, -1, -1, -1},
    {3, 10, 2, 3, 5, 10, 3, 8, 5, 4, 5, 8, 0, 1, 9, -1},
    {5, 10, 2, 5, 2, 4, 1, 9, 2, 9, 4, 2, -1, -1, -1, -1},
    {8, 4, 5, 8, 5, 3, 3, 5, 1, -1, -1, -1, -1, -1, -1, -1},
    {0, 4, 5, 1, 0, 5, -1, -1, -1, -1, -1, -1, -1, -1, -1, -1},
    {8, 4, 5, 8, 5, 3, 9, 0, 5, 0, 3, 5, -1, -1, -1, -1},
    {9, 4, 5, -1, -1, -1, -1, -1, -1, -1, -1, -1, -1, -1, -1, -1},
    {4, 11, 7, 4, 9, 11, 9, 10, 11, -1, -1, -1, -1, -1, -1, -1},
    {0, 8, 3, 4, 9, 7, 9, 11, 7, 9, 10, 11, -1, -1, -1, -1},
    {1, 10, 11, 1, 11, 4, 1, 4, 0, 7, 4, 11, -1, -1, -1, -1},
    {3, 1, 4, 3, 4, 8, 1, 10, 4, 7, 4, 11, 10, 11, 4, -1},
    {4, 11, 7, 9, 11, 4, 9, 2, 11, 9, 1, 2, -1, -1, -1, -1},
    {9, 7, 4, 9, 11, 7, 9, 1, 11, 2, 11, 1, 0, 8, 3, -1},
    {11, 7, 4, 11, 4, 2, 2, 4, 0, -1, -1, -1, -1, -1, -1, -1},
    {11, 7, 4, 11, 4, 2, 8, 3, 4, 3, 2, 4, -1, -1, -1, -1},
    {2, 9, 10, 2, 7, 9, 2, 3, 7, 7, 4, 9, -1, -1, -1, -1},
    {9, 10, 7, 9, 7, 4, 10, 2, 7, 8, 7, 0, 2, 0, 7, -1},
    {3, 7, 10, 3, 10, 2, 7, 4, 10, 1, 10, 0, 4, 0, 10, -1},
    {1, 10, 2, 8, 7, 4, -1, -1, -1, -1, -1, -1, -1, -1, -1, -1},
    {4, 9, 1, 4, 1, 7, 7, 1, 3, -1, -1, -1, -1, -1, -1, -1},
    {4, 9, 1, 4, 1, 7, 0, 8, 1, 8, 7, 1, -1, -1, -1, -1},
    {4, 0, 3, 7, 4, 3, -1, -1, -1, -1, -1, -1, -1, -1, -1, -1},
    {4, 8, 7, -1, -1, -1, -1, -1, -1, -1, -1, -1, -1, -1, -1, -1},
    {9, 10, 8, 10, 11, 8, -1, -1, -1, -1, -1, -1, -1, -1, -1, -1},
    {3, 0, 9, 3, 9, 11, 11, 9, 10, -1, -1, -1, -1, -1, -1, -1},
    {0, 1, 10, 0, 10, 8, 8, 10, 11, -1, -1, -1, -1, -1, -1, -1},
    {3, 1, 10, 11, 3, 10, -1, -1, -1, -1, -1, -1, -1, -1, -1, -1},
    {1, 2, 11, 1, 11, 9, 9, 11, 8, -1, -1, -1, -1, -1, -1, -1},
    {3, 0, 9, 3, 9, 11, 1, 2, 9, 2, 11, 9, -1, -1, -1, -1},
    {0, 2, 11, 8, 0, 11, -1, -1, -1, -1, -1, -1, -1, -1, -1, -1},
    {3, 2, 11, -1, -1, -1, -1, -1, -1, -1, -1, -1, -1, -1, -1, -1},
    {2, 3, 8, 2, 8, 10, 10, 8, 9, -1, -1, -1, -1, -1, -1, -1},
    {9, 10, 2, 0, 9, 2, -1, -1, -1, -1, -1, -1, -1, -1, -1, -1},
    {2, 3, 8, 2, 8, 10, 0, 1, 8, 1, 10, 8, -1, -1, -1, -1},
    {1, 10, 2, -1, -1, -1, -1, -1, -1, -1, -1, -1, -1, -1, -1, -1},
    {1, 3, 8, 9, 1, 8, -1, -1, -1, -1, -1, -1, -1, -1, -1, -1},
    {0, 9, 1, -1, -1, -1, -1, -1, -1, -1, -1, -1, -1, -1, -1, -1},
    {0, 3, 8, -1, -1, -1, -1, -1, -1, -1, -1, -1, -1, -1, -1, -1},
    {-1, -1, -1, -1, -1, -1, -1, -1, -1, -1, -1, -1, -1, -1, -1, -1}
};
const int kEdgeIndexPairs[12][2] = {{0, 1}, {1, 2}, {2, 3}, {3, 0}, {4, 5}, {5, 6},
                                    {6, 7}, {7, 4}, {0, 4}, {1, 5}, {2, 6}, {3, 7}};
// cube_index_offsets_ (columns = corners)
const int kCubeOffsets[8][3] = {{0, 0, 0}, {1, 0, 0}, {1, 1, 0}, {0, 1, 0},
                                {0, 0, 1}, {1, 0, 1}, {1, 1, 1}, {0, 1, 1}};

struct MeshOut {
  std::vector<V3> vertices, normals;
  std::vector<Color> colors;
};

// MarchingCubes::interpolateVertex
inline V3 mc_interpolate_vertex(V3 v1, V3 v2, float sdf1, float sdf2) {
  const float kMinSdfDifference = 1e-6f;
  const float sdf_diff = sdf1 - sdf2;
  if (std::fabs(sdf_diff) >= kMinSdfDifference) {
    const float t = sdf1 / sdf_diff;
    return v1 + (v2 - v1) * t;
  }
  return (v1 + v2) * 0.5f;
}

// MarchingCubes::meshCube
void mc_mesh_cube(const V3 corner_coords[8], const float corner_sdf[8], MeshOut* mesh) {
  int index = 0;  // calculateVertexConfiguration
  for (int i = 0; i < 8; ++i)
    if (corner_sdf[i] < 0.0f) index |= 1 << i;
  V3 edge_coords[12] = {};
  for (int e = 0; e < 12; ++e) {  // interpolateEdgeVertices
    const int a = kEdgeIndexPairs[e][0], b = kEdgeIndexPairs[e][1];
    if ((corner_sdf[a] < 0 && corner_sdf[b] >= 0) || (corner_sdf[a] >= 0 && corner_sdf[b] < 0))
      edge_coords[e] = mc_interpolate_vertex(corner_coords[a], corner_coords[b], corner_sdf[a],
                                             corner_sdf[b]);
  }
  const int* row = kTriangleTable[index];
  for (int c = 0; row[c] != -1; c += 3) {
    const V3 p0 = edge_coords[row[c + 2]], p1 = edge_coords[row[c + 1]], p2 = edge_coords[row[c]];
    mesh->vertices.push_back(p0);
    mesh->vertices.push_back(p1);
    mesh->vertices.push_back(p2);
    const V3 n = normalized(cross(p1 - p0, p2 - p0));
    for (int k = 0; k < 3; ++k) mesh->normals.push_back(n);
  }
}

// extractMeshInsideBlock / extractMeshOnBorder for the cube whose corner 0 is voxel `vi`
void mc_extract_cube(const orc_layer& L, I3 bi, const Block& blk, I3 vi, float min_weight,
                     MeshOut* mesh) {
  const V3 coords = voxel_coords(L, bi, vi);
  V3 corner_coords[8];
  float corner_sdf[8];
  for (int i = 0; i < 8; ++i) {
    I3 ci = {vi.x + kCubeOffsets[i][0], vi.y + kCubeOffsets[i][1], vi.z + kCubeOffsets[i][2]};
    const Block* src = &blk;
    if (ci.x >= kVps || ci.y >= kVps || ci.z >= kVps) {  // a different block
      I3 nb = bi;
      if (ci.x >= kVps) { nb.x += 1; ci.x -= kVps; }
      if (ci.y >= kVps) { nb.y += 1; ci.y -= kVps; }
      if (ci.z >= kVps) { nb.z += 1; ci.z -= kVps; }
      src = L.find(nb);
      if (!src) return;  // all_neighbors_observed = false
    }
    const Voxel& v = src->voxels[linear_of(ci)];
    if (v.weight <= min_weight) return;  // utils::getSdfIfValid
    corner_sdf[i] = v.distance;
    corner_coords[i] = coords + V3{kCubeOffsets[i][0] * L.voxel_size, kCubeOffsets[i][1] * L.voxel_size,
                                   kCubeOffsets[i][2] * L.voxel_size};
  }
  mc_mesh_cube(corner_coords, corner_sdf, mesh);
}

// MeshIntegrator::extractBlockMesh + updateMeshColor
void mc_block_mesh(const orc_layer& L, I3 bi, const Block& blk, float min_weight, bool use_color,
                   MeshOut* mesh) {
  const size_t first = mesh->vertices.size();
  I3 v;
  for (v.x = 0; v.x < kVps - 1; ++v.x)
    for (v.y = 0; v.y < kVps - 1; ++v.y)
      for (v.z = 0; v.z < kVps - 1; ++v.z) mc_extract_cube(L, bi, blk, v, min_weight, mesh);
  v.x = kVps - 1;  // max X plane
  for (v.z = 0; v.z < kVps; ++v.z)
    for (v.y = 0; v.y < kVps; ++v.y) mc_extract_cube(L, bi, blk, v, min_weight, mesh);
  v.y = kVps - 1;  // max Y plane
  for (v.z = 0; v.z < kVps; ++v.z)
    for (v.x = 0; v.x < kVps - 1; ++v.x) mc_extract_cube(L, bi, blk, v, min_weight, mesh);
  v.z = kVps - 1;  // max Z plane
  for (v.y = 0; v.y < kVps - 1; ++v.y)
    for (v.x = 0; v.x < kVps - 1; ++v.x) mc_extract_cube(L, bi, blk, v, min_weight, mesh);
  mesh->colors.resize(mesh->vertices.size());
  if (!use_color) return;
  const V3 origin = block_origin(L, bi);
  for (size_t i = first; i < mesh->vertices.size(); ++i) {  // nearest-neighbour colour
    const V3 vertex = mesh->vertices[i];
    const I3 vi = grid_index_int(vertex - origin, L.voxel_size_inv);  // computeVoxelIndexFromCoordinates
    const Voxel* vox = nullptr;
    if (vi.x >= 0 && vi.x < kVps && vi.y >= 0 && vi.y < kVps && vi.z >= 0 && vi.z < kVps) {
      vox = &blk.voxels[linear_of(vi)];
    } else {
      // getBlockPtrByCoordinates(vertex)->getVoxelByCoordinates(vertex): clamped voxel index.
      // (The reference dereferences a null pointer if that block is missing; here: no colour.)
      const I3 nbi = block_index_from_coords(L, vertex);
      const Block* nb = L.find(nbi);
      if (nb) {
        I3 nv = grid_index_int(vertex - block_origin(L, nbi), L.voxel_size_inv);
        nv.x = std::max(std::min(nv.x, kVps - 1), 0);
        nv.y = std::max(std::min(nv.y, kVps - 1), 0);
        nv.z = std::max(std::min(nv.z, kVps - 1), 0);
        vox = &nb->voxels[linear_of(nv)];
      }
    }
    if (vox && vox->weight > min_weight) mesh->colors[i] = vox->color;  // utils::getColorIfValid
  }
}

}  // namespace

extern "C" {

size_t orc_layer_mesh(const orc_layer* l, float min_weight, int32_t use_color, int32_t only_updated,
                      uint32_t* vertex_begin, float* vertices, float* normals, uint8_t* colors,
                      size_t capacity_vertices) {
  std::vector<I3> keys;
  keys.reserve(l->blocks.size());
  for (const auto& kv : l->blocks) keys.push_back(kv.first);
  std::sort(keys.begin(), keys.end(), zyx_less_i);
  MeshOut mesh;
  for (size_t b = 0; b < keys.size(); ++b) {
    if (vertex_begin) vertex_begin[b] = static_cast<uint32_t>(mesh.vertices.size());
    const Block* blk = l->find(keys[b]);
    if (only_updated && !blk->updated) continue;
    mc_block_mesh(*l, keys[b], *blk, min_weight, use_color != 0, &mesh);
  }
  const size_t n = mesh.vertices.size();
  if (vertex_begin) vertex_begin[keys.size()] = static_cast<uint32_t>(n);
  if (n > capacity_vertices) return n;
  for (size_t i = 0; i < n; ++i) {
    if (vertices) {
      vertices[3 * i] = mesh.vertices[i].x;
      vertices[3 * i + 1] = mesh.vertices[i].y;
      vertices[3 * i + 2] = mesh.vertices[i].z;
    }
    if (normals) {
      normals[3 * i] = mesh.normals[i].x;
      normals[3 * i + 1] = mesh.normals[i].y;
      normals[3 * i + 2] = mesh.normals[i].z;
    }
    if (colors) {
      colors[4 * i] = mesh.colors[i].r;
      colors[4 * i + 1] = mesh.colors[i].g;
      colors[4 * i + 2] = mesh.colors[i].b;
      colors[4 * i + 3] = mesh.colors[i].a;
    }
  }
  return n;
}

const int* orc_triangle_table(void) { return &kTriangleTable[0][0]; }

size_t orc_connect_mesh(const float* vertices, size_t n, uint32_t* out_indices,
                        uint32_t* first_old_index) {
  std::unordered_map<L3, size_t, L3Hash> uniques;  // LongIndexHashMapType<size_t>
  const float threshold = 1e-10f;                  // approximate_vertex_proximity_threshold
  const double threshold_inv = 1.0 / static_cast<double>(threshold);
  size_t new_vertex_index = 0;
  for (size_t i = 0; i < n; ++i) {
    const L3 cell = {static_cast<int64_t>(std::round(static_cast<double>(vertices[3 * i]) * threshold_inv)),
                     static_cast<int64_t>(std::round(static_cast<double>(vertices[3 * i + 1]) * threshold_inv)),
                     static_cast<int64_t>(std::round(static_cast<double>(vertices[3 * i + 2]) * threshold_inv))};
    auto it = uniques.find(cell);
    if (it == uniques.end()) {
      uniques.emplace(cell, new_vertex_index);
      if (first_old_index) first_old_index[new_vertex_index] = static_cast<uint32_t>(i);
      out_indices[i] = static_cast<uint32_t>(new_vertex_index++);
    } else {
      out_indices[i] = static_cast<uint32_t>(it->second);
    }
  }
  return new_vertex_index;
}

}  // extern "C"

// ================================================================ ESDF (SURVEY §8f N4, second half)
// voxblox::EsdfIntegrator::updateFromTsdfLayerBatch as called by the client's MapServer
// (coxgraph/include/coxgraph/client/map_server.h:141-145 <- coxgraph/src/client/map_server.cpp:99)
// and voxblox::createFreePointcloudFromEsdfLayer (coxgraph/src/client/map_server.cpp:112-113).
// [EXT] upstream voxblox integrator/esdf_integrator.cc, utils/bucket_queue.h,
// utils/neighbor_tools.h; PARITY UNPINNED like the rest of this file.  Sequential, in upstream's
// order of work: blocks in (z, y, x) order (upstream: hash-map order), voxels by linear index,
// then the bucketed open queue.  `parent` follows the queue order and is order-dependent upstream.
namespace {

struct EsdfVoxel {  // voxblox::EsdfVoxel
  float distance = 0.0f;
  bool observed = false;
  bool hallucinated = false;
  bool in_queue = false;
  bool fixed = false;
  int8_t parent[3] = {0, 0, 0};
};
struct EsdfBlock {
  EsdfVoxel voxels[kVoxelsPerBlock];
};

// NeighborhoodLookupTables (26-connectivity): 6 faces, 12 edges, 8 corners; kDistances in voxels
struct Neighbor {
  int dx, dy, dz;
  float dist;
};
std::vector<Neighbor> make_neighbors() {
  std::vector<Neighbor> n;
  const float s2 = std::sqrt(2.0f), s3 = std::sqrt(3.0f);
  for (int order = 1; order <= 3; ++order)
    for (int dz = -1; dz <= 1; ++dz)
      for (int dy = -1; dy <= 1; ++dy)
        for (int dx = -1; dx <= 1; ++dx)
          if (std::abs(dx) + std::abs(dy) + std::abs(dz) == order)
            n.push_back({dx, dy, dz, order == 1 ? 1.0f : order == 2 ? s2 : s3});
  return n;
}

// utils/bucket_queue.h: num_buckets FIFO queues over |priority| in [0, max_val]
struct BucketQueue {
  std::vector<std::deque<L3>> buckets;
  int num_buckets = 0, last = 0;
  double max_val = 0.0;
  size_t count = 0;
  void set(int n, double max_value) {
    num_buckets = n;
    max_val = max_value;
    buckets.assign(static_cast<size_t>(n), {});
    last = 0;
    count = 0;
  }
  void push(const L3& key, double value) {
    if (value > max_val) value = max_val;
    int b = static_cast<int>(std::floor(std::abs(value) / max_val * (num_buckets - 1)));
    if (b >= num_buckets) b = num_buckets - 1;
    if (b < last) last = b;
    buckets[static_cast<size_t>(b)].push_back(key);
    ++count;
  }
  bool empty() const { return count == 0; }
  L3 pop_front() {
    while (buckets[static_cast<size_t>(last)].empty() && last < num_buckets - 1) ++last;
    L3 k = buckets[static_cast<size_t>(last)].front();
    buckets[static_cast<size_t>(last)].pop_front();
    --count;
    return k;
  }
};

inline float signum(float x) { return x == 0.0f ? 0.0f : (x < 0.0f ? -1.0f : 1.0f); }

struct EsdfMap {
  std::unordered_map<I3, std::unique_ptr<EsdfBlock>, I3Hash> blocks;
  EsdfVoxel* voxel(const L3& g) {  // Layer::getVoxelPtrByGlobalIndex
    const I3 b = {static_cast<int32_t>(g.x >> 4), static_cast<int32_t>(g.y >> 4),
                  static_cast<int32_t>(g.z >> 4)};
    auto it = blocks.find(b);
    if (it == blocks.end()) return nullptr;
    return &it->second->voxels[(g.x & 15) + 16 * ((g.y & 15) + 16 * (g.z & 15))];
  }
};

}  // namespace

struct orc_esdf {
  EsdfMap map;
  std::vector<I3> keys;  // (z, y, x) order
  float voxel_size = 0.0f, block_size = 0.0f;
  uint64_t updates = 0;
};

extern "C" {

void orc_esdf_default_config(orc_esdf_config* c) {
  c->max_distance_m = 2.0f;
  c->default_distance_m = 2.0f;
  c->min_distance_m = 0.2f;
  c->min_diff_m = 0.001f;
  c->min_weight = 1e-6f;
  c->num_buckets = 20;
  c->multi_queue = 0;
  c->add_occupied_crust = 0;
}

orc_esdf* orc_esdf_batch(const orc_layer* tsdf, const orc_esdf_config* cfg) {
  static const std::vector<Neighbor> kNeighbors = make_neighbors();
  orc_esdf* E = new orc_esdf();
  E->voxel_size = tsdf->voxel_size;
  E->block_size = tsdf->block_size;
  const float vs = tsdf->voxel_size;
  BucketQueue open;
  open.set(cfg->num_buckets, cfg->max_distance_m);
  for (const auto& kv : tsdf->blocks) E->keys.push_back(kv.first);
  std::sort(E->keys.begin(), E->keys.end(), zyx_less_i);
  EsdfMap& M = E->map;

  // EsdfIntegrator::updateVoxelFromNeighbors: lower |distance| of a fresh voxel from the
  // neighbours already in the map
  auto update_from_neighbors = [&](const L3& g, EsdfVoxel* v) -> bool {
    bool updated = false;
    for (const Neighbor& nb : kNeighbors) {
      EsdfVoxel* n = M.voxel({g.x + nb.dx, g.y + nb.dy, g.z + nb.dz});
      if (!n || !n->observed || n->hallucinated) continue;
      const float d = nb.dist * vs;
      if (v->distance > 0.0f && n->distance > 0.0f) {
        if (n->distance + d + cfg->min_diff_m < v->distance) {
          v->distance = n->distance + d;
          v->parent[0] = static_cast<int8_t>(nb.dx);
          v->parent[1] = static_cast<int8_t>(nb.dy);
          v->parent[2] = static_cast<int8_t>(nb.dz);
          updated = true;
        }
      } else if (v->distance < 0.0f && n->distance < 0.0f) {
        if (n->distance - d - cfg->min_diff_m > v->distance) {
          v->distance = n->distance - d;
          v->parent[0] = static_cast<int8_t>(nb.dx);
          v->parent[1] = static_cast<int8_t>(nb.dy);
          v->parent[2] = static_cast<int8_t>(nb.dz);
          updated = true;
        }
      }
    }
    return updated;
  };

  // updateFromTsdfBlocks(all allocated blocks, incremental = false)
  for (const I3& bi : E->keys) {
    const Block* tb = tsdf->find(bi);
    auto& eb = M.blocks[bi];
    if (!eb) eb.reset(new EsdfBlock());
    for (int lin = 0; lin < kVoxelsPerBlock; ++lin) {
      const Voxel& tv = tb->voxels[lin];
      EsdfVoxel& ev = eb->voxels[lin];
      if (tv.weight < cfg->min_weight) {
        if (cfg->add_occupied_crust) {
          ev.distance = -cfg->default_distance_m;
          ev.observed = true;
          ev.hallucinated = true;
          ev.fixed = false;
        }
        continue;
      }
      const L3 g = {int64_t(bi.x) * 16 + (lin & 15), int64_t(bi.y) * 16 + ((lin >> 4) & 15),
                    int64_t(bi.z) * 16 + (lin >> 8)};
      const bool tsdf_fixed = std::abs(tv.distance) < cfg->min_distance_m;  // isFixed
      if (tsdf_fixed) {
        ev.distance = tv.distance;
        ev.observed = true;
        ev.hallucinated = false;
        ev.fixed = true;
        ev.parent[0] = ev.parent[1] = ev.parent[2] = 0;
        ev.in_queue = true;
        open.push(g, ev.distance);
      } else {
        ev.distance = signum(tv.distance) * cfg->default_distance_m;
        ev.observed = true;
        ev.hallucinated = false;
        ev.fixed = false;
        ev.parent[0] = ev.parent[1] = ev.parent[2] = 0;
        if (update_from_neighbors(g, &ev)) {
          ev.in_queue = true;
          open.push(g, ev.distance);
        }
      }
    }
  }
  // processRaiseSet: nothing to raise in a batch rebuild.  processOpenSet:
  while (!open.empty()) {
    const L3 g = open.pop_front();
    EsdfVoxel* v = M.voxel(g);
    v->in_queue = false;
    if (!v->observed || v->distance >= cfg->max_distance_m || v->distance <= -cfg->max_distance_m)
      continue;
    for (const Neighbor& nb : kNeighbors) {
      const L3 ng = {g.x + nb.dx, g.y + nb.dy, g.z + nb.dz};
      EsdfVoxel* n = M.voxel(ng);
      if (!n || !n->observed || n->fixed) continue;
      const float d = nb.dist * vs;
      bool lowered = false;
      if (v->distance > 0.0f && n->distance > 0.0f) {  // both outside the surface
        if (v->distance + d + cfg->min_diff_m < n->distance) {
          n->distance = v->distance + d;
          lowered = true;
        }
      } else if (v->distance < 0.0f && n->distance < 0.0f) {  // both inside
        if (v->distance - d - cfg->min_diff_m > n->distance) {
          n->distance = v->distance - d;
          lowered = true;
        }
      }
      if (lowered) {
        ++E->updates;
        n->parent[0] = static_cast<int8_t>(-nb.dx);
        n->parent[1] = static_cast<int8_t>(-nb.dy);
        n->parent[2] = static_cast<int8_t>(-nb.dz);
        if (cfg->multi_queue || !n->in_queue) {
          open.push(ng, n->distance);
          n->in_queue = true;
        }
      }
    }
  }
  return E;
}

void orc_esdf_destroy(orc_esdf* e) { delete e; }
size_t orc_esdf_num_blocks(const orc_esdf* e) { return e->keys.size(); }
uint64_t orc_esdf_updates(const orc_esdf* e) { return e->updates; }

void orc_esdf_download(const orc_esdf* e, int32_t* block_idx_xyz, float* distance, uint8_t* flags,
                       int8_t* parent) {
  for (size_t b = 0; b < e->keys.size(); ++b) {
    const I3 k = e->keys[b];
    if (block_idx_xyz) {
      block_idx_xyz[3 * b] = k.x;
      block_idx_xyz[3 * b + 1] = k.y;
      block_idx_xyz[3 * b + 2] = k.z;
    }
    const EsdfBlock& blk = *e->map.blocks.find(k)->second;
    for (int i = 0; i < kVoxelsPerBlock; ++i) {
      const EsdfVoxel& v = blk.voxels[i];
      const size_t o = b * kVoxelsPerBlock + static_cast<size_t>(i);
      if (distance) distance[o] = v.distance;
      if (flags)
        flags[o] = static_cast<uint8_t>((v.observed ? 1 : 0) | (v.hallucinated ? 2 : 0) |
                                        (v.in_queue ? 4 : 0) | (v.fixed ? 8 : 0));
      if (parent) {
        parent[3 * o] = v.parent[0];
        parent[3 * o + 1] = v.parent[1];
        parent[3 * o + 2] = v.parent[2];
      }
    }
  }
}

// createFreePointcloudFromEsdfLayer (voxblox_ros ptcloud_vis.h): observed voxels with
// distance >= min_distance, as (x, y, z, intensity = distance); blocks in (z, y, x) order
size_t orc_esdf_free_points(const orc_esdf* e, float min_distance, float* xyzi, size_t capacity) {
  size_t n = 0;
  for (const I3& k : e->keys) {
    const EsdfBlock& blk = *e->map.blocks.find(k)->second;
    const V3 origin = origin_point(k, e->block_size);
    for (int i = 0; i < kVoxelsPerBlock; ++i) {
      const EsdfVoxel& v = blk.voxels[i];
      if (!(v.observed && v.distance >= min_distance)) continue;
      if (xyzi && n < capacity) {
        // Block::computeCoordinatesFromVoxelIndex: origin + getCenterPointFromGridIndex
        xyzi[4 * n] = origin.x + center_coord(i & 15, e->voxel_size);
        xyzi[4 * n + 1] = origin.y + center_coord((i >> 4) & 15, e->voxel_size);
        xyzi[4 * n + 2] = origin.z + center_coord(i >> 8, e->voxel_size);
        xyzi[4 * n + 3] = v.distance;
      }
      ++n;
    }
  }
  return n;
}

}  // extern "C"
