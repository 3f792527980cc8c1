// cg_math.cuh — device-side geometry / voxel arithmetic of the TSDF hot path.
//
// Every float operation that decides a voxel or block index, or a voxel value, is written
// here once, in the operation order of upstream voxblox / Eigen / minkindr (SURVEY.md §8a
// R1-R10; reference call sites: coxgraph/include/coxgraph/map_comm/tsdf_recover.h:75,
// coxgraph/src/client/map_server.cpp:67-69).  The library is compiled with -fmad=false
// (no FMA contraction), IEEE division and square root, no flush-to-zero, so results are the
// plain IEEE single-precision ones.
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>

namespace cg {

constexpr float kEps = 1e-6f;  // voxblox kEpsilon / kFloatEpsilon / kCoordinateEpsilon
constexpr int kVps = 16;
constexpr int kVoxelsPerBlock = 4096;
// A default-constructed voxblox::Color: r = g = b = 0 and alpha CG_DEFAULT_ALPHA (255 unless the
// library is built with `make DEFAULT_ALPHA=0` for a fork whose Color() zeroes the alpha as well;
// only alpha bytes depend on it).  Bytes r,g,b,a.
#ifndef CG_DEFAULT_ALPHA
#define CG_DEFAULT_ALPHA 255
#endif
constexpr uint32_t kDefaultColor = static_cast<uint32_t>(CG_DEFAULT_ALPHA) << 24;
constexpr float kDefaultAlpha = static_cast<float>(CG_DEFAULT_ALPHA);

struct V3 {
  float x, y, z;
};
__device__ __forceinline__ V3 v3(float x, float y, float z) { return V3{x, y, z}; }
__device__ __forceinline__ V3 operator+(V3 a, V3 b) { return {a.x + b.x, a.y + b.y, a.z + b.z}; }
__device__ __forceinline__ V3 operator-(V3 a, V3 b) { return {a.x - b.x, a.y - b.y, a.z - b.z}; }
__device__ __forceinline__ V3 operator*(V3 a, float s) { return {a.x * s, a.y * s, a.z * s}; }
__device__ __forceinline__ V3 operator/(V3 a, float s) { return {a.x / s, a.y / s, a.z / s}; }
// Eigen's unrolled 3-element reduction: a0 + (a1 + a2)
__device__ __forceinline__ float dot3(V3 a, V3 b) { return a.x * b.x + (a.y * b.y + a.z * b.z); }
__device__ __forceinline__ float norm3(V3 a) { return sqrtf(dot3(a, a)); }
__device__ __forceinline__ V3 cross3(V3 a, V3 b) {
  return {a.y * b.z - a.z * b.y, a.z * b.x - a.x * b.z, a.x * b.y - a.y * b.x};
}
__device__ __forceinline__ V3 normalized3(V3 a) {
  const float z = dot3(a, a);
  if (z > 0.0f) return a / sqrtf(z);
  return a;
}

// kindr::minimal::QuatTransformation<float>; T[7] = qw qx qy qz tx ty tz
struct Xform {
  float w;
  V3 v;
  V3 t;
};
__host__ __device__ __forceinline__ Xform make_xform(const float* T) {
  Xform X;
  X.w = T[0];
  X.v = V3{T[1], T[2], T[3]};
  X.t = V3{T[4], T[5], T[6]};
  return X;
}
// Eigen QuaternionBase::_transformVector: uv = 2 (q.vec x v); v + w uv + q.vec x uv
__device__ __forceinline__ V3 rotate(float w, V3 qv, V3 p) {
  V3 uv = cross3(qv, p);
  uv = uv + uv;
  const V3 c = cross3(qv, uv);
  return {(p.x + w * uv.x) + c.x, (p.y + w * uv.y) + c.y, (p.z + w * uv.z) + c.z};
}
__device__ __forceinline__ V3 apply(const Xform& T, V3 p) { return rotate(T.w, T.v, p) + T.t; }
__device__ __forceinline__ Xform inverse(const Xform& T) {
  const V3 cv = {-T.v.x, -T.v.y, -T.v.z};
  const V3 r = rotate(T.w, cv, T.t);
  return Xform{T.w, cv, V3{-r.x, -r.y, -r.z}};
}
// inverse() on the host: rotate(w, conj(v), t) spelled out in the same operation order (host code
// is compiled without FMA contraction, see Makefile), so it gives the device's bits
inline Xform inverse_xform_host(const Xform& T) {
  const float w = T.w;
  const V3 cv = V3{-T.v.x, -T.v.y, -T.v.z};
  const V3 t = T.t;
  V3 uv = V3{cv.y * t.z - cv.z * t.y, cv.z * t.x - cv.x * t.z, cv.x * t.y - cv.y * t.x};
  uv = V3{uv.x + uv.x, uv.y + uv.y, uv.z + uv.z};
  const V3 cr = V3{cv.y * uv.z - cv.z * uv.y, cv.z * uv.x - cv.x * uv.z, cv.x * uv.y - cv.y * uv.x};
  const V3 r = V3{(t.x + w * uv.x) + cr.x, (t.y + w * uv.y) + cr.y, (t.z + w * uv.z) + cr.z};
  return Xform{w, cv, V3{-r.x, -r.y, -r.z}};
}

// getGridIndexFromPoint: floor(x * inv + 1e-6)
__device__ __forceinline__ int grid_index(float x, float inv) {
  return __float2int_rd(x * inv + kEps);
}
__device__ __forceinline__ int grid_index_scaled(float x) { return __float2int_rd(x + kEps); }
// getCenterPointFromGridIndex: (idx + 0.5) * grid.  Upstream evaluates in double and rounds
// once; for |idx| < 2^22 the float evaluation below rounds the same exact product once.
__device__ __forceinline__ float center_coord(int idx, float grid) {
  return (static_cast<float>(idx) + 0.5f) * grid;
}

// --- colour: bytes r,g,b,a packed little-endian in a uint32
__device__ __forceinline__ uint32_t pack_rgba(uint32_t r, uint32_t g, uint32_t b, uint32_t a) {
  return r | (g << 8) | (b << 16) | (a << 24);
}
__device__ __forceinline__ uint32_t round_u8(float v) {
  // static_cast<uint8_t>(round(v)), round half away from zero; inputs are in [0, 255]
  return static_cast<uint32_t>(static_cast<int>(roundf(v))) & 255u;
}
// Color::blendTwoColors
__device__ __forceinline__ uint32_t blend_colors(uint32_t c1, float w1, uint32_t c2, float w2) {
  const float total = w1 + w2;
  w1 = w1 / total;
  w2 = w2 / total;
  const float r = static_cast<float>(c1 & 255u) * w1 + static_cast<float>(c2 & 255u) * w2;
  const float g =
      static_cast<float>((c1 >> 8) & 255u) * w1 + static_cast<float>((c2 >> 8) & 255u) * w2;
  const float b =
      static_cast<float>((c1 >> 16) & 255u) * w1 + static_cast<float>((c2 >> 16) & 255u) * w2;
  const float a = static_cast<float>(c1 >> 24) * w1 + static_cast<float>(c2 >> 24) * w2;
  return pack_rgba(round_u8(r), round_u8(g), round_u8(b), round_u8(a));
}

// --- helpers of the sequential bundle fold (MergedTsdfIntegrator::integrateVoxel): the same
// IEEE results as the plain expressions, with a shorter dependent chain.
// num / den with r = RN(1 / den) given: two FMA correction steps give the correctly rounded
// quotient (Markstein's theorem; verified exhaustively-by-sampling in tests/test_gpu_math.py).
__device__ __forceinline__ float div_with_rcp(float num, float den, float r) {
  float q = num * r;
  float e = __fmaf_rn(-den, q, num);
  q = __fmaf_rn(e, r, q);
  e = __fmaf_rn(-den, q, num);
  q = __fmaf_rn(e, r, q);
  return q;
}
// roundf() (half away from zero) for 0 <= v < 2^23, result kept as float
__device__ __forceinline__ float round_half_away_pos(float v) {
  const float t = truncf(v);
  return (v - t >= 0.5f) ? t + 1.0f : t;
}
struct FoldState {
  V3 m;                   // merged_point_C
  float W;                // merged_weight
  float cr, cg, cb, ca;   // merged_color, one integer-valued float per channel
};
__device__ __forceinline__ void fold_reset(FoldState& s) {
  s.m = V3{0.0f, 0.0f, 0.0f};
  s.W = 0.0f;
  s.cr = s.cg = s.cb = 0.0f;
  s.ca = kDefaultAlpha;
}
__device__ __forceinline__ uint32_t fold_color(const FoldState& s) {
  return pack_rgba(static_cast<uint32_t>(s.cr), static_cast<uint32_t>(s.cg),
                   static_cast<uint32_t>(s.cb), static_cast<uint32_t>(s.ca));
}
// one point: merged = (merged * W + p * w) / (W + w); colour = blendTwoColors(colour, W, c, w)
__device__ __forceinline__ void fold_step(FoldState& s, float px, float py, float pz, uint32_t col,
                                          float w) {
  const float Wn = s.W + w;
  const float r = 1.0f / Wn;
  const float a = s.W / Wn;  // blendTwoColors: first_weight /= total
  const float b = w / Wn;    //                 second_weight /= total
  s.m.x = div_with_rcp(s.m.x * s.W + px * w, Wn, r);
  s.m.y = div_with_rcp(s.m.y * s.W + py * w, Wn, r);
  s.m.z = div_with_rcp(s.m.z * s.W + pz * w, Wn, r);
  s.cr = round_half_away_pos(s.cr * a + static_cast<float>(col & 255u) * b);
  s.cg = round_half_away_pos(s.cg * a + static_cast<float>((col >> 8) & 255u) * b);
  s.cb = round_half_away_pos(s.cb * a + static_cast<float>((col >> 16) & 255u) * b);
  s.ca = round_half_away_pos(s.ca * a + static_cast<float>(col >> 24) * b);
  s.W = Wn;
}

// --- R3: voxblox::RayCaster (integrator_utils.cc), indices as int32 (range checked by caller)
struct RayCaster {
  int cx, cy, cz;
  int sx, sy, sz;
  float tnx, tny, tnz;
  float tsx, tsy, tsz;
  unsigned steps;  // ray_length_in_steps; steps + 1 indices are produced
  int ex, ey, ez;  // voxel holding the ray end
  bool valid;
  bool in_range;  // all indices the walk can reach stay inside +-2^19

  __device__ __forceinline__ static int signum(float v) {
    return (v == 0.0f) ? 0 : (v < 0.0f ? -1 : 1);
  }

  __device__ __forceinline__ void init(V3 origin, V3 point_G, bool clearing, bool carving,
                                       float max_ray, float voxel_size_inv, float trunc) {
    const V3 unit_ray = normalized3(point_G - origin);
    V3 ray_start, ray_end;
    if (clearing) {
      float ray_length = norm3(point_G - origin);
      ray_length = fminf(fmaxf(ray_length - trunc, 0.0f), max_ray);
      ray_end = origin + unit_ray * ray_length;
      ray_start = carving ? origin : ray_end;
    } else {
      ray_end = point_G + unit_ray * trunc;
      ray_start = carving ? origin : (point_G - unit_ray * trunc);
    }
    const V3 s = ray_start * voxel_size_inv;
    const V3 e = ray_end * voxel_size_inv;
    valid = !(isnan(s.x) || isnan(s.y) || isnan(s.z) || isnan(e.x) || isnan(e.y) || isnan(e.z));
    const float lim = 524000.0f;  // < 2^19
    in_range = fabsf(s.x) < lim && fabsf(s.y) < lim && fabsf(s.z) < lim && fabsf(e.x) < lim &&
               fabsf(e.y) < lim && fabsf(e.z) < lim;
    if (!valid || !in_range) {
      steps = 0;
      valid = false;
      cx = cy = cz = 0;
      ex = ey = ez = 0;
      sx = sy = sz = 0;
      tnx = tny = tnz = tsx = tsy = tsz = 0.0f;
      return;
    }
    cx = grid_index_scaled(s.x);
    cy = grid_index_scaled(s.y);
    cz = grid_index_scaled(s.z);
    ex = grid_index_scaled(e.x);
    ey = grid_index_scaled(e.y);
    ez = grid_index_scaled(e.z);
    steps = static_cast<unsigned>(abs(ex - cx) + abs(ey - cy) + abs(ez - cz));
    const float rx = e.x - s.x, ry = e.y - s.y, rz = e.z - s.z;
    sx = signum(rx);
    sy = signum(ry);
    sz = signum(rz);
    const float shx = s.x - static_cast<float>(cx);
    const float shy = s.y - static_cast<float>(cy);
    const float shz = s.z - static_cast<float>(cz);
    // upstream's guard (abs(ray) < 0.0) never fires: plain IEEE division, inf/NaN included
    tnx = (static_cast<float>(max(0, sx)) - shx) / rx;
    tny = (static_cast<float>(max(0, sy)) - shy) / ry;
    tnz = (static_cast<float>(max(0, sz)) - shz) / rz;
    tsx = static_cast<float>(sx) / rx;
    tsy = static_cast<float>(sy) / ry;
    tsz = static_cast<float>(sz) / rz;
  }

  // (number of 16^3 blocks the walk crosses) << 32 | number of voxels it visits.  The walk is
  // monotone per axis, so it crosses |delta block index|_1 + 1 blocks when it ends in the end
  // voxel; rounding can make it end one step off (callers allow slack).
  __device__ __forceinline__ unsigned long long packed_counts() const {
    const unsigned nb = static_cast<unsigned>(abs((ex >> 4) - (cx >> 4)) + abs((ey >> 4) - (cy >> 4)) +
                                              abs((ez >> 4) - (cz >> 4))) + 1u;
    return (static_cast<unsigned long long>(nb) << 32) | (steps + 1u);
  }

  // advance to the next voxel (Eigen minCoeff: first coefficient wins ties, NaN in x sticks)
  __device__ __forceinline__ void step() {
    int m = 0;
    float best = tnx;
    if (tny < best) {
      best = tny;
      m = 1;
    }
    if (tnz < best) {
      m = 2;
    }
    if (m == 0) {
      cx += sx;
      tnx += tsx;
    } else if (m == 1) {
      cy += sy;
      tny += tsy;
    } else {
      cz += sz;
      tnz += tsz;
    }
  }
};

// --- R5: integrator parameters and updateTsdfVoxel
struct IntegratorParams {
  float trunc;
  float max_weight;
  float min_ray;
  float max_ray;
  float voxel_size;
  float voxel_size_inv;
  float sparsity_factor;
  int carving;
  int const_weight;
  int allow_clear;
  int weight_dropoff;
  int use_sparsity;
  int order_mode;
  int freespace;
  int anti_grazing;
};

__device__ __forceinline__ float voxel_weight(const IntegratorParams& p, float z_C) {
  if (p.const_weight) return 1.0f;
  const float dz = fabsf(z_C);
  if (dz > kEps) return 1.0f / (dz * dz);
  return 0.0f;
}

// returns false when the point is dropped (R1; non-finite points are dropped as well)
__device__ __forceinline__ bool point_valid(const IntegratorParams& p, V3 pc, bool* clearing) {
  if (!(isfinite(pc.x) && isfinite(pc.y) && isfinite(pc.z))) return false;
  const float d = norm3(pc);
  if (d < p.min_ray) return false;
  if (d > p.max_ray) {
    if (p.allow_clear || p.freespace) {
      *clearing = true;
      return true;
    }
    return false;
  }
  *clearing = p.freespace != 0;
  return true;
}

struct VoxelState {
  float d;
  float w;
  uint32_t c;
};

__device__ __forceinline__ void update_tsdf_voxel(const IntegratorParams& p, V3 origin, V3 point_G,
                                                  V3 center, uint32_t color, float weight,
                                                  VoxelState& v) {
  const V3 v_voxel_origin = center - origin;
  const V3 v_point_origin = point_G - origin;
  const float dist_G = norm3(v_point_origin);
  const float dist_G_V = dot3(v_voxel_origin, v_point_origin) / dist_G;
  const float sdf = dist_G - dist_G_V;
  float updated_weight = weight;
  const float dropoff_epsilon = p.voxel_size;
  if (p.weight_dropoff && sdf < -dropoff_epsilon) {
    updated_weight = weight * (p.trunc + sdf) / (p.trunc - dropoff_epsilon);
    updated_weight = fmaxf(updated_weight, 0.0f);
  }
  if (p.use_sparsity) {
    if (fabsf(sdf) < p.trunc) updated_weight *= p.sparsity_factor;
  }
  const float new_weight = v.w + updated_weight;
  if (new_weight < kEps) return;
  const float new_sdf = (sdf * updated_weight + v.d * v.w) / new_weight;
  if (fabsf(sdf) < p.trunc) v.c = blend_colors(v.c, v.w, color, updated_weight);
  v.d = (new_sdf > 0.0f) ? fminf(p.trunc, new_sdf) : fmaxf(-p.trunc, new_sdf);
  v.w = fminf(p.max_weight, new_weight);
}

// R10 mergeVoxelAIntoVoxelB
__device__ __forceinline__ void merge_voxel(float da, float wa, uint32_t ca, VoxelState& b) {
  const float cw = wa + b.w;
  if (cw > 0.0f) {
    b.d = (da * wa + b.d * b.w) / cw;
    b.c = blend_colors(ca, wa, b.c, b.w);
    b.w = cw;
  }
}

}  // namespace cg
