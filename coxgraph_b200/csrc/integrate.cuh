// integrate.cuh — what the two halves of the integrator share: the front half
// (integrate_front.cu, points -> one ray per bundle), the back half (integrate_back.cu, rays ->
// voxels) and the job driver that runs them (integrate.cu).
#pragma once
#include <stdlib.h>

#include "cg_internal.cuh"

namespace cg {

struct Ray {           // 24 B
  float px, py, pz;    // merged point, global frame
  float weight;        // merged weight
  uint32_t color;      // merged colour
  uint32_t frame_clr;  // frame index in job | clearing << 31 ; 0xFFFFFFFF = no ray
};
constexpr uint32_t kNoRay = 0xFFFFFFFFu;

// Size classes of a length (a bundle's points, a voxel's update list), 4 per octave, largest
// first: the fold and the ordered replay both hand out work longest-first by class.
constexpr int kSizeClasses = 48;
__device__ __forceinline__ int size_class(uint32_t n) {  // descending: class 0 = largest
  if (n == 0) n = 1;
  const int lg = 31 - __clz(n);                                  // floor(log2 n), 0..31
  const int frac = lg >= 2 ? static_cast<int>((n >> (lg - 2)) & 3u) : 0;  // next two bits
  const int c = min(4 * lg + frac, kSizeClasses - 1);
  return kSizeClasses - 1 - c;
}

// MergedTsdfIntegrator's optional anti-grazing (R6): a ray skips every voxel that holds points
// of the same scan (i.e. that is the key of a non-clearing bundle of its frame) except, for a
// non-clearing ray, its own bundle voxel.  The set of bundle voxels is a scratch hash set keyed by
// (frame, voxel relative to the frame's sensor voxel); the front half builds it (k_grazing_build),
// the walk probes it.
struct GrazingSet {
  const unsigned long long* keys;      // open addressing, kEmptyKey = free
  uint32_t mask;
  const unsigned long long* ray_key;   // per ray (= bundle): its own packed bundle voxel
};
__device__ __forceinline__ unsigned long long grazing_key(uint32_t frame, int rx, int ry, int rz) {
  return (static_cast<unsigned long long>(frame) << 42) |
         (static_cast<unsigned long long>(rz & 0x3FFF) << 28) |
         (static_cast<unsigned long long>(ry & 0x3FFF) << 14) |
         static_cast<unsigned long long>(rx & 0x3FFF);
}
__device__ __forceinline__ bool grazing_contains(const GrazingSet& G, unsigned long long key) {
  uint32_t h = hash_key(key) & G.mask;
  for (;;) {
    const unsigned long long k = G.keys[h];
    if (k == key) return true;
    if (k == kEmptyKey) return false;
    h = (h + 1) & G.mask;
  }
}

// ------------------------------------------------------------------ host
inline size_t env_size(const char* name, size_t dflt) {
  const char* s = getenv(name);
  if (!s || !*s) return dflt;
  return static_cast<size_t>(strtoull(s, nullptr, 10));
}

inline int ceil_log2(uint64_t v) {
  int b = 0;
  while ((uint64_t(1) << b) < v) ++b;
  return b;
}

// fills `bytes` (a multiple of 4) at p with `byte`, by a kernel on stream s (integrate.cu)
cudaError_t fill_bytes(void* p, int byte, size_t bytes, cudaStream_t s);

// Front half of frames [f0, f1) of a job (points -> one ray per bundle, R1 / R2 / R6), queued on
// stream `s` into the set `fb`: nothing here touches the layer.  The counters the back half needs
// (rays, voxel visits, segments, key extent, errors) are copied to fb.h_counters at the end; the
// caller synchronises.  *need_split: the bundle keys do not fit, the caller halves the group.
// `d_counts` (depth jobs, else null): the points of job frame f are the first d_counts[f] of its
// slots [offs[f], offs[f + 1]); the rest are holes.
int32_t front_enqueue(cg_context* ctx, FrontBufs& fb, cudaStream_t s, int32_t* d_err,
                      const cg_layer* L, const cg_integrator_config* cfg, const IntegratorParams& P,
                      const float* d_points, const uint8_t* d_colors, const uint64_t* offs,
                      const uint32_t* d_counts, size_t f0, size_t f1, int attempt, bool* need_split);

enum FrontVerdict { kFrontOk, kFrontRetry, kFrontSplit, kFrontFail };

// After the host has synchronised on a front half: book-keeping of the bundle-key box from the
// extent the job measured, and what has to happen next.
FrontVerdict front_digest(cg_context* ctx, const FrontBufs& fb, bool merged, size_t F, int attempt,
                          int32_t* rc);

// The job's poses and frame offsets (relative to its first point) into the set `fb`, queued on
// `stream`.
int32_t upload_frame_tables(FrontBufs& fb, size_t F, const float* h_poses, const uint64_t* offs,
                            cudaStream_t stream);

// Back half of one group: the rays of the set `fb` into the layer, on the context's stream.
int32_t run_back_half(cg_context* ctx, const FrontBufs& fb, cg_layer* L, const IntegratorParams& P,
                      uint32_t num_rays, size_t num_pairs, size_t num_segments,
                      cg_integrate_stats* stats);

// ---- depth jobs (integrate_depth.cu)
// pixels of one depth job at most (F * W * H): the point slots of a job are indexed like a group's
constexpr size_t kMaxDepthJobPixels = 0x7FFFFFF0ull;
// CG_OK, or CG_ERR_INVALID_ARG with the error text naming `who`
int32_t check_depth_camera(const char* who, const cg_depth_camera* cam, size_t F);
size_t depth_pixel_bytes(const cg_depth_camera& cam);
size_t color_pixel_bytes(const cg_depth_camera& cam);
// F frames of images (device memory) -> fb.depth_pts / depth_cols, a slab of W*H slots per frame,
// and fb.depth_counts[f] = kept points of frame f; two kernels on stream s, stage depth_points
int32_t unproject_depth(cg_context* ctx, FrontBufs& fb, const cg_depth_camera& cam, size_t F,
                        const void* d_depth, const uint8_t* d_color, cudaStream_t s);

}  // namespace cg
