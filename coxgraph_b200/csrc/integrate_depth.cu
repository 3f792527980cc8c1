// integrate_depth.cu — registered depth + colour images to the points the front half reads.
//
// The reference's live path builds its cloud with depth_image_proc/point_cloud_xyzrgb
// (depth_conversions.h convert<T>) and voxblox_ros TsdfServer drops the points with a non-finite
// coordinate (convertPointcloud) before integratePointCloud.  This pass does both on the device:
// every frame of a job owns a slab of W*H point slots; its kept points fill the slab from the
// front in row-major pixel order and its kept count goes to a device table, which the front half
// reads as the frame's point count (FrameTable::count).  Slots past the count are holes.
//   k_depth_tile_counts   kept points per tile of kDepthTile pixels
//   k_depth_points        tile prefix (sum of the earlier tiles of the frame) + block scan, then
//                         the kept points and colours in order; the last tile writes the count
// Arithmetic (float32, no FMA: -fmad=false): x = ((u - cx) * d) * kx, y = ((v - cy) * d) * ky,
// z = d * 0.001f (16UC1) or d (32FC1), as point_cloud_xyzrgb computes them.
#include <cub/cub.cuh>

#include <math.h>

#include "integrate.cuh"

namespace cg {

constexpr int kDepthThreads = 256, kDepthItems = 8, kDepthTile = kDepthThreads * kDepthItems;

struct DepthParams {
  float cx, cy, kx, ky;       // center_x / y, constant_x / y of convert<T>
  uint32_t width, frame_px;   // W, W * H
  uint32_t tiles;             // tiles per frame
  int r_off, g_off, b_off, pix;  // colour byte offsets and pixel size
};

// DepthTraits<T> of depth_image_proc
__device__ __forceinline__ bool depth_valid(uint16_t d) { return d != 0; }
__device__ __forceinline__ bool depth_valid(float d) { return isfinite(d); }
__device__ __forceinline__ float depth_meters(uint16_t d) { return static_cast<float>(d) * 0.001f; }
__device__ __forceinline__ float depth_meters(float d) { return d; }

// point of pixel px of a frame; false: invalid depth or a non-finite coordinate (dropped)
template <class T>
__device__ __forceinline__ bool depth_point(const DepthParams& dp, T d, uint32_t px, float3& p) {
  if (!depth_valid(d)) return false;
  const float depth = static_cast<float>(d);
  const float u = static_cast<float>(px % dp.width), v = static_cast<float>(px / dp.width);
  p.x = ((u - dp.cx) * depth) * dp.kx;
  p.y = ((v - dp.cy) * depth) * dp.ky;
  p.z = depth_meters(d);
  return isfinite(p.x) && isfinite(p.y) && isfinite(p.z);
}

// CTA b: tile b % tiles of frame b / tiles; each thread kDepthItems consecutive pixels
__device__ __forceinline__ uint32_t tile_first_pixel(const DepthParams& dp) {
  return (blockIdx.x % dp.tiles) * kDepthTile + threadIdx.x * kDepthItems;
}

template <class T>
__global__ void __launch_bounds__(kDepthThreads)
k_depth_tile_counts(DepthParams dp, const T* __restrict__ depth, uint32_t* __restrict__ tile_counts) {
  typedef cub::BlockReduce<uint32_t, kDepthThreads> Reduce;
  __shared__ typename Reduce::TempStorage tmp;
  const size_t frame0 = static_cast<size_t>(blockIdx.x / dp.tiles) * dp.frame_px;
  const uint32_t px0 = tile_first_pixel(dp);
  uint32_t kept = 0;
#pragma unroll
  for (int k = 0; k < kDepthItems; ++k) {
    const uint32_t px = px0 + k;
    float3 p;
    if (px < dp.frame_px && depth_point(dp, depth[frame0 + px], px, p)) ++kept;
  }
  kept = Reduce(tmp).Sum(kept);
  if (threadIdx.x == 0) tile_counts[blockIdx.x] = kept;
}

template <class T>
__global__ void __launch_bounds__(kDepthThreads)
k_depth_points(DepthParams dp, const T* __restrict__ depth, const uint8_t* __restrict__ color,
               const uint32_t* __restrict__ tile_counts, float* __restrict__ pts,
               uchar4* __restrict__ cols, uint32_t* __restrict__ frame_counts) {
  typedef cub::BlockReduce<uint32_t, kDepthThreads> Reduce;
  typedef cub::BlockScan<uint32_t, kDepthThreads> Scan;
  __shared__ union {
    typename Reduce::TempStorage reduce;
    typename Scan::TempStorage scan;
  } tmp;
  const uint32_t f = blockIdx.x / dp.tiles, t = blockIdx.x % dp.tiles;
  const size_t frame0 = static_cast<size_t>(f) * dp.frame_px;
  // kept points of the frame's earlier tiles
  uint32_t before = 0;
  for (uint32_t i = threadIdx.x; i < t; i += kDepthThreads) before += tile_counts[f * dp.tiles + i];
  before = Reduce(tmp.reduce).Sum(before);
  __shared__ uint32_t s_before;
  if (threadIdx.x == 0) s_before = before;
  __syncthreads();
  const uint32_t px0 = tile_first_pixel(dp);
  float3 p[kDepthItems];
  uint32_t keep = 0, kept = 0;
#pragma unroll
  for (int k = 0; k < kDepthItems; ++k) {
    const uint32_t px = px0 + k;
    if (px < dp.frame_px && depth_point(dp, depth[frame0 + px], px, p[k])) {
      keep |= 1u << k;
      ++kept;
    }
  }
  uint32_t slot, total;
  Scan(tmp.scan).ExclusiveSum(kept, slot, total);
  slot += s_before;
#pragma unroll
  for (int k = 0; k < kDepthItems; ++k) {
    if (!((keep >> k) & 1u)) continue;
    const size_t out = frame0 + slot++;
    const uint8_t* c = color + (frame0 + px0 + k) * dp.pix;
    pts[3 * out] = p[k].x;
    pts[3 * out + 1] = p[k].y;
    pts[3 * out + 2] = p[k].z;
    cols[out] = make_uchar4(c[dp.r_off], c[dp.g_off], c[dp.b_off], 255);
  }
  if (t == dp.tiles - 1 && threadIdx.x == 0) frame_counts[f] = s_before + total;
}

int32_t check_depth_camera(const char* who, const cg_depth_camera* cam, size_t F) {
  if (!cam) {
    set_error("%s: null camera", who);
    return CG_ERR_INVALID_ARG;
  }
  if (F == 0 || cam->width <= 0 || cam->height <= 0) {
    set_error("%s: frames, width and height must be positive", who);
    return CG_ERR_INVALID_ARG;
  }
  if (cam->depth_encoding != CG_DEPTH_16UC1 && cam->depth_encoding != CG_DEPTH_32FC1) {
    set_error("%s: unknown depth encoding %d", who, cam->depth_encoding);
    return CG_ERR_INVALID_ARG;
  }
  if (cam->color_encoding < CG_COLOR_RGB8 || cam->color_encoding > CG_COLOR_MONO8) {
    set_error("%s: unknown colour encoding %d", who, cam->color_encoding);
    return CG_ERR_INVALID_ARG;
  }
  if (!(std::isfinite(cam->fx) && cam->fx > 0.0) || !(std::isfinite(cam->fy) && cam->fy > 0.0) ||
      !std::isfinite(cam->cx) || !std::isfinite(cam->cy)) {
    set_error("%s: fx, fy must be finite and positive, cx, cy finite", who);
    return CG_ERR_INVALID_ARG;
  }
  // every frame is a slab of W*H point slots; the job's slots are indexed like a group's points
  const size_t px = static_cast<size_t>(cam->width) * static_cast<size_t>(cam->height);
  if (px > kMaxDepthJobPixels || F > kMaxDepthJobPixels / px) {
    set_error("%s: %zu frames of %d x %d pixels exceed the %zu pixels of one job", who, F,
              cam->width, cam->height, kMaxDepthJobPixels);
    return CG_ERR_INVALID_ARG;
  }
  return CG_OK;
}

size_t depth_pixel_bytes(const cg_depth_camera& cam) {
  return cam.depth_encoding == CG_DEPTH_16UC1 ? sizeof(uint16_t) : sizeof(float);
}
size_t color_pixel_bytes(const cg_depth_camera& cam) {
  switch (cam.color_encoding) {
    case CG_COLOR_RGBA8:
    case CG_COLOR_BGRA8:
      return 4;
    case CG_COLOR_MONO8:
      return 1;
    default:
      return 3;
  }
}

int32_t unproject_depth(cg_context* ctx, FrontBufs& fb, const cg_depth_camera& cam, size_t F,
                        const void* d_depth, const uint8_t* d_color, cudaStream_t s) {
  const size_t frame_px = static_cast<size_t>(cam.width) * cam.height, slots = F * frame_px;
  DepthParams dp;
  // image_geometry::PinholeCameraModel reports the intrinsics as doubles; convert<T> keeps
  // center_x = float(cx) and constant_x = float(toMeters(T(1)) / fx)
  const double unit = cam.depth_encoding == CG_DEPTH_16UC1 ? static_cast<double>(0.001f) : 1.0;
  dp.cx = static_cast<float>(cam.cx);
  dp.cy = static_cast<float>(cam.cy);
  dp.kx = static_cast<float>(unit / cam.fx);
  dp.ky = static_cast<float>(unit / cam.fy);
  dp.width = static_cast<uint32_t>(cam.width);
  dp.frame_px = static_cast<uint32_t>(frame_px);
  dp.tiles = static_cast<uint32_t>((frame_px + kDepthTile - 1) / kDepthTile);
  const bool bgr = cam.color_encoding == CG_COLOR_BGR8 || cam.color_encoding == CG_COLOR_BGRA8;
  const bool mono = cam.color_encoding == CG_COLOR_MONO8;
  dp.r_off = mono ? 0 : (bgr ? 2 : 0);
  dp.g_off = mono ? 0 : 1;
  dp.b_off = mono ? 0 : (bgr ? 0 : 2);
  dp.pix = static_cast<int>(color_pixel_bytes(cam));
  const size_t ctas = F * dp.tiles;
  CG_CUDA(fb.depth_pts.reserve(slots * 3 * sizeof(float)));
  CG_CUDA(fb.depth_cols.reserve(slots * 4));
  CG_CUDA(fb.depth_counts.reserve(F * sizeof(uint32_t)));
  CG_CUDA(fb.depth_tiles.reserve(ctas * sizeof(uint32_t)));
  StageScope sc(ctx, kStageDepthPoints, 2, s);
  const unsigned grid = static_cast<unsigned>(ctas);
  if (cam.depth_encoding == CG_DEPTH_16UC1) {
    const uint16_t* d = static_cast<const uint16_t*>(d_depth);
    k_depth_tile_counts<<<grid, kDepthThreads, 0, s>>>(dp, d, fb.depth_tiles.as<uint32_t>());
    k_depth_points<<<grid, kDepthThreads, 0, s>>>(dp, d, d_color, fb.depth_tiles.as<uint32_t>(),
                                                  fb.depth_pts.as<float>(), fb.depth_cols.as<uchar4>(),
                                                  fb.depth_counts.as<uint32_t>());
  } else {
    const float* d = static_cast<const float*>(d_depth);
    k_depth_tile_counts<<<grid, kDepthThreads, 0, s>>>(dp, d, fb.depth_tiles.as<uint32_t>());
    k_depth_points<<<grid, kDepthThreads, 0, s>>>(dp, d, d_color, fb.depth_tiles.as<uint32_t>(),
                                                  fb.depth_pts.as<float>(), fb.depth_cols.as<uchar4>(),
                                                  fb.depth_counts.as<uint32_t>());
  }
  CG_CUDA(cudaGetLastError());
  return CG_OK;
}

}  // namespace cg
