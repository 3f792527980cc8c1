// integrate.cu — TSDF integration of point clouds into the block-hashed layer.
//
// Replaces voxblox::TsdfIntegratorBase::integratePointCloud (Simple / Merged semantics, R1-R6 of
// SURVEY.md §8a); reference call site coxgraph/include/coxgraph/map_comm/tsdf_recover.h:75.
//
// One job = one frame, or a batch of frames fused into the same layer (the loop of
// tsdf_recover.h:71-86).  All frames of a job go through every stage together (DESIGN.md §4):
//  front half — points to one ray per bundle (R1, R2, R6)
//   k_point_keys        validity, T_G_C * p, bundle key [frame | clearing | voxel of p_G relative
//                       to the sensor voxel | visit rank]
//   radix sort (keys)   on the bits above the rank: bundles in canonical order, their points in the
//                       order the reference visits them
//   select              bundle heads
//   k_gather_sorted     the sorted points next to each other
//   k_bundle_histogram / k_bundle_order   bundles by size class, longest first
//   k_fold_wide / k_fold_bundles          the reference's *sequential* weighted mean and colour
//                       blend per bundle (bit-exact: the merged point decides which voxels and
//                       blocks the ray visits) -> one ray per bundle
//   k_grazing_build     (anti-grazing only) set of the scan's bundle voxels
//   k_bundle_rays       T_G_C * merged point, closed-form visit / block counts; k_scan_* offsets
//  back half — rays to voxels (R3, R4, R5)
//   k_walk_segments     3-D DDA per ray (voxblox::RayCaster); every visited block enters the GPU
//                       hash (allocation on first visit); one record per (ray, block); voxels
//                       whose update order matters are flagged "general"
//   k_segment_hist / k_segment_scatter    segments grouped by block
//   k_block_accumulate  per block, in shared memory: commutative weight sums of the free-space
//                       visits; visits of general voxels go out as (voxel, ray) keys
//   radix sort (keys)   per-voxel update lists in canonical order
//   k_voxel_update / k_long_partials / k_long_finish   ordered replay of the general voxels
//   k_finalize_blocks   coalesced read-modify-write of the free-space voxels of every touched block
// Per-voxel order is (frame, non-clearing before clearing, bundle key ascending) — the oracle's
// canonical order — independent of scheduling.
#include <cub/cub.cuh>
#include <thrust/iterator/counting_iterator.h>
#include <stdlib.h>
#include <string.h>

#include <algorithm>
#include <type_traits>
#include <vector>

#include "cg_internal.cuh"
#include "host_stage.cuh"

namespace cg {

// Device-side fill used instead of cudaMemsetAsync on the compute stream: a memset may be
// executed by a copy engine, where it would queue behind the (large) host->device transfers of
// the pipelined batch path and stall the kernels that follow it.
__global__ void k_fill_words(uint32_t* __restrict__ p, uint32_t v, size_t n) {
  for (size_t i = blockIdx.x * static_cast<size_t>(blockDim.x) + threadIdx.x; i < n;
       i += static_cast<size_t>(gridDim.x) * blockDim.x)
    p[i] = v;
}
__global__ void k_copy_words(uint32_t* __restrict__ dst, const uint32_t* __restrict__ src, size_t n) {
  const size_t i = blockIdx.x * static_cast<size_t>(blockDim.x) + threadIdx.x;
  if (i < n) dst[i] = src[i];
}
static inline cudaError_t fill_bytes(void* p, int byte, size_t bytes, cudaStream_t s) {
  const size_t n = bytes / 4;
  if (n == 0) return cudaSuccess;
  const uint32_t v = 0x01010101u * static_cast<uint32_t>(byte & 0xFF);
  const unsigned grid = static_cast<unsigned>(std::min<size_t>((n + 255) / 256, 148 * 8));
  k_fill_words<<<grid, 256, 0, s>>>(static_cast<uint32_t*>(p), v, n);
  return cudaGetLastError();
}

struct Ray {           // 24 B
  float px, py, pz;    // merged point, global frame
  float weight;        // merged weight
  uint32_t color;      // merged colour
  uint32_t frame_clr;  // frame index in job | clearing << 31 ; 0xFFFFFFFF = no ray
};
constexpr uint32_t kNoRay = 0xFFFFFFFFu;

// Bundle key (u64): [clearing(1) | z | y | x | frame (frame_bits) | visit rank (rank_bits)].
// z, y, x: voxel index of the point relative to the voxel holding the sensor origin, minus the
// lower corner `lo` of the box the layout covers, bits[a] wide; visit rank: position of the point in
// the reference's visiting order of its frame.  The keys are written in (frame, rank) order and
// sorted on the (clearing, voxel) bits only (keys-only radix sort, begin_bit = rank_bits +
// frame_bits): a stable sort keeps the points of one (clearing, voxel) in (frame, rank) order, so a
// bundle — one frame's points in one voxel — is a contiguous run in visiting order, the point
// index is recovered from (frame, rank) and no value array travels through the sort; leaving the
// frame field out of the sorted bits saves a radix pass at the C2 shape (24 bits instead of 29).
// The position of a bundle in the canonical (frame, clearing, voxel) order the back half replays
// in — its ray id — is then a stable partition of the bundles by frame (k_bundle_histogram /
// k_frame_scan / k_bundle_order).  The box is chosen per group by the host from the extent
// earlier jobs on the context measured — a room-sized scene needs 9 + 8 + 6 bits where a cube
// around the sensor wide enough for clearing points needs 3 x 10; a point outside the box is
// detected on the device and the group is redone with the measured extent.
struct KeyLayout {
  int rank_bits;
  int frame_bits;
  int bits[3];  // x, y, z
  int lo[3];
  __host__ __device__ __forceinline__ int frame_shift() const { return rank_bits; }
  __host__ __device__ __forceinline__ int voxel_shift() const { return rank_bits + frame_bits; }
  __host__ __device__ __forceinline__ int shift(int a) const {
    return voxel_shift() + (a > 0 ? bits[0] : 0) + (a > 1 ? bits[1] : 0);
  }
  __host__ __device__ __forceinline__ int clear_bit() const {
    return voxel_shift() + bits[0] + bits[1] + bits[2];
  }
  __device__ __forceinline__ bool clearing(uint64_t key) const { return (key >> clear_bit()) & 1; }
  __device__ __forceinline__ uint32_t frame(uint64_t key) const {
    return static_cast<uint32_t>(key >> frame_shift()) & ((1u << frame_bits) - 1u);
  }
  __device__ __forceinline__ uint32_t rank(uint64_t key) const {
    return static_cast<uint32_t>(key & ((1ull << rank_bits) - 1ull));
  }
  // voxel of the bundle relative to its frame's sensor voxel
  __device__ __forceinline__ int rel(uint64_t key, int a) const {
    return static_cast<int>((key >> shift(a)) & ((1ull << bits[a]) - 1ull)) + lo[a];
  }
};
constexpr int kMaxRelBits = 13;
// |rel| <= 8191 voxels: what a single frame's key can hold (14 bits per axis; the anti-grazing set
// packs the same).  A point further from the sensor than that — 410 m at 5 cm voxels, 164 m at
// 2 cm: a stray return; it can only be a clearing point — is dropped and counted
// (cg_integrate_stats.points_beyond_reach) instead of failing the frame; the reference would carve
// along its first max_ray_length metres.
constexpr int kKeySlack = 16, kKeyLimit = 8191;
constexpr size_t kMaxGroupFrames = 8192;  // frames per group: per-frame bins in shared memory

__device__ __forceinline__ int order_index(int k, int n, int mode) {
  // voxblox MixedThreadSafeIndex: groups of 1024 visited round-robin
  if (mode != 0) return k;
  const int groups = n / 1024;
  if (groups * 1024 <= k) return k;
  return (k % groups) * 1024 + (k / groups);
}

// inverse of order_index: the visiting rank of point i
__device__ __forceinline__ int visit_rank(int i, int n, int mode) {
  if (mode != 0) return i;
  const int groups = n / 1024;
  if (groups * 1024 <= i) return i;
  return (i % 1024) * groups + (i / 1024);
}

__device__ __forceinline__ V3 load_point(const float* pts, size_t i) {
  return V3{pts[3 * i], pts[3 * i + 1], pts[3 * i + 2]};
}

// Frames of one group: offs points at the group's first entry of the job's offset table (F + 1
// entries are read), base = offs[0]; slots and point indices are relative to the group.
struct FrameTable {
  const uint64_t* offs;
  uint64_t base;
  int F;
  __device__ __forceinline__ uint64_t start(int f) const { return offs[f] - base; }
  __device__ __forceinline__ int frame_of(uint64_t g) const {
    int lo = 0, hi = F;  // start(lo) <= g < start(hi)
    while (hi - lo > 1) {
      const int mid = (lo + hi) >> 1;
      if (start(mid) <= g) lo = mid; else hi = mid;
    }
    return lo;
  }
};

// ------------------------------------------------------------------ front half
// One thread per point in input order (coalesced reads); its key goes to the slot of its visiting
// rank k (the scattered 8-byte writes of a wave merge in L2).
__global__ void k_point_keys(IntegratorParams P, KeyLayout kl, const float* __restrict__ poses,
                             FrameTable ft, const float* __restrict__ pts, uint64_t total,
                             uint64_t* __restrict__ keys, int32_t* err, int* key_bounds,
                             CallCounters* counters) {
  // key_bounds != nullptr: also measure the extent of the job's points (see below)
  __shared__ int s_bounds[6];
  if (key_bounds && threadIdx.x < 6) s_bounds[threadIdx.x] = threadIdx.x < 3 ? 0x3FFFFFFF : -0x3FFFFFFF;
  const uint64_t g = blockIdx.x * static_cast<uint64_t>(blockDim.x) + threadIdx.x;
  // the CTA's points are consecutive: one binary search for its first point, then each thread
  // walks on from that frame (zero or one step unless the frames are tiny)
  __shared__ int s_first_frame;
  if (threadIdx.x == 0) {
    const uint64_t g0 = blockIdx.x * static_cast<uint64_t>(blockDim.x);
    s_first_frame = ft.frame_of(g0 < total ? g0 : total - 1);
  }
  __syncthreads();
  int rx = 0, ry = 0, rz = 0;
  bool have = false;
  if (g < total) {
    int f = s_first_frame;
    while (f + 1 < ft.F && ft.start(f + 1) <= g) ++f;
    const uint64_t base = ft.start(f);
    const int n = static_cast<int>(ft.start(f + 1) - base);
    const int i = static_cast<int>(g - base);
    const uint32_t k = static_cast<uint32_t>(visit_rank(i, n, P.order_mode));
    const V3 pc = load_point(pts, g);
    bool clearing = false;
    uint64_t key = kInvalidPointKey;
    if (point_valid(P, pc, &clearing)) {
      const Xform T = make_xform(poses + 7 * f);
      const V3 pg = apply(T, pc);
      const float lim = 524000.0f * P.voxel_size;
      if (fabsf(pg.x) < lim && fabsf(pg.y) < lim && fabsf(pg.z) < lim && fabsf(T.t.x) < lim &&
          fabsf(T.t.y) < lim && fabsf(T.t.z) < lim) {
        rx = grid_index(pg.x, P.voxel_size_inv) - grid_index(T.t.x, P.voxel_size_inv);
        ry = grid_index(pg.y, P.voxel_size_inv) - grid_index(T.t.y, P.voxel_size_inv);
        rz = grid_index(pg.z, P.voxel_size_inv) - grid_index(T.t.z, P.voxel_size_inv);
        const bool far = max(max(abs(rx), abs(ry)), abs(rz)) > kKeyLimit;
        have = !far;
        const uint32_t ux = static_cast<uint32_t>(rx - kl.lo[0]), uy = static_cast<uint32_t>(ry - kl.lo[1]),
                       uz = static_cast<uint32_t>(rz - kl.lo[2]);
        if (far) {
          atomicAdd(&counters->far_points, 1ull);  // beyond any key box: dropped, counted
        } else if ((ux >> kl.bits[0]) == 0 && (uy >> kl.bits[1]) == 0 && ((uz + 1u) >> kl.bits[2]) == 0) {
          // (uz + 1: the z field is never all ones, so that the key of a dropped point — all ones —
          // sorts behind every real key on the sorted bits alone)
          key = (static_cast<uint64_t>(f) << kl.frame_shift()) |
                (static_cast<uint64_t>(clearing) << kl.clear_bit()) |
                (static_cast<uint64_t>(uz) << kl.shift(2)) | (static_cast<uint64_t>(uy) << kl.shift(1)) |
                (static_cast<uint64_t>(ux) << kl.shift(0)) | k;
        } else {
          // outside the box this group's key layout covers: the host redoes the group with the
          // extent measured below (fewer frames per group if the bits run out)
          atomicOr(err, kErrKeyRange);
        }
      } else {
        atomicOr(err, kErrOutOfRange);
      }
    }
    keys[base + k] = key;
  }
  // Extent of the job's points (relative voxel indices): it sizes the key layout of later jobs.
  // Only measured when the host asks (first job of a context, the retry after a point fell outside
  // the box, and now and then to let the box shrink): warp minimum / maximum, then shared memory,
  // then six atomics per CTA.
  if (!key_bounds) return;
  const unsigned full = 0xFFFFFFFFu;
  const int big = 0x3FFFFFFF;
  const int mnx = __reduce_min_sync(full, have ? rx : big), mxx = __reduce_max_sync(full, have ? rx : -big);
  const int mny = __reduce_min_sync(full, have ? ry : big), mxy = __reduce_max_sync(full, have ? ry : -big);
  const int mnz = __reduce_min_sync(full, have ? rz : big), mxz = __reduce_max_sync(full, have ? rz : -big);
  if ((threadIdx.x & 31) == 0 && mnx != big) {
    atomicMin(&s_bounds[0], mnx);
    atomicMin(&s_bounds[1], mny);
    atomicMin(&s_bounds[2], mnz);
    atomicMax(&s_bounds[3], mxx);
    atomicMax(&s_bounds[4], mxy);
    atomicMax(&s_bounds[5], mxz);
  }
  __syncthreads();
  if (threadIdx.x < 3 && s_bounds[threadIdx.x] != big) atomicMin(key_bounds + threadIdx.x, s_bounds[threadIdx.x]);
  if (threadIdx.x >= 3 && threadIdx.x < 6 && s_bounds[threadIdx.x] != -big)
    atomicMax(key_bounds + threadIdx.x, s_bounds[threadIdx.x]);
}

struct BundleHead {
  const uint64_t* keys;
  int rank_bits;
  __device__ __forceinline__ bool operator()(uint32_t i) const {
    // the first invalid key is a head too: it terminates the last real bundle
    return i == 0 || (keys[i] >> rank_bits) != (keys[i - 1] >> rank_bits);
  }
};

// Gather the sorted points next to each other: (x, y, z, rgba) per sorted slot, so that the
// sequential fold streams contiguous memory.  The point index comes from the key's (frame, rank).
__global__ void k_gather_sorted(KeyLayout kl, int order_mode, const uint64_t* __restrict__ keys,
                                uint32_t total, FrameTable ft, const float* __restrict__ pts,
                                const uint32_t* __restrict__ cols, float4* __restrict__ out) {
  const uint32_t j = blockIdx.x * blockDim.x + threadIdx.x;
  if (j >= total) return;
  const uint64_t key = keys[j];
  if (key == kInvalidPointKey) return;
  const int f = static_cast<int>(kl.frame(key));
  const uint64_t base = ft.start(f);
  const int n = static_cast<int>(ft.start(f + 1) - base);
  const size_t i = base + order_index(static_cast<int>(kl.rank(key)), n, order_mode);
  out[j] = make_float4(pts[3 * i], pts[3 * i + 1], pts[3 * i + 2], __uint_as_float(cols[i]));
}

// MergedTsdfIntegrator::integrateVoxel, first half: the reference's *sequential* weighted mean and
// colour blend over the points of a bundle (bit-exact: the merged point decides which voxels and
// blocks the ray visits).  The recurrence cannot be re-associated, so a bundle is one lane's
// work; what is left to arrange is that the 32 lanes of a warp get bundles of (nearly) the same
// length and that the longest bundles start first:
//   k_bundle_histogram  bundle sizes -> 48 size classes (4 per octave), largest class first
//   k_bundle_order      counting-sort scatter of the bundle ids by class
//   k_fold_bundles      warp g of the persistent grid folds bundles order[32 g .. 32 g + 31]; every
//                       lane streams its own run of `sorted` with a 4-deep register prefetch.
constexpr int kSizeClasses = 48;
__device__ __forceinline__ int size_class(uint32_t n) {  // descending: class 0 = largest
  if (n == 0) n = 1;
  const int lg = 31 - __clz(n);                                  // floor(log2 n), 0..31
  const int frac = lg >= 2 ? static_cast<int>((n >> (lg - 2)) & 3u) : 0;  // next two bits
  const int c = min(4 * lg + frac, kSizeClasses - 1);
  return kSizeClasses - 1 - c;
}
struct BundleInfo {
  uint32_t start, n;
  uint64_t key;
};
__device__ __forceinline__ BundleInfo bundle_info(const uint64_t* __restrict__ keys, uint32_t total,
                                                  const uint32_t* __restrict__ heads, uint32_t nb,
                                                  uint32_t b) {
  BundleInfo bi;
  bi.start = heads[b];
  bi.n = ((b + 1 < nb) ? heads[b + 1] : total) - bi.start;
  bi.key = keys[bi.start];
  return bi;
}
// a clearing bundle only uses its first point with a valid weight: it is short whatever its size
__device__ __forceinline__ uint32_t fold_length(const KeyLayout& kl, const BundleInfo& bi) {
  return kl.clearing(bi.key) ? 1u : bi.n;
}

// Ray ids.  Bundle b (position in the sorted keys: (clearing, voxel)-major, frames interleaved)
// becomes ray  frame_start[f] + #{b' < b of the same frame f}: within a frame the bundles already
// are in (clearing, voxel) order, so this stable partition by frame IS the canonical (frame,
// clearing, voxel) order.  Every CTA owns a contiguous chunk of bundles; frame_count[f * G + cta]
// holds its bundles of frame f (bin F: the sentinel bundle of dropped points, which so gets the
// last id), an exclusive scan over that array in (f, cta) order gives each (frame, chunk) its
// first id, and k_bundle_order ranks the bundles of a chunk in ascending b.
__device__ __forceinline__ void bundle_chunk(uint32_t nb, uint32_t& lo, uint32_t& hi) {
  const uint32_t per = (nb + gridDim.x - 1) / gridDim.x;
  lo = min(nb, blockIdx.x * per);
  hi = min(nb, lo + per);
}

// class_count[0 .. kSizeClasses): histogram; [kSizeClasses .. 2 kSizeClasses): scatter cursors
__global__ void k_bundle_histogram(KeyLayout kl, const uint64_t* __restrict__ keys, uint32_t total,
                                   const uint32_t* __restrict__ heads,
                                   const uint32_t* __restrict__ num_heads, uint32_t* class_count,
                                   uint32_t* __restrict__ frame_count, int F) {
  extern __shared__ uint32_t s_frames[];  // F + 1 bins
  __shared__ uint32_t hist[kSizeClasses];
  if (threadIdx.x < kSizeClasses) hist[threadIdx.x] = 0;
  for (int f = threadIdx.x; f <= F; f += blockDim.x) s_frames[f] = 0;
  __syncthreads();
  const uint32_t nb = *num_heads;
  uint32_t lo, hi;
  bundle_chunk(nb, lo, hi);
  for (uint32_t b = lo + threadIdx.x; b < hi; b += blockDim.x) {
    const BundleInfo bi = bundle_info(keys, total, heads, nb, b);
    if (bi.key == kInvalidPointKey) {
      atomicAdd(&s_frames[F], 1u);
    } else {
      atomicAdd(&s_frames[kl.frame(bi.key)], 1u);
      atomicAdd(&hist[size_class(fold_length(kl, bi))], 1u);
    }
  }
  __syncthreads();
  if (threadIdx.x < kSizeClasses && hist[threadIdx.x])
    atomicAdd(&class_count[threadIdx.x], hist[threadIdx.x]);
  for (int f = threadIdx.x; f <= F; f += blockDim.x)
    frame_count[static_cast<size_t>(f) * gridDim.x + blockIdx.x] = s_frames[f];
}

// exclusive scan of the (frame, chunk) counts, in place; one CTA
__global__ void __launch_bounds__(1024) k_frame_scan(uint32_t* __restrict__ counts, uint32_t n) {
  typedef cub::BlockScan<uint32_t, 1024> Scan;
  __shared__ typename Scan::TempStorage tmp;
  __shared__ uint32_t carry;
  if (threadIdx.x == 0) carry = 0;
  __syncthreads();
  for (uint32_t i0 = 0; i0 < n; i0 += 1024) {
    const uint32_t i = i0 + threadIdx.x;
    const uint32_t v = i < n ? counts[i] : 0u;
    uint32_t ex, sum;
    Scan(tmp).ExclusiveSum(v, ex, sum);
    if (i < n) counts[i] = carry + ex;
    __syncthreads();
    if (threadIdx.x == 0) carry += sum;
    __syncthreads();
  }
}

__global__ void __launch_bounds__(256)
k_bundle_order(KeyLayout kl, const uint64_t* __restrict__ keys, uint32_t total,
               const uint32_t* __restrict__ heads, const uint32_t* __restrict__ num_heads,
               uint32_t* class_count, const uint32_t* __restrict__ frame_base, int F,
               uint32_t* __restrict__ order, uint32_t* __restrict__ ray_id,
               Ray* __restrict__ folded) {
  extern __shared__ uint32_t s_next[];  // F + 1: next ray id of each frame within this chunk
  __shared__ uint32_t base[kSizeClasses];
  __shared__ uint32_t hist[kSizeClasses];
  __shared__ uint32_t offs[kSizeClasses];
  const unsigned full = 0xFFFFFFFFu;
  const int lane = threadIdx.x & 31, wib = threadIdx.x >> 5;
  if (threadIdx.x == 0) {
    uint32_t acc = 0;
    for (int c = 0; c < kSizeClasses; ++c) {
      base[c] = acc;
      acc += class_count[c];
    }
  }
  for (int f = threadIdx.x; f <= F; f += blockDim.x)
    s_next[f] = frame_base[static_cast<size_t>(f) * gridDim.x + blockIdx.x];
  const uint32_t nb = *num_heads;
  uint32_t lo, hi;
  bundle_chunk(nb, lo, hi);
  for (uint32_t b0 = lo; b0 < hi; b0 += blockDim.x) {
    __syncthreads();
    if (threadIdx.x < kSizeClasses) hist[threadIdx.x] = 0;
    __syncthreads();
    const uint32_t b = b0 + threadIdx.x;
    int c = -1;
    uint32_t rank = 0;
    uint32_t f = static_cast<uint32_t>(F) + 1u;  // no bundle in this lane
    if (b < hi) {
      const BundleInfo bi = bundle_info(keys, total, heads, nb, b);
      if (bi.key != kInvalidPointKey) {
        c = size_class(fold_length(kl, bi));
        rank = atomicAdd(&hist[c], 1u);
        f = kl.frame(bi.key);
      } else {
        f = static_cast<uint32_t>(F);
      }
    }
    // ray id: lanes of the same frame in lane order, warps in turn
    const unsigned same = __match_any_sync(full, f);
    const int leader = __ffs(same) - 1;
    const uint32_t before = __popc(same & ((1u << lane) - 1u));
    uint32_t first = 0;
    for (int w = 0; w < static_cast<int>(blockDim.x >> 5); ++w) {
      if (wib == w && lane == leader && f <= static_cast<uint32_t>(F)) {
        first = s_next[f];
        s_next[f] = first + __popc(same);
      }
      __syncthreads();
    }
    first = __shfl_sync(full, first, leader);
    if (threadIdx.x < kSizeClasses && hist[threadIdx.x])
      offs[threadIdx.x] = atomicAdd(&class_count[kSizeClasses + threadIdx.x], hist[threadIdx.x]);
    __syncthreads();
    if (c >= 0) order[base[c] + offs[c] + rank] = b;
    if (b < hi) {
      ray_id[b] = first + before;
      if (c < 0) folded[first + before].frame_clr = kNoRay;  // sentinel bundle of dropped points
    }
  }
}

// bundles of 64 points or more are the first n_wide entries of `order`
constexpr int kWideClasses = kSizeClasses - 4 * 6;  // classes with floor(log2 n) >= 6
__device__ __forceinline__ uint32_t wide_count(const uint32_t* __restrict__ class_count, int lane) {
  uint32_t n = (lane < kWideClasses) ? class_count[lane] : 0u;
#pragma unroll
  for (int d = 16; d >= 1; d >>= 1) n += __shfl_xor_sync(0xFFFFFFFFu, n, d);
  return n;
}

// Long bundles: 8 lanes per bundle, 4 bundles per warp.  The recurrence itself stays sequential,
// but everything that does not depend on the running mean is taken off its critical path: per
// chunk of 8 points the lanes compute, in parallel, the point weights, then (one short
// sequential pass over the chunk's weights, read back from shared memory) the running weight W_k,
// then the per-point reciprocal and blend factors and the products p_k w_k, c_k b_k; what remains
// per point is the 7-operation chain
//   m <- (m W_{k-1} + p_k w_k) / W_k          (div_with_rcp: exact IEEE quotient)
// and the colour blend, run as 7 independent chains (x, y, z, r, g, b, a) on 7 of the 8 lanes; a
// chain step reads its point's four factors with one 16-byte load and its operand with another.
// The warps take groups of 4 bundles from a queue over the longest-first order: the kernel lasts
// as long as its longest bundle (it is bound by that chain, not by instruction issue: 4 lanes per
// bundle and 8 bundles per warp issue a third fewer instructions and take 0.126 ms against 0.100),
// and few resident warps per scheduler keep the chains fed.
constexpr int kWideWarps = 4;
constexpr int kWideGroup = 8;  // lanes per bundle = points per chunk
constexpr int kWideOpStride = 72;  // words per bundle in s_op: 8 points x 8 chains + 8 (banks)
__device__ __forceinline__ void
fold_wide(const IntegratorParams& P, const KeyLayout& kl, const uint64_t* __restrict__ keys,
          uint32_t total, const uint32_t* __restrict__ heads, const uint32_t* __restrict__ num_heads,
          const float4* __restrict__ sorted, const uint32_t* __restrict__ class_count,
          const uint32_t* __restrict__ order, const uint32_t* __restrict__ ray_id, uint32_t* queue,
          Ray* __restrict__ folded) {
  __shared__ __align__(16) float s_wt[kWideWarps][32];    // the chunk's point weights
  __shared__ float4 s_fac[kWideWarps][32];                // per point: W_{k-1}, W_k, 1/W_k, W_{k-1}/W_k
  __shared__ __align__(16) float s_op[kWideWarps][4 * kWideOpStride];  // [bundle][point][chain]
  const unsigned full = 0xFFFFFFFFu;
  const int lane = threadIdx.x & 31, wib = threadIdx.x >> 5;
  const int sub = lane >> 3, l8 = lane & 7, gbase = lane & ~7;
  const uint32_t nb = *num_heads;
  const uint32_t n_wide = wide_count(class_count, lane);
  const int chain = l8;  // 0..2 mean, 3..6 colour, 7 idle
  for (;;) {
    uint32_t g = 0;
    if (lane == 0) g = atomicAdd(queue, 4u);
    g = __shfl_sync(full, g, 0);
    if (g >= n_wide) break;
    const bool have = g + sub < n_wide;
    uint32_t b = 0, start = 0, end = 0;
    uint64_t key = 0;
    if (have) {
      b = order[g + sub];
      const BundleInfo bi = bundle_info(keys, total, heads, nb, b);
      start = bi.start;
      end = bi.start + bi.n;
      key = bi.key;
    }
    float W = 0.0f;                            // running weight (same in the 8 lanes of a group)
    float val = (chain == 6) ? kDefaultAlpha : 0.0f;  // this lane's chain state (default colour)
    float4 pt = (start + l8 < end) ? sorted[start + l8] : make_float4(0.0f, 0.0f, 0.0f, 0.0f);
    for (uint32_t c0 = start; __any_sync(full, c0 < end); c0 += kWideGroup) {
      const uint32_t cnt = c0 < end ? min(static_cast<uint32_t>(kWideGroup), end - c0) : 0u;
      const float4 p = pt;
      if (c0 + kWideGroup + l8 < end) pt = sorted[c0 + kWideGroup + l8];  // next chunk, in flight
      const bool valid = static_cast<uint32_t>(l8) < cnt;
      const float w = valid ? voxel_weight(P, p.z) : 0.0f;
      const bool skip = !valid || w < kEps;  // reference: "if (w < kEps) continue"
      s_wt[wib][lane] = skip ? 0.0f : w;
      const unsigned skip_bits = (__ballot_sync(full, skip) >> gbase) & 0xFFu;
      __syncwarp();
      // running weight: the reference's sequential float sum, every lane over its bundle's chunk
      const float4 wa = *reinterpret_cast<const float4*>(&s_wt[wib][gbase]);
      const float4 wb = *reinterpret_cast<const float4*>(&s_wt[wib][gbase + 4]);
      const float wt[kWideGroup] = {wa.x, wa.y, wa.z, wa.w, wb.x, wb.y, wb.z, wb.w};
      float w_prev_mine = 0.0f, w_mine = 0.0f;
#pragma unroll
      for (int t = 0; t < kWideGroup; ++t) {
        const float Wn = W + wt[t];
        if (l8 == t) {
          w_prev_mine = W;
          w_mine = Wn;
        }
        W = Wn;
      }
      // per-point factors, all lanes in parallel (same values as fold_step: r = RN(1 / W_k) makes
      // div_with_rcp the exact quotient)
      const float r = 1.0f / w_mine;
      const float a = div_with_rcp(w_prev_mine, w_mine, r);
      const float bb = div_with_rcp(w, w_mine, r);
      const uint32_t col = __float_as_uint(p.w);
      s_fac[wib][lane] = make_float4(w_prev_mine, w_mine, r, a);
      float* ops = &s_op[wib][sub * kWideOpStride + l8 * 8];
      *reinterpret_cast<float4*>(ops) =
          make_float4(p.x * w, p.y * w, p.z * w, static_cast<float>(col & 255u) * bb);
      *reinterpret_cast<float4*>(ops + 4) =
          make_float4(static_cast<float>((col >> 8) & 255u) * bb,
                      static_cast<float>((col >> 16) & 255u) * bb,
                      static_cast<float>(col >> 24) * bb, 0.0f);
      __syncwarp();
      // the sequential chains of the 4 bundles side by side
      const float* op = &s_op[wib][sub * kWideOpStride + chain];
#pragma unroll
      for (int t = 0; t < kWideGroup; ++t) {
        const float4 fc = s_fac[wib][gbase + t];
        const float o = op[t * 8];
        const float mean = div_with_rcp(val * fc.x + o, fc.y, fc.z);
        const float colr = round_half_away_pos(val * fc.w + o);
        const float nv = chain < 3 ? mean : colr;
        if (!((skip_bits >> t) & 1u)) val = nv;
      }
    }
    const float mx = __shfl_sync(full, val, gbase + 0), my = __shfl_sync(full, val, gbase + 1);
    const float mz = __shfl_sync(full, val, gbase + 2);
    const float cr = __shfl_sync(full, val, gbase + 3), cg = __shfl_sync(full, val, gbase + 4);
    const float cb = __shfl_sync(full, val, gbase + 5), ca = __shfl_sync(full, val, gbase + 6);
    if (have && l8 == 0) {
      Ray ray;
      ray.px = mx;  // camera frame; k_bundle_rays moves it to the global frame
      ray.py = my;
      ray.pz = mz;
      ray.weight = W;
      ray.color = pack_rgba(static_cast<uint32_t>(cr), static_cast<uint32_t>(cg),
                            static_cast<uint32_t>(cb), static_cast<uint32_t>(ca));
      ray.frame_clr = kl.frame(key);
      folded[ray_id[b]] = ray;
    }
  }
}

constexpr int kFoldDepth = 4;  // points in flight per lane

// Shorter bundles: one lane each, the 32 lanes of a warp on 32 consecutive bundles of the
// longest-first order (nearly equal lengths), kFoldDepth points in flight per lane.  `cta` of
// `num_ctas`: the CTAs of k_fold that run this part.
__device__ __forceinline__ void
fold_short(const IntegratorParams& P, const KeyLayout& kl, const uint64_t* __restrict__ keys,
           uint32_t total, const uint32_t* __restrict__ heads, const uint32_t* __restrict__ num_heads,
           const float4* __restrict__ sorted, const uint32_t* __restrict__ class_count,
           const uint32_t* __restrict__ order, const uint32_t* __restrict__ ray_id,
           Ray* __restrict__ folded, uint32_t cta, uint32_t num_ctas) {
  const unsigned full = 0xFFFFFFFFu;
  const int lane = threadIdx.x & 31;
  const uint32_t nb = *num_heads;
  // bundles in `order` = all but the sentinel = the total of the histogram
  uint32_t n_order = 0;
  for (int c = lane; c < kSizeClasses; c += 32) n_order += class_count[c];
#pragma unroll
  for (int d = 16; d >= 1; d >>= 1) n_order += __shfl_xor_sync(full, n_order, d);
  const uint32_t n_wide = wide_count(class_count, lane);
  const uint32_t warp = (cta * blockDim.x + threadIdx.x) >> 5;
  const uint32_t num_warps = (num_ctas * blockDim.x) >> 5;
  for (uint32_t g = warp; n_wide + g * 32u < n_order; g += num_warps) {
    const uint32_t i = n_wide + g * 32u + lane;
    uint32_t b = 0, cur = 0, n = 0, frame_clr = 0;
    bool clearing = false;
    if (i < n_order) {
      b = order[i];
      const BundleInfo bi = bundle_info(keys, total, heads, nb, b);
      cur = bi.start;
      n = bi.n;
      clearing = kl.clearing(bi.key);
      frame_clr = kl.frame(bi.key) | (clearing ? 0x80000000u : 0u);
    }
    const uint32_t end = cur + n;
    float4 q[kFoldDepth];
#pragma unroll
    for (int u = 0; u < kFoldDepth; ++u)
      q[u] = (cur + u < end) ? sorted[cur + u] : make_float4(0.0f, 0.0f, 0.0f, 0.0f);
    FoldState st;
    fold_reset(st);
    bool done = n == 0;
    // all lanes of the warp have nearly the same length: run to the longest
    while (__any_sync(full, !done)) {
#pragma unroll
      for (int u = 0; u < kFoldDepth; ++u) {
        const float4 p = q[u];
        if (cur + kFoldDepth < end) q[u] = sorted[cur + kFoldDepth];
        if (!done) {
          const float w = voxel_weight(P, p.z);
          if (!(w < kEps)) {
            fold_step(st, p.x, p.y, p.z, __float_as_uint(p.w), w);
            if (clearing) done = true;  // only the first point of a clearing bundle is used
          }
          ++cur;
          if (cur >= end) done = true;
        }
      }
    }
    if (i < n_order) {
      Ray r;
      r.px = st.m.x;  // camera frame; k_bundle_rays moves it to the global frame
      r.py = st.m.y;
      r.pz = st.m.z;
      r.weight = st.W;
      r.color = fold_color(st);
      r.frame_clr = frame_clr;
      folded[ray_id[b]] = r;
    }
  }
}

// Both folds in one launch: the first `wide_ctas` CTAs run the long bundles (bound by the longest
// chain, few warps busy towards the end), the others the short ones, which fill the machine
// meanwhile.
static_assert(kWideWarps * 32 == 128, "k_fold: one CTA shape for both parts");
__global__ void __launch_bounds__(128)
k_fold(IntegratorParams P, KeyLayout kl, const uint64_t* __restrict__ keys, uint32_t total,
       const uint32_t* __restrict__ heads, const uint32_t* __restrict__ num_heads,
       const float4* __restrict__ sorted, const uint32_t* __restrict__ class_count,
       const uint32_t* __restrict__ order, const uint32_t* __restrict__ ray_id, uint32_t* queue,
       Ray* __restrict__ folded, uint32_t wide_ctas) {
  if (blockIdx.x < wide_ctas)
    fold_wide(P, kl, keys, total, heads, num_heads, sorted, class_count, order, ray_id, queue, folded);
  else
    fold_short(P, kl, keys, total, heads, num_heads, sorted, class_count, order, ray_id, folded,
               blockIdx.x - wide_ctas, gridDim.x - wide_ctas);
}

// one thread per bundle: T_G_C * merged point, ray set-up, pair count
__global__ void k_bundle_rays(IntegratorParams P, const float* __restrict__ poses,
                              const uint32_t* __restrict__ num_heads, Ray* __restrict__ rays,
                              unsigned long long* __restrict__ ray_count) {
  const uint32_t nb = *num_heads;
  for (uint32_t b = blockIdx.x * blockDim.x + threadIdx.x; b < nb; b += gridDim.x * blockDim.x) {
    Ray ray = rays[b];
    if (ray.frame_clr == kNoRay) {
      ray_count[b] = 0;
      continue;
    }
    const Xform T = make_xform(poses + 7 * (ray.frame_clr & 0x7FFFFFFFu));
    const V3 pg = apply(T, V3{ray.px, ray.py, ray.pz});
    RayCaster rc;
    rc.init(T.t, pg, (ray.frame_clr >> 31) != 0, P.carving != 0, P.max_ray, P.voxel_size_inv,
            P.trunc);
    rays[b].px = pg.x;
    rays[b].py = pg.y;
    rays[b].pz = pg.z;
    ray_count[b] = rc.valid ? rc.packed_counts() : 0ull;
  }
}

// SIMPLE: one ray per valid point, in (frame, visit rank) order
struct ValidSlot {
  IntegratorParams P;
  FrameTable ft;
  const float* pts;
  __device__ __forceinline__ bool operator()(uint32_t g) const {
    const int f = ft.frame_of(g);
    const uint64_t base = ft.start(f);
    const int n = static_cast<int>(ft.start(f + 1) - base);
    bool clearing;
    return point_valid(P, load_point(pts, base + order_index(static_cast<int>(g - base), n,
                                                             P.order_mode)), &clearing);
  }
};

__global__ void k_simple_rays(IntegratorParams P, const float* __restrict__ poses, FrameTable ft,
                              const uint32_t* __restrict__ slots,
                              const uint32_t* __restrict__ num_slots, const float* __restrict__ pts,
                              const uint32_t* __restrict__ cols, Ray* __restrict__ rays,
                              unsigned long long* __restrict__ ray_count) {
  const uint32_t r = blockIdx.x * blockDim.x + threadIdx.x;
  if (r >= *num_slots) return;
  const uint32_t g = slots[r];
  const int f = ft.frame_of(g);
  const uint64_t base = ft.start(f);
  const int n = static_cast<int>(ft.start(f + 1) - base);
  const size_t i = base + order_index(static_cast<int>(g - base), n, P.order_mode);
  const V3 pc = load_point(pts, i);
  bool clearing = false;
  point_valid(P, pc, &clearing);
  const Xform T = make_xform(poses + 7 * f);
  const V3 pg = apply(T, pc);
  RayCaster rc;
  rc.init(T.t, pg, clearing, P.carving != 0, P.max_ray, P.voxel_size_inv, P.trunc);
  Ray ray;
  ray.px = pg.x;
  ray.py = pg.y;
  ray.pz = pg.z;
  ray.weight = voxel_weight(P, pc.z);
  ray.color = cols[i];
  ray.frame_clr = static_cast<uint32_t>(f) | (clearing ? 0x80000000u : 0u);
  rays[r] = ray;
  ray_count[r] = rc.valid ? rc.packed_counts() : 0ull;
}

// Exclusive scan of the packed per-ray counts over the first *num_rays entries only (the host
// knows just the upper bound "one ray per point", 25x larger at the C2 shape): per-CTA partial
// sums over contiguous ranges, a one-CTA scan of the partials, then a block scan per range.
constexpr int kScanThreads = 256;
__device__ __forceinline__ void scan_range(uint32_t n, uint32_t& lo, uint32_t& hi) {
  const uint32_t per = (n + gridDim.x - 1) / gridDim.x;
  lo = min(n, blockIdx.x * per);
  hi = min(n, lo + per);
}
__global__ void __launch_bounds__(kScanThreads)
k_scan_partials(const uint32_t* __restrict__ num_rays, const unsigned long long* __restrict__ in,
                unsigned long long* __restrict__ partials) {
  typedef cub::BlockReduce<unsigned long long, kScanThreads> Reduce;
  __shared__ typename Reduce::TempStorage tmp;
  uint32_t lo, hi;
  scan_range(*num_rays, lo, hi);
  unsigned long long sum = 0;
  for (uint32_t i = lo + threadIdx.x; i < hi; i += kScanThreads) sum += in[i];
  sum = Reduce(tmp).Sum(sum);
  if (threadIdx.x == 0) partials[blockIdx.x] = sum;
}
// one CTA: exclusive scan of the partials in place; totals -> counters
__global__ void __launch_bounds__(1024)
k_scan_totals(const uint32_t* __restrict__ num_rays, unsigned long long* __restrict__ partials,
              int num_partials, CallCounters* c, int32_t* err, int* key_bounds) {
  typedef cub::BlockScan<unsigned long long, 1024> Scan;
  __shared__ typename Scan::TempStorage tmp;
  unsigned long long v = static_cast<int>(threadIdx.x) < num_partials ? partials[threadIdx.x] : 0ull;
  unsigned long long total = 0;
  Scan(tmp).ExclusiveSum(v, v, total);
  if (static_cast<int>(threadIdx.x) < num_partials) partials[threadIdx.x] = v;
  if (threadIdx.x == 0) {
    // a point outside the group's key layout: the host widens it / regroups (atomic: a prepared
    // front half runs beside another job's back half, which may flag errors in the same word)
    const int e = atomicAnd(err, ~kErrKeyRange);
    c->err = e & (kErrKeyRange | kErrOutOfRange);
    for (int a = 0; a < 3; ++a) {
      c->key_lo[a] = key_bounds[a];
      c->key_hi[a] = key_bounds[3 + a];
      key_bounds[a] = 0x3FFFFFFF;
      key_bounds[3 + a] = -0x3FFFFFFF;
    }
    c->rays = *num_rays;
    c->far_dropped = c->far_points;  // counted by k_point_keys; reset for the next front half
    c->far_points = 0;
    c->pairs = total & 0xFFFFFFFFull;  // voxel visits (the host splits jobs that reach 2^32)
    c->segments = total >> 32;         // (ray, block) segments
    c->touched = 0;
  }
}
__global__ void __launch_bounds__(kScanThreads)
k_scan_apply(const uint32_t* __restrict__ num_rays, const unsigned long long* __restrict__ in,
             const unsigned long long* __restrict__ partials, unsigned long long* __restrict__ out) {
  typedef cub::BlockScan<unsigned long long, kScanThreads> Scan;
  __shared__ typename Scan::TempStorage tmp;
  uint32_t lo, hi;
  scan_range(*num_rays, lo, hi);
  unsigned long long running = partials[blockIdx.x];
  for (uint32_t i0 = lo; i0 < hi; i0 += kScanThreads) {
    const uint32_t i = i0 + threadIdx.x;
    const unsigned long long v = i < hi ? in[i] : 0ull;
    unsigned long long ex, agg;
    Scan(tmp).ExclusiveSum(v, ex, agg);
    if (i < hi) out[i] = running + ex;
    running += agg;
    __syncthreads();
  }
}

// ------------------------------------------------------------------ back half
// The voxels a job visits fall in two classes.  Nearly all of them (the carved free space) only
// ever see observations with sdf >= truncation while being fresh or already saturated at
// +truncation: for those updateTsdfVoxel degenerates to "D = trunc, W = min(max_weight, W + sum
// of the ray weights)", which needs no ordering — a fixed-point sum per voxel (deterministic, the
// adds commute exactly).  The rest ("general" voxels: any observation inside the truncation band
// or behind the surface, or a previous state that is not saturated) replay their updates in the
// reference's order.  Two walks over the rays:
//   k_walk_accumulate  DDA (voxblox::RayCaster), block allocation on first visit (R4), weight
//                      accumulation for every visit, "general" bit for every visit whose sdf is
//                      below the truncation distance (only the tail of a ray can be)
//   k_mark_existing    voxels of previously existing blocks whose state is not saturated
//   k_walk_emit        DDA again; visits of general voxels are appended as (voxel, ray) keys
//   radix sort         keys only: per-voxel update lists in ray (= canonical) order
//   k_voxel_update     ordered replay of the general voxels
//   k_finalize_blocks  one CTA per touched block: coalesced read-modify-write of the remaining
//                      voxels from the accumulators; resets the per-call scratch.

// Per-call "touch set": a block gets an ordinal when the first ray of the job visits it; the
// per-call scratch is indexed by ordinal.
struct TouchView {
  int32_t* ord;             // [hash_cap]   hash entry -> ordinal; -1 untouched, -2 being claimed
  uint32_t* entry;          // [cap]        ordinal -> hash entry
  unsigned long long* acc;  // [cap * 4096] fixed-point sum of the ray weights of all visits
  uint32_t* general;        // [cap * 128]  bit per voxel: replay its updates in order
  uint32_t* count;          // ordinals claimed (exceeds cap on overflow: the job is redone)
  uint32_t cap;
};

__device__ __forceinline__ uint32_t touch_ordinal(const TouchView& Tv, int entry, int32_t* err) {
  volatile int32_t* p = Tv.ord + entry;
  for (;;) {
    const int32_t o = *p;
    if (o >= 0) return static_cast<uint32_t>(o);
    if (o == -1 && atomicCAS(Tv.ord + entry, -1, -2) == -1) {
      uint32_t n = atomicAdd(Tv.count, 1u);
      if (n < Tv.cap) {
        Tv.entry[n] = static_cast<uint32_t>(entry);
      } else {
        atomicOr(err, kErrTouchFull);
        n = n % Tv.cap;  // stays addressable; the host grows the scratch and redoes the walks
      }
      __threadfence();
      *p = static_cast<int32_t>(n);
      return n;
    }
  }
}

constexpr int kWalkThreads = 128;

// Per-CTA direct-mapped cache block index -> ordinal in shared memory.  The rays of a CTA are
// neighbours (bundles are sorted by voxel), so they cross the same few blocks; a hit replaces the
// two dependent L2 round trips of the hash probe and the ordinal lookup.  One 64-bit word per
// entry (tag << 20 | ordinal), written with a single store, so a reader never sees a torn pair.
// Ordinals are immutable for the duration of the job.
constexpr int kBlockCacheSize = 512;
__device__ __forceinline__ bool block_cache_tag(int bx, int by, int bz, unsigned long long& tag,
                                                uint32_t& idx) {
  const uint32_t ux = static_cast<uint32_t>(bx + 8192), uy = static_cast<uint32_t>(by + 8192),
                 uz = static_cast<uint32_t>(bz + 8192);
  if ((ux | uy | uz) >> 14) return false;  // far from the origin: not cached
  tag = ((static_cast<unsigned long long>(uz) << 28) | (static_cast<unsigned long long>(uy) << 14) |
         ux) + 1ull;
  idx = (ux + 7u * uy + 61u * uz) & (kBlockCacheSize - 1);
  return true;
}
// dynamic work distribution: each warp takes the next batch of 32 consecutive rays
__device__ __forceinline__ uint32_t next_ray_batch(uint32_t* work_counter, int lane) {
  uint32_t b = 0;
  if (lane == 0) b = atomicAdd(work_counter, 1u);
  return __shfl_sync(0xFFFFFFFFu, b, 0);
}

struct WalkRay {
  RayCaster rc;
  Ray ray;
  V3 origin;  // sensor origin of the ray's frame
  uint32_t remaining;
};
__device__ __forceinline__ WalkRay load_walk_ray(const IntegratorParams& P,
                                                 const float* __restrict__ poses,
                                                 const Ray* __restrict__ rays, uint32_t r,
                                                 uint32_t num_rays, int32_t* err) {
  WalkRay w;
  w.rc.valid = false;
  w.rc.steps = 0;
  w.ray.frame_clr = kNoRay;
  w.ray.weight = 0.0f;
  w.origin = V3{0.0f, 0.0f, 0.0f};
  if (r < num_rays) {
    w.ray = rays[r];
    if (w.ray.frame_clr != kNoRay) {
      const float* T = poses + 7 * (w.ray.frame_clr & 0x7FFFFFFFu);
      w.origin = V3{T[4], T[5], T[6]};
      w.rc.init(w.origin, V3{w.ray.px, w.ray.py, w.ray.pz},
                (w.ray.frame_clr >> 31) != 0, P.carving != 0, P.max_ray, P.voxel_size_inv, P.trunc);
      if (!w.rc.valid && !w.rc.in_range && err) atomicOr(err, kErrOutOfRange);
    }
  }
  w.remaining = w.rc.valid ? w.rc.steps + 1u : 0u;
  return w;
}

// state-independent part of updateTsdfVoxel for one (ray, voxel) visit
struct Visit {
  float sdf, w;
  uint32_t col;
};
__device__ __forceinline__ Visit make_visit(const IntegratorParams& P, V3 origin, const Ray& ray,
                                            V3 center) {
  const V3 pg = V3{ray.px, ray.py, ray.pz};
  // computeDistance + weight drop-off / sparsity compensation
  const V3 v_voxel_origin = center - origin;
  const V3 v_point_origin = pg - origin;
  const float dist_G = norm3(v_point_origin);
  const float dist_G_V = dot3(v_voxel_origin, v_point_origin) / dist_G;
  Visit v;
  v.sdf = dist_G - dist_G_V;
  v.w = ray.weight;
  if (P.weight_dropoff && v.sdf < -P.voxel_size) {
    v.w = v.w * (P.trunc + v.sdf) / (P.trunc - P.voxel_size);
    v.w = fmaxf(v.w, 0.0f);
  }
  if (P.use_sparsity && fabsf(v.sdf) < P.trunc) v.w *= P.sparsity_factor;
  v.col = ray.color;
  return v;
}
__device__ __forceinline__ Visit make_visit(const IntegratorParams& P, const float* __restrict__ poses,
                                            const Ray& ray, V3 center) {
  const float* T = poses + 7 * (ray.frame_clr & 0x7FFFFFFFu);
  return make_visit(P, V3{T[4], T[5], T[6]}, ray, center);
}

// MergedTsdfIntegrator's optional anti-grazing (R6): a ray skips every voxel that holds points
// of the same scan (i.e. that is the key of a non-clearing bundle of its frame) except, for a
// non-clearing ray, its own bundle voxel.  The set of bundle voxels is a scratch hash set keyed by
// (frame, voxel relative to the frame's sensor voxel).
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
__global__ void k_grazing_build(KeyLayout kl, const uint64_t* __restrict__ keys, uint32_t total,
                                const uint32_t* __restrict__ heads,
                                const uint32_t* __restrict__ num_heads,
                                const uint32_t* __restrict__ ray_id,
                                unsigned long long* set_keys, uint32_t set_mask,
                                unsigned long long* __restrict__ ray_key) {
  const uint32_t nb = *num_heads;
  for (uint32_t b = blockIdx.x * blockDim.x + threadIdx.x; b < nb; b += gridDim.x * blockDim.x) {
    const BundleInfo bi = bundle_info(keys, total, heads, nb, b);
    if (bi.key == kInvalidPointKey) continue;
    const int rx = kl.rel(bi.key, 0), ry = kl.rel(bi.key, 1), rz = kl.rel(bi.key, 2);
    const unsigned long long gk = grazing_key(kl.frame(bi.key), rx, ry, rz);
    ray_key[ray_id[b]] = gk;
    if (kl.clearing(bi.key)) continue;  // only non-clearing bundles are in the set
    uint32_t h = hash_key(gk) & set_mask;
    for (;;) {
      const unsigned long long k = set_keys[h];
      if (k == gk) break;
      if (k == kEmptyKey) {
        const unsigned long long old = atomicCAS(&set_keys[h], kEmptyKey, gk);
        if (old == kEmptyKey || old == gk) break;
      }
      h = (h + 1) & set_mask;
    }
  }
}

// (ray, block) segment: the part of a ray's walk that lies inside one 16^3 block, with the
// RayCaster state at its first voxel so that the block pass can replay it on its own.
struct SegRecord {      // 32 B
  uint32_t ray;
  uint32_t packed;      // lx | ly << 4 | lz << 8 | (sx+1) << 12 | (sy+1) << 14 | (sz+1) << 16 | visits << 18
  float tnx, tny, tnz;  // t_to_next_boundary at the first voxel
  float tsx, tsy, tsz;  // t_step_size
};
static_assert(sizeof(SegRecord) == 32, "SegRecord is written as two 16-byte stores");

// Walk.  One lane per ray, the warp advances in lock step: DDA exactly as voxblox::RayCaster,
// block allocation on first visit (R4), one SegRecord per (ray, block), "general" bit for every
// visit with sdf < truncation (only the last `tail_visits` visits of a ray can be such,
// walk_tail_visits()).  Ray r owns the record slots [seg_first(r), seg_first(r) + its closed-form
// block count + slack); unused slots get the null key.
template <bool kGrazing>
__global__ void __launch_bounds__(kWalkThreads)
k_walk_segments(IntegratorParams P, const float* __restrict__ poses, const Ray* __restrict__ rays,
                uint32_t num_rays, const unsigned long long* __restrict__ ray_count,
                const unsigned long long* __restrict__ ray_offset, uint32_t slack, LayerView L,
                TouchView Tv, uint32_t tail_visits, uint32_t null_key, uint32_t* work_counter,
                uint32_t* __restrict__ seg_keys, uint32_t* __restrict__ seg_idx,
                uint4* __restrict__ seg_recs, GrazingSet G) {
  __shared__ unsigned long long cache[kBlockCacheSize];
  const unsigned full = 0xFFFFFFFFu;
  const int lane = threadIdx.x & 31;
  for (int i = threadIdx.x; i < kBlockCacheSize; i += blockDim.x) cache[i] = 0ull;
  __syncthreads();
  for (;;) {
    const uint32_t r0 = next_ray_batch(work_counter, lane) * 32u;
    if (r0 >= num_rays) break;
    const uint32_t r = r0 + lane;
    WalkRay w = load_walk_ray(P, poses, rays, r, num_rays, L.err);
    RayCaster& rc = w.rc;
    uint32_t seg_pos = 0, seg_end = 0;
    if (r < num_rays) {
      seg_pos = static_cast<uint32_t>(ray_offset[r] >> 32) + r * slack;
      seg_end = seg_pos + static_cast<uint32_t>(ray_count[r] >> 32) + slack;
    }
    uint32_t ord = 0, s_entry = 0, s_visits = 0;
    float s_tnx = 0.0f, s_tny = 0.0f, s_tnz = 0.0f;
    // anti-grazing: sensor voxel of the ray's frame and the ray's own bundle voxel
    int svx = 0, svy = 0, svz = 0;
    unsigned long long own_key = kEmptyKey;
    uint32_t g_frame = 0;
    if (kGrazing && w.remaining > 0) {
      g_frame = w.ray.frame_clr & 0x7FFFFFFFu;
      const float* T = poses + 7 * g_frame;
      svx = grid_index(T[4], P.voxel_size_inv);
      svy = grid_index(T[5], P.voxel_size_inv);
      svz = grid_index(T[6], P.voxel_size_inv);
      if (!(w.ray.frame_clr >> 31)) own_key = G.ray_key[r];
    }
    const uint32_t sign_bits = (static_cast<uint32_t>(rc.sx + 1) << 12) |
                               (static_cast<uint32_t>(rc.sy + 1) << 14) |
                               (static_cast<uint32_t>(rc.sz + 1) << 16);
    auto emit = [&]() {
      if (seg_pos < seg_end) {
        seg_keys[seg_pos] = ord;
        seg_idx[seg_pos] = seg_pos;
        seg_recs[2 * size_t(seg_pos)] =
            make_uint4(r, s_entry | sign_bits | (s_visits << 18), __float_as_uint(s_tnx),
                       __float_as_uint(s_tny));
        seg_recs[2 * size_t(seg_pos) + 1] =
            make_uint4(__float_as_uint(s_tnz), __float_as_uint(rc.tsx), __float_as_uint(rc.tsy),
                       __float_as_uint(rc.tsz));
      } else {
        atomicOr(L.err, kErrSegmentFull);  // the host redoes the job with more slack
      }
      ++seg_pos;
    };
    {
      // The per-visit work is what this kernel issues.  (1) The lanes are aligned at the END of
      // their rays — a lane joins when the warp's countdown `left` reaches its own length, so all
      // rays of the warp finish together and the costly tail (sdf of the last visits) runs
      // converged — hence an active lane's remaining count IS `left`: "in the tail" and "last
      // visit" are warp-uniform, the tail code sits in a second loop, and neither a per-lane
      // counter nor a visit counter is kept (a segment's visit count is the difference of two
      // countdown values).  (2) The position inside the current block is one packed word,
      // (l + 64) per byte for x, y, z: a step is one add of the stepped axis' increment, "left the
      // block" one mask test; global voxel coordinates are rebuilt from the block origin only
      // where they are needed (a new block, the tail, the anti-grazing test).
      const uint32_t len = w.remaining;
      // the first voxel must look like a block entry: its x field is given one block too many
      int ox = (rc.cx & ~15) - 16, oy = rc.cy & ~15, oz = rc.cz & ~15;  // origin voxel of the block
      uint32_t loc = static_cast<uint32_t>(((rc.cx & 15) + 16 + 64) | (((rc.cy & 15) + 64) << 8) |
                                           (((rc.cz & 15) + 64) << 16));
      const int dx = rc.sx, dy = rc.sy * 256, dz = rc.sz * 65536;
      float tnx = rc.tnx, tny = rc.tny, tnz = rc.tnz;
      const float tsx = rc.tsx, tsy = rc.tsy, tsz = rc.tsz;
      uint32_t seg_left = 0;  // countdown value at the first voxel of the open segment (0: none)
      bool after_skip = false;  // anti-grazing: the voxel before was skipped, a new segment starts
      auto close_segment = [&](uint32_t left) {
        s_visits = seg_left - left;
        emit();
        seg_left = 0;
      };
      // RayCaster::step: first minimum wins ties, NaN in x sticks
      auto step = [&]() {
        const bool yx = tny < tnx;
        const bool pz = tnz < (yx ? tny : tnx);
        int d = yx ? dy : dx;
        d = pz ? dz : d;
        loc += static_cast<uint32_t>(d);
        if (pz) {
          tnz += tsz;
        } else if (yx) {
          tny += tsy;
        } else {
          tnx += tsx;
        }
      };
      auto visit = [&](uint32_t left, auto tail) {
        if (kGrazing) {
          const int cx = ox + static_cast<int>(loc & 0xFFu) - 64,
                    cy = oy + static_cast<int>((loc >> 8) & 0xFFu) - 64,
                    cz = oz + static_cast<int>((loc >> 16) & 0xFFu) - 64;
          const int rx = cx - svx, ry = cy - svy, rz = cz - svz;
          bool skip = false;
          if (abs(rx) < 8192 && abs(ry) < 8192 && abs(rz) < 8192) {
            const unsigned long long gk = grazing_key(g_frame, rx, ry, rz);
            skip = gk != own_key && grazing_contains(G, gk);
          }
          if (skip) {
            // the reference "continue"s before it even looks the voxel up: no allocation, no
            // update; the segment ends here and a new one starts at the next voxel that counts
            if (seg_left) close_segment(left);
            after_skip = true;
            step();
            return;
          }
        }
        if ((loc & 0x707070u) != 0x404040u || (kGrazing && after_skip)) {
          // the voxel lies in another block than the last one (or follows a skipped voxel)
          after_skip = false;
          if (seg_left) close_segment(left);
          const int cx = ox + static_cast<int>(loc & 0xFFu) - 64,
                    cy = oy + static_cast<int>((loc >> 8) & 0xFFu) - 64,
                    cz = oz + static_cast<int>((loc >> 16) & 0xFFu) - 64;
          ox = cx & ~15;
          oy = cy & ~15;
          oz = cz & ~15;
          s_entry = static_cast<uint32_t>((cx & 15) | ((cy & 15) << 4) | ((cz & 15) << 8));
          loc = static_cast<uint32_t>((cx & 15) | ((cy & 15) << 8) | ((cz & 15) << 16)) + 0x404040u;
          const int bx = cx >> 4, by = cy >> 4, bz = cz >> 4;
          unsigned long long tag = 0ull;
          uint32_t ci = 0;
          const bool cacheable = block_cache_tag(bx, by, bz, tag, ci);
          const unsigned long long cw = cacheable ? cache[ci] : 0ull;
          if (cacheable && (cw >> 20) == tag) {
            ord = static_cast<uint32_t>(cw & 0xFFFFFu);
          } else {
            const int entry = L.insert_entry(pack_block_key(bx, by, bz));
            ord = touch_ordinal(Tv, entry, L.err);
            if (cacheable) cache[ci] = (tag << 20) | ord;
          }
          seg_left = left;
          s_tnx = tnx;
          s_tny = tny;
          s_tnz = tnz;
        }
        if (decltype(tail)::value) {
          const int lx = static_cast<int>(loc & 0xFFu) - 64, ly = static_cast<int>((loc >> 8) & 0xFFu) - 64,
                    lz = static_cast<int>((loc >> 16) & 0xFFu) - 64;
          const V3 center = V3{center_coord(ox + lx, P.voxel_size), center_coord(oy + ly, P.voxel_size),
                               center_coord(oz + lz, P.voxel_size)};
          const float sdf = make_visit(P, w.origin, w.ray, center).sdf;
          if (!(sdf >= P.trunc)) {
            const uint32_t vid = (ord << 12) | static_cast<uint32_t>(lx + 16 * (ly + 16 * lz));
            atomicOr(Tv.general + (vid >> 5), 1u << (vid & 31));
          }
        }
        step();
      };
      uint32_t left = __reduce_max_sync(full, len);
      for (; left > tail_visits; --left)
        if (left <= len) visit(left, std::false_type());
      for (; left > 0; --left)
        if (left <= len) visit(left, std::true_type());
      if (seg_left) close_segment(0u);
    }
    for (; seg_pos < seg_end; ++seg_pos) {  // unused slots sort behind every real segment
      seg_keys[seg_pos] = null_key;
      seg_idx[seg_pos] = seg_pos;
    }
  }
}

// Voxels of blocks that existed before the job and whose state is neither fresh nor saturated
// at +truncation need the ordered replay even if the job only observes them as free space.
__global__ void __launch_bounds__(128)
k_mark_existing(IntegratorParams P, LayerView L, TouchView Tv, int32_t blocks_before) {
  const unsigned full = 0xFFFFFFFFu;
  const uint32_t n = min(*Tv.count, Tv.cap);
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  for (uint32_t o = blockIdx.x; o < n; o += gridDim.x) {
    const int slot = L.hash_vals[Tv.entry[o]];
    if (slot < 0 || slot >= blocks_before) continue;
    const float* dp = L.dist_plane(slot);
    const float* wp = L.weight_plane(slot);
    for (int word = warp; word < kVoxelsPerBlock / 32; word += 4) {
      const int lin = word * 32 + lane;
      const bool g = wp[lin] > 0.0f && dp[lin] != P.trunc;
      const unsigned m = __ballot_sync(full, g);
      if (lane == 0 && m) atomicOr(Tv.general + o * (kVoxelsPerBlock / 32) + word, m);
    }
  }
}

// Counting sort of the segment slots by block ordinal (a few hundred distinct values, no order
// needed inside a block): per-CTA histograms in shared memory, a scan of the global histogram,
// then each CTA reserves one range per ordinal and scatters its tile.  Replaces two library radix
// passes; unused (null) slots are dropped on the way.
constexpr int kSortBins = 4096;      // ordinals handled in shared memory
constexpr uint32_t kSortTile = 4096;  // slots per CTA round
__global__ void __launch_bounds__(256)
k_segment_hist(const uint32_t* __restrict__ keys, uint32_t num_slots, uint32_t null_key,
               uint32_t* __restrict__ hist) {
  __shared__ uint32_t s_hist[kSortBins];
  for (int i = threadIdx.x; i < kSortBins; i += blockDim.x) s_hist[i] = 0;
  __syncthreads();
  for (uint32_t t0 = blockIdx.x * kSortTile; t0 < num_slots; t0 += gridDim.x * kSortTile) {
    const uint32_t t1 = min(num_slots, t0 + kSortTile);
    for (uint32_t i = t0 + threadIdx.x; i < t1; i += blockDim.x) {
      const uint32_t k = keys[i];
      if (k < null_key) atomicAdd(&s_hist[k], 1u);
    }
  }
  __syncthreads();
  for (uint32_t i = threadIdx.x; i < null_key; i += blockDim.x)
    if (s_hist[i]) atomicAdd(&hist[i], s_hist[i]);
}
__global__ void __launch_bounds__(256)
k_segment_scatter(const uint32_t* __restrict__ keys, const uint32_t* __restrict__ idx,
                  uint32_t num_slots, uint32_t null_key, const uint32_t* __restrict__ bin_base,
                  uint32_t* __restrict__ cursor, uint32_t* __restrict__ keys_out,
                  uint32_t* __restrict__ idx_out) {
  __shared__ uint32_t s_cnt[kSortBins];   // per tile: count, then running position
  for (uint32_t t0 = blockIdx.x * kSortTile; t0 < num_slots; t0 += gridDim.x * kSortTile) {
    const uint32_t t1 = min(num_slots, t0 + kSortTile);
    for (uint32_t i = threadIdx.x; i < null_key; i += blockDim.x) s_cnt[i] = 0;
    __syncthreads();
    for (uint32_t i = t0 + threadIdx.x; i < t1; i += blockDim.x) {
      const uint32_t k = keys[i];
      if (k < null_key) atomicAdd(&s_cnt[k], 1u);
    }
    __syncthreads();
    for (uint32_t i = threadIdx.x; i < null_key; i += blockDim.x) {
      const uint32_t c = s_cnt[i];
      s_cnt[i] = c ? bin_base[i] + atomicAdd(&cursor[i], c) : 0u;  // start of this tile's range
    }
    __syncthreads();
    for (uint32_t i = t0 + threadIdx.x; i < t1; i += blockDim.x) {
      const uint32_t k = keys[i];
      if (k < null_key) {
        const uint32_t pos = atomicAdd(&s_cnt[k], 1u);
        keys_out[pos] = k;
        idx_out[pos] = idx[i];
      }
    }
    __syncthreads();
  }
}

// Block pass.  The segments are sorted by block; a CTA takes a chunk of the sorted list and, per
// block run inside it, replays the segments against a shared-memory tile of the block:
// fixed-point weight accumulation with shared-memory atomics (deterministic: integer adds
// commute), "general" test from the block's bit tile, general visits appended as
// (voxel << ray_bits | ray) keys (warp-staged, one global atomic per flush; the append order is
// irrelevant because the sort key contains the ray rank).  The tile is then added to the
// per-job accumulators in global memory — one add per touched voxel and chunk instead of one
// per visit (measured: per-visit global atomics cost 0.4 ms of a 0.6 ms walk on the C2 step).
constexpr int kAccThreads = 256;
constexpr uint32_t kSegChunk = 1024;  // segments per work item
constexpr uint32_t kTileMinRun = 64;   // shorter block runs add straight to global memory
constexpr int kEmitBuf = 128;
__global__ void __launch_bounds__(kAccThreads)
k_block_accumulate(IntegratorParams P, const Ray* __restrict__ rays,
                   const uint32_t* __restrict__ seg_keys, const uint32_t* __restrict__ seg_idx,
                   const uint4* __restrict__ seg_recs, uint32_t num_slots_host,
                   const uint32_t* __restrict__ bin_base, uint32_t null_key, TouchView Tv,
                   float acc_scale, uint32_t ray_bits,
                   unsigned long long* __restrict__ out, uint32_t* out_count, uint32_t out_cap,
                   uint32_t* work_counter) {
  // Accumulators as two 20-bit limbs in 32-bit words: shared memory has native 32-bit atomic adds
  // only (a 64-bit add is a compare-and-swap loop).  A segment visits a voxel at most once (the
  // walk is monotone), so a tile sees at most kSegChunk <= 2^11 adds per voxel before it is
  // flushed and neither limb sum can overflow; the fixed-point weights are below 2^40 (host).
  // No carry, no returned value to wait for, and the result is exact whatever the order.
  __shared__ uint32_t tile_lo[kVoxelsPerBlock], tile_hi[kVoxelsPerBlock];
  __shared__ uint32_t bits[kVoxelsPerBlock / 32];
  __shared__ unsigned long long buf[kAccThreads / 32][kEmitBuf];
  __shared__ uint32_t s_chunk;
  const unsigned full = 0xFFFFFFFFu;
  const int lane = threadIdx.x & 31, wib = threadIdx.x >> 5;
  const unsigned lt = (1u << lane) - 1u;
  // (through an opaque move: otherwise the compiler rematerialises the window base — five uniform
  // instructions — next to every use inside the loop)
  uint32_t s_lo, s_hi, s_bits;
  asm volatile("mov.u32 %0, %1;" : "=r"(s_lo) : "r"(static_cast<uint32_t>(__cvta_generic_to_shared(tile_lo))));
  asm volatile("mov.u32 %0, %1;" : "=r"(s_hi) : "r"(static_cast<uint32_t>(__cvta_generic_to_shared(tile_hi))));
  asm volatile("mov.u32 %0, %1;" : "=r"(s_bits) : "r"(static_cast<uint32_t>(__cvta_generic_to_shared(bits))));
  // counting-sort path: bin_base[o] = first sorted segment of block ordinal o, bin_base[null_key]
  // = number of real segments (only known on the device)
  const uint32_t num_slots = bin_base ? bin_base[null_key] : num_slots_host;
  uint32_t cnt = 0;
  auto flush = [&]() {
    __syncwarp();
    uint32_t base = 0;
    if (lane == 0) base = atomicAdd(out_count, cnt);
    base = __shfl_sync(full, base, 0);
    for (uint32_t i = lane; i < cnt; i += 32)
      if (base + i < out_cap) out[base + i] = buf[wib][i];
    __syncwarp();
    cnt = 0;
  };
  for (;;) {
    __syncthreads();
    if (threadIdx.x == 0) s_chunk = atomicAdd(work_counter, 1u);
    __syncthreads();
    const uint32_t c_lo = s_chunk * kSegChunk;
    if (c_lo >= num_slots) break;
    const uint32_t c_hi = min(num_slots, c_lo + kSegChunk);
    uint32_t pos = c_lo;
    while (pos < c_hi) {
      const uint32_t o = seg_keys[pos];
      if (o >= null_key) break;  // unused slots are sorted last
      uint32_t lo = pos, hi = c_hi;  // end of this block's run inside the chunk
      if (bin_base) {
        hi = min(c_hi, bin_base[o + 1]);
      } else {
        while (hi - lo > 1) {
          const uint32_t mid = (lo + hi) >> 1;
          if (seg_keys[mid] == o) lo = mid; else hi = mid;
        }
      }
      const bool use_tile = hi - pos >= kTileMinRun;
      if (use_tile)
        for (int i = threadIdx.x; i < kVoxelsPerBlock; i += kAccThreads) tile_lo[i] = tile_hi[i] = 0u;
      if (threadIdx.x < kVoxelsPerBlock / 32)
        bits[threadIdx.x] = Tv.general[size_t(o) * (kVoxelsPerBlock / 32) + threadIdx.x];
      __syncthreads();
      unsigned long long* acc = Tv.acc + size_t(o) * kVoxelsPerBlock;
      for (uint32_t i0 = pos + wib * 32; i0 < hi; i0 += kAccThreads) {
        const uint32_t i = i0 + lane;
        uint32_t visits = 0, ray = 0, lin = 0;
        int dx = 0, dy = 0, dz = 0;  // change of the linear voxel index per step along x / y / z
        float tnx = 0.0f, tny = 0.0f, tnz = 0.0f, tsx = 0.0f, tsy = 0.0f, tsz = 0.0f;
        unsigned long long wq = 0ull;
        if (i < hi) {
          const uint32_t slot = seg_idx[i];
          const uint4 ra = seg_recs[2 * size_t(slot)], rb = seg_recs[2 * size_t(slot) + 1];
          ray = ra.x;
          lin = (ra.y & 15u) + 16u * (((ra.y >> 4) & 15u) + 16u * ((ra.y >> 8) & 15u));
          dx = static_cast<int>((ra.y >> 12) & 3) - 1;
          dy = (static_cast<int>((ra.y >> 14) & 3) - 1) * 16;
          dz = (static_cast<int>((ra.y >> 16) & 3) - 1) * 256;
          visits = ra.y >> 18;
          tnx = __uint_as_float(ra.z);
          tny = __uint_as_float(ra.w);
          tnz = __uint_as_float(rb.x);
          tsx = __uint_as_float(rb.y);
          tsy = __uint_as_float(rb.z);
          tsz = __uint_as_float(rb.w);
          wq = __float2ull_rn(fminf(fmaxf(rays[ray].weight, 0.0f), P.max_weight) * acc_scale);
        }
        const uint32_t w_lo = static_cast<uint32_t>(wq) & 0xFFFFFu, w_hi = static_cast<uint32_t>(wq >> 20);
        const uint32_t vmax = __reduce_max_sync(full, visits);
        // the per-visit loop is what this kernel issues (~50 instructions per visit before): the
        // shared-memory operands are addressed through 32-bit shared-window addresses computed once
        // (the generic form recomputes the window base every iteration), the tile / no-tile choice
        // is made outside the loop, the step works on the linear voxel index
        auto replay = [&](auto tile) {
          for (uint32_t v = 0; v < vmax; ++v) {
            uint32_t g = 0;
            const uint32_t cur = lin;
            if (v < visits) {
              if (decltype(tile)::value) {
                asm volatile("red.shared.add.u32 [%0], %1;" ::"r"(s_lo + cur * 4u), "r"(w_lo) : "memory");
                asm volatile("red.shared.add.u32 [%0], %1;" ::"r"(s_hi + cur * 4u), "r"(w_hi) : "memory");
              } else {
                atomicAdd(acc + cur, wq);
              }
              uint32_t word;
              asm volatile("ld.shared.u32 %0, [%1];" : "=r"(word) : "r"(s_bits + (cur >> 5) * 4u));
              g = (word >> (cur & 31u)) & 1u;
              // RayCaster::step (first minimum wins ties) on the linear index: the segment ends
              // before the walk leaves the block, so the index stays inside it while it is used
              const bool yx = tny < tnx;
              const bool pz = tnz < (yx ? tny : tnx);
              int d = yx ? dy : dx;
              d = pz ? dz : d;
              lin += static_cast<uint32_t>(d);
              if (pz) {
                tnz += tsz;
              } else if (yx) {
                tny += tsy;
              } else {
                tnx += tsx;
              }
            }
            const unsigned gm = __ballot_sync(full, g != 0u);
            if (gm) {
              if (g) buf[wib][cnt + __popc(gm & lt)] =
                  (static_cast<unsigned long long>((o << 12) | cur) << ray_bits) | ray;
              cnt += __popc(gm);
              if (cnt > kEmitBuf - 32) flush();
            }
          }
        };
        if (use_tile) replay(std::true_type()); else replay(std::false_type());
      }
      __syncthreads();
      if (use_tile)
        for (int i = threadIdx.x; i < kVoxelsPerBlock; i += kAccThreads) {
          const unsigned long long a =
              (static_cast<unsigned long long>(tile_hi[i]) << 20) + tile_lo[i];
          if (a) atomicAdd(acc + i, a);
        }
      __syncthreads();
      pos = hi;
    }
  }
  if (cnt) flush();
}

struct SegmentHead {
  const unsigned long long* keys;
  uint32_t ray_bits;
  __device__ __forceinline__ bool operator()(uint32_t i) const {
    return i == 0 || (keys[i] >> ray_bits) != (keys[i - 1] >> ray_bits);
  }
};

// x -> clamp(a x + b, lo, hi), a >= 0.  Closed under composition.
struct ClampedAffine {
  float a, b, lo, hi;
};
__device__ __forceinline__ ClampedAffine compose(const ClampedAffine& f, const ClampedAffine& g) {
  // g after f
  ClampedAffine r;
  r.a = g.a * f.a;
  r.b = g.a * f.b + g.b;
  r.lo = fminf(fmaxf(g.a * f.lo + g.b, g.lo), g.hi);
  r.hi = fminf(fmaxf(g.a * f.hi + g.b, g.lo), g.hi);
  return r;
}
constexpr float kBig = 1.0e30f;

// voxel addressed by a pair key
struct VoxelRef {
  int slot;
  V3 center;
  float* dp;
  float* wp;
  uint32_t* cp;
};
__device__ __forceinline__ VoxelRef voxel_ref(const IntegratorParams& P, const LayerView& L,
                                              const TouchView& Tv, uint32_t vid) {
  VoxelRef r;
  const uint32_t entry = Tv.entry[vid >> 12];
  const int lin = static_cast<int>(vid & 4095u);
  r.slot = L.hash_vals[entry];
  int bx, by, bz;
  unpack_block_key(L.hash_keys[entry], bx, by, bz);
  r.center = V3{center_coord(bx * 16 + (lin & 15), P.voxel_size),
                center_coord(by * 16 + ((lin >> 4) & 15), P.voxel_size),
                center_coord(bz * 16 + (lin >> 8), P.voxel_size)};
  const int s = r.slot < 0 ? 0 : r.slot;
  r.dp = L.dist_plane(s) + lin;
  r.wp = L.weight_plane(s) + lin;
  r.cp = L.color_plane(s) + lin;
  return r;
}

// The state-independent part of every ordered update — signed distance along the ray, effective
// weight (drop-off, sparsity compensation), colour — computed by one thread per (voxel, ray) key,
// fully parallel and with coalesced stores: what is left for the ordered replay is the short
// dependent chain on (D, W, C).  Same operations, in the same order, as updateTsdfVoxel (R5).
__global__ void __launch_bounds__(256)
k_visit_precompute(IntegratorParams P, const float* __restrict__ poses, const Ray* __restrict__ rays,
                   const unsigned long long* __restrict__ keys, uint32_t ray_bits,
                   const uint32_t* __restrict__ num_keys_dev, uint32_t num_keys, LayerView L,
                   TouchView Tv, float4* __restrict__ visits) {
  const uint32_t n = num_keys_dev ? min(*num_keys_dev, num_keys) : num_keys;
  const uint32_t ray_mask = (1u << ray_bits) - 1u;
  for (uint32_t i = blockIdx.x * blockDim.x + threadIdx.x; i < n; i += gridDim.x * blockDim.x) {
    const unsigned long long key = keys[i];
    const uint32_t vid = static_cast<uint32_t>(key >> ray_bits);
    const uint32_t entry = Tv.entry[vid >> 12];
    const int lin = static_cast<int>(vid & 4095u);
    int bx, by, bz;
    unpack_block_key(L.hash_keys[entry], bx, by, bz);
    const V3 center = V3{center_coord(bx * 16 + (lin & 15), P.voxel_size),
                         center_coord(by * 16 + ((lin >> 4) & 15), P.voxel_size),
                         center_coord(bz * 16 + (lin >> 8), P.voxel_size)};
    const Visit v = make_visit(P, poses, rays[static_cast<uint32_t>(key) & ray_mask], center);
    visits[i] = make_float4(v.sdf, v.w, __uint_as_float(v.col), 0.0f);
  }
}
// second half of updateTsdfVoxel: one precomputed visit applied to the voxel state
__device__ __forceinline__ void apply_visit(const IntegratorParams& p, float sdf, float updated_weight,
                                            uint32_t color, VoxelState& v) {
  const float new_weight = v.w + updated_weight;
  if (new_weight < kEps) return;
  const float new_sdf = (sdf * updated_weight + v.d * v.w) / new_weight;
  if (fabsf(sdf) < p.trunc) v.c = blend_colors(v.c, v.w, color, updated_weight);
  v.d = (new_sdf > 0.0f) ? fminf(p.trunc, new_sdf) : fmaxf(-p.trunc, new_sdf);
  v.w = fminf(p.max_weight, new_weight);
}

// Replays updates [start, end) of one voxel on (D, W, C), 32 at a time: weights by prefix sum,
// the clamped weighted average as an ordered tree reduction of clamped affine maps, colours
// sequentially for the updates inside the truncation band.  The ray records of chunk c+1 and the
// ray ids of chunk c+2 are in flight while chunk c is reduced.
__device__ __forceinline__ void replay_segment(const IntegratorParams& P,
                                               const float4* __restrict__ visits, uint32_t start,
                                               uint32_t end, int lane, float& D, float& W,
                                               uint32_t& C) {
  const unsigned full = 0xFFFFFFFFu;
  float4 next = (start + lane < end) ? visits[start + lane] : make_float4(0.0f, 0.0f, 0.0f, 0.0f);
  for (uint32_t c0 = start; c0 < end; c0 += 32) {
    const float4 cur = next;
    if (c0 + 32 + lane < end) next = visits[c0 + 32 + lane];  // next chunk in flight
    const bool act = c0 + lane < end;
    Visit v;
    v.sdf = cur.x;
    v.w = act ? cur.y : 0.0f;
    v.col = __float_as_uint(cur.z);
    const float sdf = v.sdf;
    // "new_weight < kFloatEpsilon -> return" leaves the voxel untouched, weight included.  The
    // weights are >= 0, so updates are skipped only while the stored weight is still below
    // epsilon: every update before the first one with W + w >= epsilon (all of them see the same
    // W), none after it.  Skipped updates must not enter the running weight.
    const unsigned okb = __ballot_sync(full, act && !(W + v.w < kEps));
    const int first_ok = okb ? __ffs(okb) - 1 : 32;
    const bool skip = !act || lane < first_ok;
    const float w = skip ? 0.0f : v.w;
    // weights: W_k = min(max_weight, W_{k-1} + w_k)  ==  min(max_weight, W_0 + sum w)
    float pre = w;
#pragma unroll
    for (int d = 1; d < 32; d <<= 1) {
      const float o = __shfl_up_sync(full, pre, d);
      if (lane >= d) pre += o;
    }
    const float w_prev = fminf(P.max_weight, W + (pre - w));
    const float w_new = w_prev + w;
    const float inv = 1.0f / w_new;
    ClampedAffine f;
    f.a = skip ? 1.0f : w_prev * inv;
    f.b = skip ? 0.0f : (sdf * w) * inv;
    f.lo = skip ? -kBig : -P.trunc;
    f.hi = skip ? kBig : P.trunc;
#pragma unroll
    for (int d = 1; d < 32; d <<= 1) {  // ordered tree reduction into lane 0
      ClampedAffine g;
      g.a = __shfl_down_sync(full, f.a, d);
      g.b = __shfl_down_sync(full, f.b, d);
      g.lo = __shfl_down_sync(full, f.lo, d);
      g.hi = __shfl_down_sync(full, f.hi, d);
      if ((lane & (2 * d - 1)) == 0) f = compose(f, g);
    }
    const float fa = __shfl_sync(full, f.a, 0), fb = __shfl_sync(full, f.b, 0);
    const float flo = __shfl_sync(full, f.lo, 0), fhi = __shfl_sync(full, f.hi, 0);
    D = fminf(fmaxf(fa * D + fb, flo), fhi);
    // Colours (Color::blendTwoColors, rounded to uint8 after every blend) stay sequential over the
    // updates inside the truncation band, but only the 3-operation chain per channel: the blend
    // factors and products are computed by the update's own lane, the 4 channels run on 4 lanes.
    unsigned band = __ballot_sync(full, !skip && fabsf(sdf) < P.trunc);
    if (band) {
      const float total = w_prev + w;
      const float w1n = w_prev / total, w2n = w / total;
      const float pr0 = static_cast<float>(v.col & 255u) * w2n;
      const float pr1 = static_cast<float>((v.col >> 8) & 255u) * w2n;
      const float pr2 = static_cast<float>((v.col >> 16) & 255u) * w2n;
      const float pr3 = static_cast<float>(v.col >> 24) * w2n;
      float ch = static_cast<float>((C >> (8 * (lane & 3))) & 255u);
      while (band) {
        const int t = __ffs(band) - 1;
        band &= band - 1;
        const float a = __shfl_sync(full, w1n, t);
        const float q0 = __shfl_sync(full, pr0, t), q1 = __shfl_sync(full, pr1, t);
        const float q2 = __shfl_sync(full, pr2, t), q3 = __shfl_sync(full, pr3, t);
        const float mine = (lane & 2) ? ((lane & 1) ? q3 : q2) : ((lane & 1) ? q1 : q0);
        ch = round_half_away_pos(ch * a + mine);
      }
      const uint32_t k0 = static_cast<uint32_t>(__shfl_sync(full, ch, 0));
      const uint32_t k1 = static_cast<uint32_t>(__shfl_sync(full, ch, 1));
      const uint32_t k2 = static_cast<uint32_t>(__shfl_sync(full, ch, 2));
      const uint32_t k3 = static_cast<uint32_t>(__shfl_sync(full, ch, 3));
      C = pack_rgba(k0 & 255u, k1 & 255u, k2 & 255u, k3 & 255u);
    }
    const float w_after = skip ? w_prev : fminf(P.max_weight, w_new);
    W = __shfl_sync(full, w_after, 31);
  }
}

// Lists of kWideSegment updates or more are replayed by a warp each (k_long_finish); long
// segments (>= kLongSegment updates) are first split into sub-blocks that many warps reduce in
// parallel, see k_long_partials.
constexpr uint32_t kWideSegment = 96;
constexpr uint32_t kLongSegment = 2048;
constexpr uint32_t kLongSub = 1024;
struct LongSeg {
  uint32_t start, end;    // pair range
  uint32_t item_base;     // first sub-block index
  uint32_t pad;
};
struct LongPartial {
  float sum_w;            // sum of the effective weights of the sub-block
  uint32_t not_free;      // any update with sdf < trunc (not a pure free-space observation)
};

// Update lists ordered by size class (largest first), as the bundles are: the lanes of a warp
// then hold lists of nearly the same length, so they finish — and fetch their next list, a chain
// of dependent global loads — together instead of stalling one another every few updates.
__device__ __forceinline__ uint32_t segment_length(const uint32_t* __restrict__ seg_start, uint32_t ns,
                                                   uint32_t num_pairs, uint32_t sidx) {
  return ((sidx + 1 < ns) ? seg_start[sidx + 1] : num_pairs) - seg_start[sidx];
}
__global__ void k_segment_histogram(const uint32_t* __restrict__ seg_start,
                                    const uint32_t* __restrict__ num_segs, uint32_t num_pairs,
                                    uint32_t* class_count) {
  __shared__ uint32_t hist[kSizeClasses];
  if (threadIdx.x < kSizeClasses) hist[threadIdx.x] = 0;
  __syncthreads();
  const uint32_t ns = *num_segs;
  for (uint32_t i = blockIdx.x * blockDim.x + threadIdx.x; i < ns; i += gridDim.x * blockDim.x)
    atomicAdd(&hist[size_class(segment_length(seg_start, ns, num_pairs, i))], 1u);
  __syncthreads();
  if (threadIdx.x < kSizeClasses && hist[threadIdx.x])
    atomicAdd(&class_count[threadIdx.x], hist[threadIdx.x]);
}
// ... and the lists of kWideSegment updates or more go to the list of the warp-cooperative
// kernels, which so do not have to wait for k_voxel_update.
__global__ void k_segment_order(const uint32_t* __restrict__ seg_start,
                                const uint32_t* __restrict__ num_segs, uint32_t num_pairs,
                                uint32_t* class_count, uint32_t* __restrict__ order,
                                unsigned long long* long_counter, LongSeg* __restrict__ long_list,
                                uint32_t long_cap) {
  __shared__ uint32_t base[kSizeClasses];
  __shared__ uint32_t hist[kSizeClasses];
  __shared__ uint32_t offs[kSizeClasses];
  if (threadIdx.x == 0) {
    uint32_t acc = 0;
    for (int c = 0; c < kSizeClasses; ++c) {
      base[c] = acc;
      acc += class_count[c];
    }
  }
  const uint32_t ns = *num_segs;
  for (uint32_t i0 = blockIdx.x * blockDim.x; i0 < ns; i0 += gridDim.x * blockDim.x) {
    __syncthreads();
    if (threadIdx.x < kSizeClasses) hist[threadIdx.x] = 0;
    __syncthreads();
    const uint32_t i = i0 + threadIdx.x;
    int c = -1;
    uint32_t rank = 0;
    if (i < ns) {
      const uint32_t len = segment_length(seg_start, ns, num_pairs, i);
      c = size_class(len);
      rank = atomicAdd(&hist[c], 1u);
      if (len >= kWideSegment) {
        const uint32_t start = seg_start[i];
        const uint32_t nsub = len >= kLongSegment ? (len + kLongSub - 1) / kLongSub : 0u;
        // one 64-bit atomic hands out the list index (high word) and the sub-block range
        const unsigned long long old =
            atomicAdd(long_counter, (1ull << 32) | static_cast<unsigned long long>(nsub));
        const uint32_t idx = static_cast<uint32_t>(old >> 32);
        if (idx < long_cap) long_list[idx] = LongSeg{start, start + len, static_cast<uint32_t>(old), 0u};
      }
    }
    __syncthreads();
    if (threadIdx.x < kSizeClasses && hist[threadIdx.x])
      offs[threadIdx.x] = atomicAdd(&class_count[kSizeClasses + threadIdx.x], hist[threadIdx.x]);
    __syncthreads();
    if (c >= 0) order[base[c] + offs[c] + rank] = i;
  }
}

// General voxels, short update lists: persistent lanes, one voxel per lane at a time, the
// reference's updateTsdfVoxel applied update by update (R5, in the reference's own operation
// order).  Lists of kWideSegment updates or more go to a list for the warp-cooperative kernels
// below (k_long_partials / k_long_finish).
constexpr int kUpdateInner = 8;
__global__ void __launch_bounds__(128)
k_voxel_update(IntegratorParams P, const float4* __restrict__ visits,
               const unsigned long long* __restrict__ keys, uint32_t ray_bits, uint32_t num_pairs,
               const uint32_t* __restrict__ seg_start, const uint32_t* __restrict__ num_segs,
               const uint32_t* __restrict__ order, uint32_t* work_counter, LayerView L,
               TouchView Tv) {
  // A warp takes 32 consecutive lists of the size-class order (nearly equal lengths), one per
  // lane, and runs them to the end of the longest before it fetches the next 32: the chain of
  // dependent loads that sets a list up (order -> list bounds -> key -> block -> voxel state) is
  // paid once per batch.  (Handing a lane its next list as soon as it ran out stalled the whole
  // warp on that chain every few updates: 0.09 ms for 3 M warp instructions.)
  const unsigned full = 0xFFFFFFFFu;
  const int lane = threadIdx.x & 31;
  const uint32_t ns = *num_segs;
  for (;;) {
    uint32_t batch = 0;
    if (lane == 0) batch = atomicAdd(work_counter, 1u);
    batch = __shfl_sync(full, batch, 0);
    if (batch * 32u >= ns) break;
    const uint32_t oidx = batch * 32u + lane;
    uint32_t cur = 0, end = 0;
    VoxelRef vr;
    vr.dp = vr.wp = nullptr;
    vr.cp = nullptr;
    VoxelState st{0.0f, 0.0f, 0u};
    float4 q[kUpdateInner];  // the next visits of this lane's list, in flight
#pragma unroll
    for (int u = 0; u < kUpdateInner; ++u) q[u] = make_float4(0.0f, 0.0f, 0.0f, 0.0f);
    if (oidx < ns) {
      const uint32_t sidx = order[oidx];
      const uint32_t start = seg_start[sidx];
      const uint32_t stop = (sidx + 1 < ns) ? seg_start[sidx + 1] : num_pairs;
      if (stop - start < kWideSegment) {  // the others: k_long_partials / k_long_finish
        vr = voxel_ref(P, L, Tv, static_cast<uint32_t>(keys[start] >> ray_bits));
        if (vr.slot >= 0) {  // else: pool exhausted, error already flagged
          cur = start;
          end = stop;
#pragma unroll
          for (int u = 0; u < kUpdateInner; ++u)
            if (start + u < stop) q[u] = visits[start + u];
          st.d = *vr.dp;
          st.w = *vr.wp;
          st.c = *vr.cp;
        }
      }
    }
    // the precomputed visits stream through a kUpdateInner-deep register queue; what is sequential
    // per update is the short chain of apply_visit
    while (__any_sync(full, cur < end)) {
#pragma unroll
      for (int t = 0; t < kUpdateInner; ++t) {
        if (cur < end) {
          const float4 v = q[t];
          if (cur + kUpdateInner < end) q[t] = visits[cur + kUpdateInner];
          apply_visit(P, v.x, v.y, __float_as_uint(v.z), st);
          if (++cur >= end) {
            *vr.dp = st.d;
            *vr.wp = st.w;
            *vr.cp = st.c;
          }
        }
      }
    }
  }
}

// sub-block t of the long segments: sum of weights + "all free space" flag (one warp each)
__global__ void __launch_bounds__(256)
k_long_partials(IntegratorParams P, const float4* __restrict__ visits,
                const unsigned long long* __restrict__ long_counter,
                const LongSeg* __restrict__ long_list, uint32_t long_cap,
                LongPartial* __restrict__ partials) {
  const unsigned full = 0xFFFFFFFFu;
  const int lane = threadIdx.x & 31;
  const uint32_t warp = (blockIdx.x * blockDim.x + threadIdx.x) >> 5;
  const uint32_t num_warps = (gridDim.x * blockDim.x) >> 5;
  const unsigned long long cnt = *long_counter;
  const uint32_t nlong = min(static_cast<uint32_t>(cnt >> 32), long_cap);
  const uint32_t nitems = static_cast<uint32_t>(cnt);
  for (uint32_t t = warp; t < nitems; t += num_warps) {
    // long_list is ordered by item_base (both come from the same atomic): binary search
    uint32_t lo = 0, hi = nlong;
    while (hi - lo > 1) {
      const uint32_t mid = (lo + hi) >> 1;
      if (long_list[mid].item_base <= t) lo = mid; else hi = mid;
    }
    const LongSeg seg = long_list[lo];
    if (t < seg.item_base) continue;
    const uint32_t a = seg.start + (t - seg.item_base) * kLongSub;
    const uint32_t b = min(seg.end, a + kLongSub);
    float sum = 0.0f;
    bool not_free = false;
    for (uint32_t c0 = a; c0 < b; c0 += 32) {
      const uint32_t j = c0 + lane;
      float w = 0.0f;
      if (j < b) {
        const float4 v = visits[j];
        w = v.y;
        not_free = not_free || !(v.x >= P.trunc);
      }
#pragma unroll
      for (int d = 16; d >= 1; d >>= 1) w += __shfl_xor_sync(full, w, d);
      sum += w;
    }
    const bool any_not_free = __any_sync(full, not_free);
    if (lane == 0) partials[t] = LongPartial{sum, any_not_free ? 1u : 0u};
  }
}

// one warp per long segment: closed form when every update is a free-space observation of a
// voxel that is fresh or already at +truncation, otherwise the general replay.
__global__ void __launch_bounds__(256)
k_long_finish(IntegratorParams P, const float4* __restrict__ visits,
              const unsigned long long* __restrict__ keys, uint32_t ray_bits,
              const unsigned long long* __restrict__ long_counter,
              const LongSeg* __restrict__ long_list, uint32_t long_cap, LayerView L, TouchView Tv,
              const LongPartial* __restrict__ partials) {
  const int lane = threadIdx.x & 31;
  const uint32_t warp = (blockIdx.x * blockDim.x + threadIdx.x) >> 5;
  const uint32_t num_warps = (gridDim.x * blockDim.x) >> 5;
  const unsigned long long cnt = *long_counter;
  const uint32_t nlong = min(static_cast<uint32_t>(cnt >> 32), long_cap);
  for (uint32_t i = warp; i < nlong; i += num_warps) {
    const LongSeg seg = long_list[i];
    const VoxelRef vr = voxel_ref(P, L, Tv, static_cast<uint32_t>(keys[seg.start] >> ray_bits));
    if (vr.slot < 0) continue;  // pool exhausted, error already flagged
    float D = *vr.dp, W = *vr.wp;
    uint32_t C = *vr.cp;
    const bool is_long = seg.end - seg.start >= kLongSegment;
    const uint32_t nsub = is_long ? (seg.end - seg.start + kLongSub - 1) / kLongSub : 0u;
    float sum = 0.0f;
    bool not_free = !is_long;
    for (uint32_t t = 0; t < nsub; ++t) {  // fixed order: deterministic
      const LongPartial p = partials[seg.item_base + t];
      sum += p.sum_w;
      not_free = not_free || p.not_free != 0;
    }
    const bool fresh_or_saturated = (W == 0.0f) || (D == P.trunc);
    if (!not_free && fresh_or_saturated && P.trunc > 0.0f) {
      const float w_total = W + sum;
      if (!(w_total < kEps)) {
        D = P.trunc;
        W = fminf(P.max_weight, w_total);
      }
    } else {
      replay_segment(P, visits, seg.start, seg.end, lane, D, W, C);
    }
    if (lane == 0) {
      *vr.dp = D;
      *vr.wp = W;
      *vr.cp = C;
    }
  }
}

// One CTA per touched block: every voxel that is not general and was visited becomes
// (D = trunc, W = min(max_weight, W + sum of ray weights)) — coalesced read-modify-write of the
// weight and distance planes — and the per-call scratch of the block goes back to zero.
__global__ void __launch_bounds__(256)
k_finalize_blocks(IntegratorParams P, LayerView L, TouchView Tv, float acc_inv_scale) {
  const uint32_t o = blockIdx.x;
  const uint32_t entry = Tv.entry[o];
  const int slot = L.hash_vals[entry];
  unsigned long long* acc = Tv.acc + static_cast<size_t>(o) * kVoxelsPerBlock;
  uint32_t* bits = Tv.general + static_cast<size_t>(o) * (kVoxelsPerBlock / 32);
  float* dp = slot >= 0 ? L.dist_plane(slot) : nullptr;
  float* wp = slot >= 0 ? L.weight_plane(slot) : nullptr;
  for (int lin = threadIdx.x; lin < kVoxelsPerBlock; lin += blockDim.x) {
    const unsigned long long a = acc[lin];
    if (a != 0ull) {
      acc[lin] = 0ull;
      const bool general = (bits[lin >> 5] >> (lin & 31)) & 1u;
      if (!general && slot >= 0) {
        const float w_total = wp[lin] + static_cast<float>(a) * acc_inv_scale;
        if (!(w_total < kEps)) {
          dp[lin] = P.trunc;
          wp[lin] = fminf(P.max_weight, w_total);
        }
      }
    }
  }
  __syncthreads();
  if (threadIdx.x < kVoxelsPerBlock / 32) bits[threadIdx.x] = 0u;
  if (threadIdx.x == 0) {
    Tv.ord[entry] = -1;
    if (slot >= 0) L.updated[slot] = 1;
  }
}

// ------------------------------------------------------------------ host orchestration
static IntegratorParams make_params(const cg_layer* L, const cg_integrator_config* c, int freespace) {
  IntegratorParams P;
  P.trunc = c->default_truncation_distance;
  P.max_weight = c->max_weight;
  P.min_ray = c->min_ray_length_m;
  P.max_ray = c->max_ray_length_m;
  P.voxel_size = L->v.voxel_size;
  P.voxel_size_inv = L->v.voxel_size_inv;
  P.sparsity_factor = c->sparsity_compensation_factor;
  P.carving = c->voxel_carving_enabled;
  P.const_weight = c->use_const_weight;
  P.allow_clear = c->allow_clear;
  P.weight_dropoff = c->use_weight_dropoff;
  P.use_sparsity = c->use_sparsity_compensation_factor;
  P.order_mode = c->integration_order_mode;
  P.freespace = freespace;
  // anti-grazing belongs to the merged integrator only (the simple one never looks at it)
  P.anti_grazing = (c->enable_anti_grazing && c->method == CG_METHOD_MERGED) ? 1 : 0;
  return P;
}

static size_t env_size(const char* name, size_t dflt) {
  const char* s = getenv(name);
  if (!s || !*s) return dflt;
  return static_cast<size_t>(strtoull(s, nullptr, 10));
}

// number of trailing visits of a ray that can have sdf < truncation.  A visit with k DDA steps
// left lies at L1 voxel distance k from the end voxel, hence at Euclidean distance >=
// (k - 1.5) / sqrt(3) voxels from the ray end; the voxel centre is within sqrt(3)/2 voxels of
// the ray, and the end lies trunc behind the surface point, so sdf >= trunc is guaranteed once
// ((k - 1.5) / sqrt(3))^2 - 3/4 >= (2 trunc / voxel + 1/2)^2.  (Clearing rays end before the
// point: the same bound holds with more slack.)
static uint32_t walk_tail_visits(const IntegratorParams& P) {
  const float m = 2.0f * P.trunc * P.voxel_size_inv;
  const float k = 1.5f + 1.7321f * (m + 0.5f + 0.87f);
  return static_cast<uint32_t>(std::min(1.0e6f, ceilf(k))) + 2u;
}

static int ceil_log2(uint64_t v) {
  int b = 0;
  while ((uint64_t(1) << b) < v) ++b;
  return b;
}

// per-call touch scratch for at least `cap` blocks, all clear
static int32_t ensure_touch(cg_context* ctx, const cg_layer* L, size_t cap) {
  cudaStream_t s = ctx->stream;
  bool wipe = !ctx->touch_clean;
  const size_t ord_bytes = L->hash_cap * sizeof(int32_t);
  if (ctx->touch_ord.cap < ord_bytes) {
    CG_CUDA(ctx->touch_ord.reserve(ord_bytes));
    wipe = true;
  }
  if (cap > ctx->touch_cap) {
    CG_CUDA(ctx->touch_entry.reserve(cap * sizeof(uint32_t)));
    CG_CUDA(ctx->touch_acc.reserve(cap * kVoxelsPerBlock * sizeof(unsigned long long)));
    CG_CUDA(ctx->touch_bits.reserve(cap * (kVoxelsPerBlock / 32) * sizeof(uint32_t)));
    ctx->touch_cap = cap;
    wipe = true;
  }
  if (wipe) {
    CG_CUDA(fill_bytes(ctx->touch_ord.p, 0xFF, ctx->touch_ord.cap, s));
    CG_CUDA(fill_bytes(ctx->touch_acc.p, 0, ctx->touch_acc.cap, s));
    CG_CUDA(fill_bytes(ctx->touch_bits.p, 0, ctx->touch_bits.cap, s));
  }
  CG_CUDA(fill_bytes(ctx->d_touch_count, 0, 2 * sizeof(uint32_t), s));  // + pair count
  ctx->touch_clean = true;
  return CG_OK;
}

__global__ void k_collect_walk(LayerView L, const uint32_t* touch_count, CallCounters* c) {
  c->touched = touch_count[0];
  c->general_pairs = touch_count[1];
  c->num_blocks = min(*L.num_blocks, L.max_blocks);
  const int e = *L.err;
  c->err = e;
  if (e & (kErrTouchFull | kErrSegmentFull)) *L.err = e & ~(kErrTouchFull | kErrSegmentFull);
}

static int32_t run_back_half(cg_context* ctx, const FrontBufs& fb, cg_layer* L,
                             const IntegratorParams& P, uint32_t num_rays, size_t num_pairs,
                             size_t num_segments, cg_integrate_stats* stats) {
  cudaStream_t s = ctx->stream;
  if (num_pairs >= 0xFFFFFFF0ull) {
    set_error("too many voxel visits in one group");
    return CG_ERR_INVALID_ARG;
  }
  CG_CUDA(ctx->pkey_a.reserve(num_pairs * sizeof(unsigned long long)));
  CG_CUDA(ctx->pkey_b.reserve(num_pairs * sizeof(unsigned long long)));
  const uint32_t ray_bits = static_cast<uint32_t>(std::max(1, ceil_log2(num_rays)));
  const int weight_bits = ceil_log2(static_cast<uint64_t>(std::min(std::max(P.max_weight, 1.0f), 1.0e9f)) + 1);
  const int shift = std::max(0, std::min(40 - weight_bits, 62 - weight_bits - ceil_log2(uint64_t(num_rays) + 1)));
  const float acc_scale = ldexpf(1.0f, shift), acc_inv_scale = ldexpf(1.0f, -shift);
  const uint32_t tail_visits = walk_tail_visits(P);
  const unsigned walk_grid = std::min<unsigned>(grid_for(num_rays, kWalkThreads),
                                                static_cast<unsigned>(ctx->num_sms) * 10u);
  size_t cap = std::max<size_t>(ctx->touch_cap, std::min<size_t>(L->max_blocks, env_size("CG_TOUCH_CAP", 1024)));
  // spare record slots per ray: a walk can end one step off its closed-form end voxel; with
  // anti-grazing every skipped voxel also splits a segment
  uint32_t slack = static_cast<uint32_t>(env_size("CG_SEGMENT_SLACK", P.anti_grazing ? 8 : 1));
  uint32_t n_touched = 0, n_general = 0;
  int64_t blocks_after = L->num_blocks;
  for (;;) {
    int32_t rc = ensure_touch(ctx, L, cap);
    if (rc) return rc;
    ctx->touch_clean = false;
    TouchView tv{ctx->touch_ord.as<int32_t>(), ctx->touch_entry.as<uint32_t>(),
                 ctx->touch_acc.as<unsigned long long>(), ctx->touch_bits.as<uint32_t>(),
                 ctx->d_touch_count, static_cast<uint32_t>(ctx->touch_cap)};
    // record slots: the closed-form block count of every ray + `slack` spare slots per ray
    const size_t num_slots = num_segments + size_t(num_rays) * slack;
    if (num_slots >= 0xFFFFFFF0ull) {
      set_error("too many (ray, block) segments in one group");
      return CG_ERR_INVALID_ARG;
    }
    CG_CUDA(ctx->seg_keys_a.reserve(num_slots * sizeof(uint32_t)));
    CG_CUDA(ctx->seg_keys_b.reserve(num_slots * sizeof(uint32_t)));
    CG_CUDA(ctx->seg_idx_a.reserve(num_slots * sizeof(uint32_t)));
    CG_CUDA(ctx->seg_idx_b.reserve(num_slots * sizeof(uint32_t)));
    CG_CUDA(ctx->seg_recs.reserve(num_slots * sizeof(SegRecord)));
    const int ord_bits = std::max(1, ceil_log2(ctx->touch_cap));
    const uint32_t null_key = 1u << ord_bits;  // above every ordinal
    cub::DoubleBuffer<uint32_t> sk(ctx->seg_keys_a.as<uint32_t>(), ctx->seg_keys_b.as<uint32_t>());
    cub::DoubleBuffer<uint32_t> sv(ctx->seg_idx_a.as<uint32_t>(), ctx->seg_idx_b.as<uint32_t>());
    size_t tmp_seg = 0;
    CG_CUDA(cub::DeviceRadixSort::SortPairs(nullptr, tmp_seg, sk, sv, static_cast<int>(num_slots), 0,
                                            ord_bits + 1, s));
    CG_CUDA(ctx->cub_tmp.reserve(tmp_seg));
    CG_CUDA(fill_bytes(ctx->d_walk_counters, 0, 2 * sizeof(uint32_t), s));
    {
      StageScope sc(ctx, kStageWalkSegments, 2);
      const GrazingSet gz{fb.grazing_keys.as<unsigned long long>(), fb.grazing_mask,
                          fb.grazing_ray_key.as<unsigned long long>()};
      if (P.anti_grazing)
        k_walk_segments<true><<<walk_grid, kWalkThreads, 0, s>>>(
            P, fb.group_poses, fb.rays.as<Ray>(), num_rays,
            fb.ray_count.as<unsigned long long>(), fb.ray_offset.as<unsigned long long>(),
            slack, L->v, tv, tail_visits, null_key, ctx->d_walk_counters, sk.Current(),
            sv.Current(), ctx->seg_recs.as<uint4>(), gz);
      else
        k_walk_segments<false><<<walk_grid, kWalkThreads, 0, s>>>(
            P, fb.group_poses, fb.rays.as<Ray>(), num_rays,
            fb.ray_count.as<unsigned long long>(), fb.ray_offset.as<unsigned long long>(),
            slack, L->v, tv, tail_visits, null_key, ctx->d_walk_counters, sk.Current(),
            sv.Current(), ctx->seg_recs.as<uint4>(), gz);
      if (L->num_blocks > 0)
        k_mark_existing<<<ctx->num_sms * 4, 128, 0, s>>>(P, L->v, tv,
                                                         static_cast<int32_t>(L->num_blocks));
    }
    const uint32_t* sorted_keys = nullptr;
    const uint32_t* sorted_idx = nullptr;
    const uint32_t* num_real = nullptr;
    if (null_key <= static_cast<uint32_t>(kSortBins)) {
      StageScope sc(ctx, kStageSegmentSort, 3);
      // hist[null_key + 1] | bin_base[null_key + 1] | cursor[null_key]
      const size_t words = 3 * (size_t(null_key) + 1);
      CG_CUDA(ctx->seg_bins.reserve(words * sizeof(uint32_t)));
      uint32_t* hist = ctx->seg_bins.as<uint32_t>();
      uint32_t* bin_base = hist + null_key + 1;
      uint32_t* cursor = bin_base + null_key + 1;
      CG_CUDA(fill_bytes(hist, 0, words * sizeof(uint32_t), s));
      const unsigned sgrid = std::min<unsigned>(grid_for(num_slots, kSortTile), ctx->num_sms * 4u);
      k_segment_hist<<<sgrid, 256, 0, s>>>(sk.Current(), static_cast<uint32_t>(num_slots), null_key,
                                           hist);
      size_t tmp_bins = 0;
      CG_CUDA(cub::DeviceScan::ExclusiveSum(nullptr, tmp_bins, hist, bin_base,
                                            static_cast<int>(null_key + 1), s));
      if (tmp_bins > ctx->cub_tmp.cap) CG_CUDA(ctx->cub_tmp.reserve(tmp_bins));
      CG_CUDA(cub::DeviceScan::ExclusiveSum(ctx->cub_tmp.p, tmp_bins, hist, bin_base,
                                            static_cast<int>(null_key + 1), s));
      k_segment_scatter<<<sgrid, 256, 0, s>>>(sk.Current(), sv.Current(),
                                              static_cast<uint32_t>(num_slots), null_key, bin_base,
                                              cursor, sk.Alternate(), sv.Alternate());
      sorted_keys = sk.Alternate();
      sorted_idx = sv.Alternate();
      num_real = bin_base;  // run boundaries; [null_key] = total number of real segments
    } else {
      StageScope sc(ctx, kStageSegmentSort, 0);
      CG_CUDA(cub::DeviceRadixSort::SortPairs(ctx->cub_tmp.p, tmp_seg, sk, sv,
                                              static_cast<int>(num_slots), 0, ord_bits + 1, s));
      sorted_keys = sk.Current();
      sorted_idx = sv.Current();
    }
    {
      StageScope sc(ctx, kStageBlockAccumulate, 2);
      k_block_accumulate<<<ctx->num_sms * 5, kAccThreads, 0, s>>>(
          P, fb.rays.as<Ray>(), sorted_keys, sorted_idx, ctx->seg_recs.as<uint4>(),
          static_cast<uint32_t>(num_slots), num_real, null_key, tv, acc_scale, ray_bits,
          ctx->pkey_a.as<unsigned long long>(), ctx->d_touch_count + 1,
          static_cast<uint32_t>(num_pairs), ctx->d_walk_counters + 1);
      k_collect_walk<<<1, 1, 0, s>>>(L->v, ctx->d_touch_count, ctx->d_counters);
    }
    CG_CUDA(cudaMemcpyAsync(ctx->h_counters, ctx->d_counters, sizeof(CallCounters),
                            cudaMemcpyDeviceToHost, s));
    CG_CUDA(cudaStreamSynchronize(s));
    CG_CUDA(cudaGetLastError());
    n_touched = static_cast<uint32_t>(ctx->h_counters->touched);
    n_general = static_cast<uint32_t>(ctx->h_counters->general_pairs);
    blocks_after = ctx->h_counters->num_blocks;
    const int err = ctx->h_counters->err;
    if (!(err & (kErrTouchFull | kErrSegmentFull))) break;
    if (err & kErrTouchFull) {
      // more blocks touched than the scratch holds: grow it (wiped by ensure_touch) and redo
      cap = 1024;
      while (cap < n_touched + n_touched / 4) cap <<= 1;
      if (cap > (size_t(1) << 19)) {
        set_error("a single job touches %u blocks; split the point cloud", n_touched);
        return CG_ERR_INVALID_ARG;
      }
    }
    if (err & kErrSegmentFull) {
      // a walk ended off its closed-form end voxel by more steps than the slack allows
      if (slack >= 256) {
        set_error("ray walk needs more than its closed-form block count + 256 segment records");
        return CG_ERR_INVALID_ARG;
      }
      slack *= 4;
    }
  }
  TouchView tv{ctx->touch_ord.as<int32_t>(), ctx->touch_entry.as<uint32_t>(),
               ctx->touch_acc.as<unsigned long long>(), ctx->touch_bits.as<uint32_t>(),
               ctx->d_touch_count, static_cast<uint32_t>(ctx->touch_cap)};
  if (n_general > num_pairs) n_general = static_cast<uint32_t>(num_pairs);  // cannot happen
  if (n_general > 0) {
    CG_CUDA(ctx->seg_start.reserve(size_t(n_general) * sizeof(uint32_t)));
    uint32_t* d_num = ctx->d_select_count;
    cub::DoubleBuffer<unsigned long long> dk(ctx->pkey_a.as<unsigned long long>(),
                                             ctx->pkey_b.as<unsigned long long>());
    const int key_bits = static_cast<int>(ray_bits) + 12 + std::max(1, ceil_log2(n_touched));
    size_t tmp = 0, tmp2 = 0;
    CG_CUDA(cub::DeviceRadixSort::SortKeys(nullptr, tmp, dk, static_cast<int>(n_general), 0,
                                           key_bits, s));
    thrust::counting_iterator<uint32_t> iota(0);
    CG_CUDA(cub::DeviceSelect::If(nullptr, tmp2, iota, ctx->seg_start.as<uint32_t>(), d_num,
                                  static_cast<int>(n_general), SegmentHead{nullptr, ray_bits}, s));
    CG_CUDA(ctx->cub_tmp.reserve(std::max(tmp, tmp2)));
    {
      StageScope sc(ctx, kStagePairSort, 0);
      CG_CUDA(cub::DeviceRadixSort::SortKeys(ctx->cub_tmp.p, tmp, dk, static_cast<int>(n_general), 0,
                                             key_bits, s));
    }
    {
      StageScope sc(ctx, kStageSegments, 0);
      CG_CUDA(cub::DeviceSelect::If(ctx->cub_tmp.p, tmp2, iota, ctx->seg_start.as<uint32_t>(), d_num,
                                    static_cast<int>(n_general),
                                    SegmentHead{dk.Current(), ray_bits}, s));
    }
    {  // the state-independent part of every ordered update, one thread per key
      StageScope sc(ctx, kStageVisits, 1);
      CG_CUDA(ctx->visits.reserve(size_t(n_general) * sizeof(float4)));
      k_visit_precompute<<<std::min<unsigned>(grid_for(n_general, 256), ctx->num_sms * 16u), 256, 0, s>>>(
          P, fb.group_poses, fb.rays.as<Ray>(), dk.Current(), ray_bits, nullptr, n_general, L->v, tv,
          ctx->visits.as<float4>());
    }
    const uint32_t long_cap = static_cast<uint32_t>(n_general / kWideSegment + 1);
    const size_t max_items = n_general / kLongSub + long_cap + 1;
    CG_CUDA(ctx->long_list.reserve(long_cap * sizeof(LongSeg)));
    CG_CUDA(ctx->long_partials.reserve(max_items * sizeof(LongPartial)));
    CG_CUDA(ctx->seg_order.reserve(size_t(n_general) * sizeof(uint32_t)));
    // lists shorter than kWideSegment (one lane each) beside the longer ones (a warp each): they
    // update different voxels
    FrontBufs& own = *ctx;  // the context's own side stream (fb may be a prepared set)
    const bool forked = side_stream(own, s);
    const cudaStream_t ls = forked ? own.side : s;
    {
      StageScope sc(ctx, kStageVoxelUpdate, 3);
      CG_CUDA(fill_bytes(ctx->d_work_counter, 0, sizeof(uint32_t), s));
      CG_CUDA(fill_bytes(ctx->d_long_counter, 0, sizeof(unsigned long long), s));
      CG_CUDA(fill_bytes(ctx->d_class_count, 0, 2 * kSizeClasses * sizeof(uint32_t), s));
      const unsigned ogrid = std::min<unsigned>(grid_for(n_general, 256), ctx->num_sms * 4u);
      k_segment_histogram<<<ogrid, 256, 0, s>>>(ctx->seg_start.as<uint32_t>(), d_num, n_general,
                                                ctx->d_class_count);
      k_segment_order<<<ogrid, 256, 0, s>>>(ctx->seg_start.as<uint32_t>(), d_num, n_general,
                                            ctx->d_class_count, ctx->seg_order.as<uint32_t>(),
                                            ctx->d_long_counter, ctx->long_list.as<LongSeg>(), long_cap);
      if (forked) {
        CG_CUDA(cudaEventRecord(own.ev_fork, s));
        CG_CUDA(cudaStreamWaitEvent(own.side, own.ev_fork, 0));
      }
      k_voxel_update<<<ctx->num_sms * 8, 128, 0, s>>>(
          P, ctx->visits.as<float4>(), dk.Current(), ray_bits, n_general,
          ctx->seg_start.as<uint32_t>(), d_num, ctx->seg_order.as<uint32_t>(), ctx->d_work_counter,
          L->v, tv);
    }
    {
      StageScope sc(ctx, kStageReplayWide, 2, ls);
      k_long_partials<<<ctx->num_sms * 8, 256, 0, ls>>>(
          P, ctx->visits.as<float4>(), ctx->d_long_counter, ctx->long_list.as<LongSeg>(), long_cap,
          ctx->long_partials.as<LongPartial>());
      k_long_finish<<<ctx->num_sms * 4, 256, 0, ls>>>(
          P, ctx->visits.as<float4>(), dk.Current(), ray_bits,
          ctx->d_long_counter, ctx->long_list.as<LongSeg>(), long_cap, L->v, tv,
          ctx->long_partials.as<LongPartial>());
    }
    if (forked) {
      CG_CUDA(cudaEventRecord(own.ev_join, own.side));
      CG_CUDA(cudaStreamWaitEvent(s, own.ev_join, 0));
    }
  }
  if (n_touched > 0) {
    StageScope sc(ctx, kStageFinalize, 1);
    k_finalize_blocks<<<n_touched, 256, 0, s>>>(P, L->v, tv, acc_inv_scale);
  }
  CG_CUDA(cudaGetLastError());
  ctx->touch_clean = true;
  L->num_blocks = blocks_after;  // the next group of the job must see these blocks as existing
  if (stats) {
    stats->blocks_touched += n_touched;
    stats->general_updates += n_general;
  }
  return CG_OK;
}

// Front half of frames [f0, f1) of a job (points -> one ray per bundle, R1 / R2 / R6), queued on
// stream `s` into the set `fb`: nothing here touches the layer.  The counters the back half needs
// (rays, voxel visits, segments, key extent, errors) are copied to fb.h_counters at the end; the
// caller synchronises.  *need_split: the bundle keys do not fit, the caller halves the group.
static int32_t front_enqueue(cg_context* ctx, FrontBufs& fb, cudaStream_t s, int32_t* d_err,
                             const cg_layer* L, const cg_integrator_config* cfg,
                             const IntegratorParams& P, const float* d_points,
                             const uint8_t* d_colors, const uint64_t* offs, size_t f0, size_t f1,
                             int attempt, bool* need_split) {
  *need_split = false;
  const size_t F = f1 - f0;
  const size_t total = offs[f1] - offs[f0];  // points of the group = upper bound on rays
  const size_t upper = total + 1;  // + the sentinel bundle of dropped points
  CG_CUDA(fb.rays.reserve(upper * sizeof(Ray)));
  CG_CUDA(fb.ray_count.reserve(upper * sizeof(unsigned long long)));
  CG_CUDA(fb.ray_offset.reserve(upper * sizeof(unsigned long long)));
  CG_CUDA(fb.scan.reserve(upper * sizeof(uint32_t)));  // bundle heads / valid slots
  const bool merged = cfg->method == CG_METHOD_MERGED;
  if (merged) {
    CG_CUDA(fb.key_a.reserve(total * sizeof(uint64_t)));
    CG_CUDA(fb.key_b.reserve(total * sizeof(uint64_t)));
    CG_CUDA(fb.sorted_pts.reserve(total * sizeof(float4)));
  }
  // bundle key layout of this group: as many bits per voxel axis as fit beside the frame field
  // and the visit rank (at most 13: +-4096 voxels around the sensor)
  int frame_bits = 0;
  while ((size_t(1) << frame_bits) < F) ++frame_bits;
  size_t max_frame_points = 1;
  for (size_t f = f0; f < f1; ++f) max_frame_points = std::max<size_t>(max_frame_points, offs[f + 1] - offs[f]);
  KeyLayout kl;
  kl.rank_bits = std::max(1, ceil_log2(max_frame_points));
  kl.frame_bits = frame_bits;
  if (merged && F > kMaxGroupFrames) {  // per-frame bins of the ray-id partition (shared memory)
    *need_split = true;
    return CG_OK;
  }
  // voxel fields: the box earlier jobs on this context measured (kept as a running union, with
  // some slack around it), or — first job — a cube around the sensor sized for the sensor range
  // with x4 head room for clearing points beyond max_ray.  Fewer bits = fewer radix passes.  A
  // point outside the box flags kErrKeyRange and the group is redone with the measured extent.
  // measuring the extent costs a few hundred thousand atomics: first job, retries, every 64th job
  // (CG_KEY_MEASURE_PERIOD overrides the 64; the tests set it to 1 to reach the shrinking window)
  const unsigned period = static_cast<unsigned>(std::max<size_t>(1, env_size("CG_KEY_MEASURE_PERIOD", 64)));
  const bool measure = !ctx->key_box_valid || attempt > 0 || (ctx->key_jobs++ % period) == period - 1;
  const int avail_total = 63 - frame_bits - kl.rank_bits - 1;
  // attempt 1 follows a point outside a box that was not being measured: the wide cube again
  if (!ctx->key_box_valid || (attempt == 1 && !ctx->key_retry_measured)) {
    const int half = 1 << (std::min(kMaxRelBits, ceil_log2(static_cast<uint64_t>(P.max_ray * P.voxel_size_inv) + 4) + 3) - 1);
    for (int a = 0; a < 3; ++a) {
      kl.lo[a] = -half;
      kl.bits[a] = ceil_log2(2 * static_cast<uint64_t>(half));
    }
  } else {
    for (int a = 0; a < 3; ++a) {
      kl.lo[a] = std::max(-kKeyLimit, ctx->key_lo[a] - kKeySlack);
      const int hi = std::min(kKeyLimit, ctx->key_hi[a] + kKeySlack);
      kl.bits[a] = std::max(1, ceil_log2(static_cast<uint64_t>(hi - kl.lo[a]) + 1));
    }
  }
  if (merged && kl.bits[0] + kl.bits[1] + kl.bits[2] > avail_total) {
    if (F > 1) {  // fewer frames per group leave more bits for the voxel fields
      *need_split = true;
      return CG_OK;
    }
    set_error("a single frame of %zu points is too large; split the point cloud", total);
    return CG_ERR_INVALID_ARG;
  }
  // sorted bits: (clearing, voxel); the frame and rank fields below stay in input order
  const int bundle_begin_bit = kl.voxel_shift(), bundle_end_bit = kl.clear_bit() + 1;
  cub::DoubleBuffer<uint64_t> dk(fb.key_a.as<uint64_t>(), fb.key_b.as<uint64_t>());
  thrust::counting_iterator<uint32_t> iota(0);
  uint32_t* d_num = fb.d_select_count;
  // the job's poses and frame offsets were uploaded once by integrate_job
  const float* pts = d_points + 3 * offs[f0];
  const uint32_t* cols = reinterpret_cast<const uint32_t*>(d_colors) + offs[f0];
  const FrameTable ft{fb.frame_base.as<uint64_t>() + f0, offs[f0] - offs[0], static_cast<int>(F)};
  fb.group_poses = fb.poses.as<float>() + 7 * f0;
  fb.group_frames = static_cast<int>(F);
  ValidSlot valid{P, ft, pts};
  size_t tmp_sort = 0, tmp_sel = 0;
  if (merged) {
    cub::DeviceRadixSort::SortKeys(nullptr, tmp_sort, dk, static_cast<int>(total),
                                   bundle_begin_bit, bundle_end_bit, s);
    cub::DeviceSelect::If(nullptr, tmp_sel, iota, fb.scan.as<uint32_t>(), d_num,
                          static_cast<int>(total), BundleHead{nullptr, 0}, s);
  } else {
    cub::DeviceSelect::If(nullptr, tmp_sel, iota, fb.scan.as<uint32_t>(), d_num,
                          static_cast<int>(total), valid, s);
  }
  CG_CUDA(fb.cub_tmp.reserve(std::max(tmp_sort, tmp_sel)));
  if (merged) {
    {
      StageScope sc(ctx, kStagePointKeys, 1, s);
      k_point_keys<<<grid_for(total, 256), 256, 0, s>>>(P, kl, fb.group_poses, ft, pts, total,
                                                        fb.key_a.as<uint64_t>(), d_err,
                                                        measure ? fb.d_key_bounds : nullptr,
                                                        fb.d_counters);
    }
    {
      StageScope sc(ctx, kStageBundleSort, 0, s);
      CG_CUDA(cub::DeviceRadixSort::SortKeys(fb.cub_tmp.p, tmp_sort, dk, static_cast<int>(total),
                                             bundle_begin_bit, bundle_end_bit, s));
    }
    // the gather only needs the sorted keys: it runs beside the bundle heads and their ordering
    const bool forked = side_stream(fb, s);
    const cudaStream_t gs = forked ? fb.side : s;
    if (forked) {
      CG_CUDA(cudaEventRecord(fb.ev_fork, s));
      CG_CUDA(cudaStreamWaitEvent(fb.side, fb.ev_fork, 0));
    }
    {
      StageScope sc(ctx, kStageGather, 1, gs);
      k_gather_sorted<<<grid_for(total, 256), 256, 0, gs>>>(
          kl, P.order_mode, dk.Current(), static_cast<uint32_t>(total), ft, pts, cols,
          fb.sorted_pts.as<float4>());
    }
    if (forked) CG_CUDA(cudaEventRecord(fb.ev_join, fb.side));
    {
      StageScope sc(ctx, kStageBundleScan, 0, s);
      CG_CUDA(cub::DeviceSelect::If(fb.cub_tmp.p, tmp_sel, iota, fb.scan.as<uint32_t>(), d_num,
                                    static_cast<int>(total), BundleHead{dk.Current(), kl.rank_bits}, s));
    }
    // upper bound on the number of bundles: one per point + the sentinel
    const unsigned bgrid = std::min<unsigned>(grid_for(upper, 256), ctx->num_sms * 8u);
    // chunks of the ray-id partition (contiguous bundles per CTA)
    const unsigned cgrid = std::min<unsigned>(grid_for(upper, 256), ctx->num_sms * 2u);
    const size_t frame_smem = (F + 1) * sizeof(uint32_t);
    CG_CUDA(fb.frame_count.reserve((F + 1) * cgrid * sizeof(uint32_t)));
    CG_CUDA(fb.ray_id.reserve(upper * sizeof(uint32_t)));
    {
      StageScope sc(ctx, kStageBundleOrder, 4, s);
      CG_CUDA(fill_bytes(fb.d_class_count, 0, 128 * sizeof(uint32_t), s));  // + the fold queue
      k_bundle_histogram<<<cgrid, 256, frame_smem, s>>>(
          kl, dk.Current(), static_cast<uint32_t>(total), fb.scan.as<uint32_t>(), d_num,
          fb.d_class_count, fb.frame_count.as<uint32_t>(), static_cast<int>(F));
      k_frame_scan<<<1, 1024, 0, s>>>(fb.frame_count.as<uint32_t>(),
                                      static_cast<uint32_t>((F + 1) * cgrid));
      k_bundle_order<<<cgrid, 256, frame_smem, s>>>(
          kl, dk.Current(), static_cast<uint32_t>(total), fb.scan.as<uint32_t>(), d_num,
          fb.d_class_count, fb.frame_count.as<uint32_t>(), static_cast<int>(F),
          fb.ray_offset.as<uint32_t>(), fb.ray_id.as<uint32_t>(), fb.rays.as<Ray>());
    }
    if (forked) CG_CUDA(cudaStreamWaitEvent(s, fb.ev_join, 0));
    {
      // 4 CTAs per SM for the long bundles: measured 0.126 / 0.100 / 0.104 / 0.106 ms for
      // 2 / 4 / 8 / 12 with the long bundles alone
      StageScope sc(ctx, kStageFoldWide, 1, s);
      static const unsigned wide_per_sm = static_cast<unsigned>(env_size("CG_FOLD_WIDE_CTAS", 4));
      static const unsigned short_per_sm = static_cast<unsigned>(env_size("CG_FOLD_SHORT_CTAS", 4));
      const unsigned wide_ctas = ctx->num_sms * wide_per_sm;
      k_fold<<<wide_ctas + ctx->num_sms * short_per_sm, 128, 0, s>>>(
          P, kl, dk.Current(), static_cast<uint32_t>(total), fb.scan.as<uint32_t>(), d_num,
          fb.sorted_pts.as<float4>(), fb.d_class_count, fb.ray_offset.as<uint32_t>(),
          fb.ray_id.as<uint32_t>(), fb.d_class_count + 2 * kSizeClasses, fb.rays.as<Ray>(),
          wide_ctas);
    }
    {
      StageScope sc(ctx, kStageBundleRays, 1, s);
      k_bundle_rays<<<bgrid, 256, 0, s>>>(P, fb.group_poses, d_num, fb.rays.as<Ray>(),
                                          fb.ray_count.as<unsigned long long>());
    }
    if (P.anti_grazing) {  // set of the scan's bundle voxels (at most one per point)
      size_t gcap = 1024;
      while (gcap < 2 * total) gcap <<= 1;
      CG_CUDA(fb.grazing_keys.reserve(gcap * sizeof(unsigned long long)));
      CG_CUDA(fb.grazing_ray_key.reserve(upper * sizeof(unsigned long long)));
      fb.grazing_mask = static_cast<uint32_t>(gcap - 1);
      CG_CUDA(fill_bytes(fb.grazing_keys.p, 0xFF, gcap * sizeof(unsigned long long), s));
      k_grazing_build<<<bgrid, 256, 0, s>>>(kl, dk.Current(), static_cast<uint32_t>(total),
                                            fb.scan.as<uint32_t>(), d_num, fb.ray_id.as<uint32_t>(),
                                            fb.grazing_keys.as<unsigned long long>(),
                                            fb.grazing_mask,
                                            fb.grazing_ray_key.as<unsigned long long>());
    }
  } else {
    {
      StageScope sc(ctx, kStageBundleScan, 0, s);
      CG_CUDA(cub::DeviceSelect::If(fb.cub_tmp.p, tmp_sel, iota, fb.scan.as<uint32_t>(), d_num,
                                    static_cast<int>(total), valid, s));
    }
    StageScope sc(ctx, kStageBundleRays, 1, s);
    k_simple_rays<<<grid_for(total, 256), 256, 0, s>>>(
        P, fb.group_poses, ft, fb.scan.as<uint32_t>(), d_num, pts,
        cols, fb.rays.as<Ray>(), fb.ray_count.as<unsigned long long>());
  }
  {
    StageScope sc(ctx, kStageRayScan, 3, s);
    const int sgrid = std::min(1024, ctx->num_sms * 4);
    CG_CUDA(fb.scan_partials.reserve(1024 * sizeof(unsigned long long)));
    k_scan_partials<<<sgrid, kScanThreads, 0, s>>>(d_num, fb.ray_count.as<unsigned long long>(),
                                                   fb.scan_partials.as<unsigned long long>());
    k_scan_totals<<<1, 1024, 0, s>>>(d_num, fb.scan_partials.as<unsigned long long>(), sgrid,
                                     fb.d_counters, d_err, fb.d_key_bounds);
    k_scan_apply<<<sgrid, kScanThreads, 0, s>>>(d_num, fb.ray_count.as<unsigned long long>(),
                                                fb.scan_partials.as<unsigned long long>(),
                                                fb.ray_offset.as<unsigned long long>());
  }
  CG_CUDA(cudaMemcpyAsync(fb.h_counters, fb.d_counters, sizeof(CallCounters),
                          cudaMemcpyDeviceToHost, s));
  CG_CUDA(cudaGetLastError());
  return CG_OK;
}

enum FrontVerdict { kFrontOk, kFrontRetry, kFrontSplit, kFrontFail };

// After the host has synchronised on a front half: book-keeping of the bundle-key box from the
// extent the job measured, and what has to happen next.
static FrontVerdict front_digest(cg_context* ctx, const FrontBufs& fb, bool merged, size_t F,
                                 int attempt, int32_t* rc) {
  const size_t num_pairs = fb.h_counters->pairs;
  const size_t max_pairs = env_size("CG_MAX_PAIRS", size_t(768) << 20);
  const bool key_range = (fb.h_counters->err & kErrKeyRange) != 0;
  // The box = union of the extents measured by the jobs of this context (relative voxel indices
  // of every valid point).  A second union over a window of 8 jobs replaces it when it needs
  // fewer bits, so that one outlier (a stray far return) does not widen the keys for good.
  if (merged && fb.h_counters->key_lo[0] <= fb.h_counters->key_hi[0]) {
    int lo[3], hi[3];
    for (int a = 0; a < 3; ++a) {
      lo[a] = std::max(-kKeyLimit, fb.h_counters->key_lo[a]);
      hi[a] = std::min(kKeyLimit, fb.h_counters->key_hi[a]);
      ctx->key_lo[a] = ctx->key_box_valid ? std::min(ctx->key_lo[a], lo[a]) : lo[a];
      ctx->key_hi[a] = ctx->key_box_valid ? std::max(ctx->key_hi[a], hi[a]) : hi[a];
      ctx->key_win_lo[a] = ctx->key_win_jobs ? std::min(ctx->key_win_lo[a], lo[a]) : lo[a];
      ctx->key_win_hi[a] = ctx->key_win_jobs ? std::max(ctx->key_win_hi[a], hi[a]) : hi[a];
    }
    ctx->key_box_valid = true;
    if (++ctx->key_win_jobs == 8) {
      int box_bits = 0, win_bits = 0;
      for (int a = 0; a < 3; ++a) {
        box_bits += ceil_log2(static_cast<uint64_t>(ctx->key_hi[a] - ctx->key_lo[a] + 2 * kKeySlack) + 1);
        win_bits += ceil_log2(static_cast<uint64_t>(ctx->key_win_hi[a] - ctx->key_win_lo[a] + 2 * kKeySlack) + 1);
      }
      if (win_bits < box_bits)
        for (int a = 0; a < 3; ++a) {
          ctx->key_lo[a] = ctx->key_win_lo[a];
          ctx->key_hi[a] = ctx->key_win_hi[a];
        }
      ctx->key_win_jobs = 0;
    }
  }
  if (key_range) {
    const bool measured = fb.h_counters->key_lo[0] <= fb.h_counters->key_hi[0];
    bool reachable = attempt < 3;
    for (int a = 0; a < 3 && measured; ++a)
      reachable = reachable && fb.h_counters->key_lo[a] >= -kKeyLimit &&
                  fb.h_counters->key_hi[a] <= kKeyLimit;
    // redo the group: with the extent just measured the box covers its points; if this pass did
    // not measure, the next one does (and may have to be redone once more)
    if (reachable) {
      if (getenv("CG_TRACE_KEYS"))
        fprintf(stderr, "[cg] bundle-key box exceeded (attempt %d, measured %d): box x[%d,%d] y[%d,%d] z[%d,%d]\n",
                attempt, int(measured), ctx->key_lo[0], ctx->key_hi[0], ctx->key_lo[1], ctx->key_hi[1],
                ctx->key_lo[2], ctx->key_hi[2]);
      ctx->key_retry_measured = measured;
      return kFrontRetry;
    }
    if (F == 1) {
      set_error("a point lies more than %d voxels from the sensor", kKeyLimit);
      *rc = CG_ERR_OUT_OF_RANGE;
      return kFrontFail;
    }
  }
  if (key_range || num_pairs > max_pairs || num_pairs >= 0x7FFFFFF0ull) {
    if (F > 1) return kFrontSplit;  // the front half never touches the layer: safe to redo in two halves
    if (num_pairs >= 0x7FFFFFF0ull) {
      set_error("a single frame produces %zu voxel updates; split the point cloud", num_pairs);
      *rc = CG_ERR_INVALID_ARG;
      return kFrontFail;
    }
  }
  return kFrontOk;
}

// frames [f0, f1) of the job as one group; splits itself when the pair list would not fit
static int32_t integrate_group(cg_layer* L, const cg_integrator_config* cfg,
                               const IntegratorParams& P, const float* h_poses,
                               const float* d_points, const uint8_t* d_colors,
                               const uint64_t* offs, size_t f0, size_t f1,
                               cg_integrate_stats* stats, int attempt = 0) {
  cg_context* ctx = L->ctx;
  cudaStream_t s = ctx->stream;
  const size_t F = f1 - f0;
  const size_t total = offs[f1] - offs[f0];  // points of the group = upper bound on rays
  if (total == 0) return CG_OK;
  if (total > 0x7FFFFFF0ull || F > (1u << 20)) {
    set_error("too many points / frames in one group");
    return CG_ERR_INVALID_ARG;
  }
  auto halves = [&]() -> int32_t {
    const size_t mid = f0 + F / 2;
    int32_t rc = integrate_group(L, cfg, P, h_poses, d_points, d_colors, offs, f0, mid, stats);
    if (rc) return rc;
    return integrate_group(L, cfg, P, h_poses, d_points, d_colors, offs, mid, f1, stats);
  };
  bool need_split = false;
  int32_t rc = front_enqueue(ctx, *ctx, s, L->v.err, L, cfg, P, d_points, d_colors, offs, f0, f1,
                             attempt, &need_split);
  if (rc) return rc;
  if (need_split) return halves();
  CG_CUDA(cudaStreamSynchronize(s));
  CG_CUDA(cudaGetLastError());
  switch (front_digest(ctx, *ctx, cfg->method == CG_METHOD_MERGED, F, attempt, &rc)) {
    case kFrontRetry:
      return integrate_group(L, cfg, P, h_poses, d_points, d_colors, offs, f0, f1, stats, attempt + 1);
    case kFrontSplit:
      return halves();
    case kFrontFail:
      return rc;
    case kFrontOk:
      break;
  }
  const uint32_t num_rays = static_cast<uint32_t>(ctx->h_counters->rays);
  const size_t num_pairs = ctx->h_counters->pairs;
  if (stats) stats->points_beyond_reach += ctx->h_counters->far_dropped;
  if (num_rays == 0 || num_pairs == 0) return CG_OK;
  if (stats) {
    stats->rays += num_rays;
    stats->voxel_updates += num_pairs;
  }
  return run_back_half(ctx, *ctx, L, P, num_rays, num_pairs, ctx->h_counters->segments, stats);
}

// The job's poses and frame offsets (relative to its first point) go up once per job, through a
// pinned, device-mapped host buffer and a copy KERNEL: an H2D memcpy would be queued on the copy
// engine behind the point data that the staging / pipelined paths have in flight.
static int32_t upload_frame_tables(FrontBufs& fb, size_t F, const float* h_poses,
                                   const uint64_t* offs, cudaStream_t stream) {
  const size_t pose_words = F * 7, off_words = (F + 1) * 2;
  const size_t bytes = (pose_words + off_words) * sizeof(uint32_t);
  if (bytes > fb.h_tables_cap) {
    if (fb.h_tables) cudaFreeHost(fb.h_tables);
    fb.h_tables = nullptr;
    fb.h_tables_cap = 0;
    CG_CUDA(cudaHostAlloc(&fb.h_tables, bytes * 2, cudaHostAllocMapped));
    fb.h_tables_cap = bytes * 2;
  }
  CG_CUDA(fb.poses.reserve(pose_words * sizeof(float)));
  CG_CUDA(fb.frame_base.reserve((F + 1) * sizeof(uint64_t)));
  uint32_t* h = static_cast<uint32_t*>(fb.h_tables);
  memcpy(h, h_poses, pose_words * sizeof(float));
  uint64_t* ho = reinterpret_cast<uint64_t*>(h + pose_words + (pose_words & 1));
  for (size_t f = 0; f <= F; ++f) ho[f] = offs[f] - offs[0];
  void* d_alias = nullptr;
  CG_CUDA(cudaHostGetDevicePointer(&d_alias, fb.h_tables, 0));
  const uint32_t* src = static_cast<const uint32_t*>(d_alias);
  k_copy_words<<<grid_for(pose_words, 256), 256, 0, stream>>>(fb.poses.as<uint32_t>(), src,
                                                              pose_words);
  k_copy_words<<<grid_for(off_words, 256), 256, 0, stream>>>(
      fb.frame_base.as<uint32_t>(), src + pose_words + (pose_words & 1), off_words);
  CG_CUDA(cudaGetLastError());
  return CG_OK;
}

static int32_t integrate_job(cg_layer* L, const cg_integrator_config* cfg, size_t F,
                             const float* h_poses, const float* d_points, const uint8_t* d_colors,
                             const uint64_t* offs, int freespace, cg_integrate_stats* stats) {
  if (cfg->method == CG_METHOD_FAST) {
    set_error("method FAST is order- and wall-clock-dependent in the reference and has no "
              "deterministic device form; use MERGED or SIMPLE");
    return CG_ERR_UNSUPPORTED;
  }
  if (cfg->method != CG_METHOD_MERGED && cfg->method != CG_METHOD_SIMPLE) return CG_ERR_INVALID_ARG;
  if (!(cfg->default_truncation_distance > 0.0f) || !(cfg->max_ray_length_m > 0.0f)) {
    set_error("invalid integrator config");
    return CG_ERR_INVALID_ARG;
  }
  CG_CUDA(cudaSetDevice(L->ctx->device));
  const IntegratorParams P = make_params(L, cfg, freespace);
  const int64_t blocks_before = L->num_blocks;
  if (stats) {
    memset(stats, 0, sizeof(*stats));
    stats->points_in = offs[F] - offs[0];
  }
  const size_t max_group_points = env_size("CG_MAX_GROUP_POINTS", size_t(48) << 20);
  // poses and frame offsets (relative to the job's first point) go up once per job
  int32_t rc = upload_frame_tables(*L->ctx, F, h_poses, offs, L->ctx->stream);
  if (rc) return rc;
  size_t f0 = 0;
  while (f0 < F && rc == CG_OK) {
    size_t f1 = f0 + 1;
    while (f1 < F && offs[f1 + 1] - offs[f0] <= max_group_points) ++f1;
    rc = integrate_group(L, cfg, P, h_poses, d_points, d_colors, offs, f0, f1, stats);
    f0 = f1;
  }
  const int32_t rc2 = finish_call(L, nullptr);
  if (stats) stats->blocks_allocated = L->num_blocks - blocks_before;
  return rc ? rc : rc2;
}

static int32_t stage_inputs(cg_context* ctx, const float* pts, const uint8_t* cols, size_t n) {
  CG_CUDA(cudaSetDevice(ctx->device));
  CG_CUDA(ctx->points.reserve(n * 3 * sizeof(float)));
  CG_CUDA(ctx->colors.reserve(n * 4));
  StageScope sc(ctx, kStageTransfer, 0);
  // pageable inputs (std::vector clouds of the drop-in call) go through worker threads and a
  // pinned bounce buffer (host_stage.cu); CG_STAGE_THREADS=0 restores the plain copies
  static const int threads = static_cast<int>(env_size("CG_STAGE_THREADS", 3));
  CG_CUDA(stage_begin(ctx->stager, ctx->stream));
  CG_CUDA(stage_to_device(&ctx->stager, ctx->points.p, pts, n * 3 * sizeof(float), ctx->stream,
                          threads));
  CG_CUDA(stage_to_device(&ctx->stager, ctx->colors.p, cols, n * 4, ctx->stream, threads));
  return CG_OK;
}


// ---- pipelined jobs: the front half of a later job beside the back half of the current one
static int32_t prepare_job(cg_layer* L, const cg_integrator_config* cfg, size_t F,
                           const float* poses, const float* d_pts, const uint8_t* d_cols,
                           const uint64_t* offs, int32_t freespace, int32_t slot,
                           cudaEvent_t inputs_ready) {
  if (!L || !cfg || !poses || !offs || slot < 0 || slot > 1) {
    set_error("cg_prepare_batch: invalid argument");
    return CG_ERR_INVALID_ARG;
  }
  for (size_t f = 0; f < F; ++f)
    if (offs[f + 1] < offs[f]) {
      set_error("frame_offsets must be non-decreasing");
      return CG_ERR_INVALID_ARG;
    }
  cg_context* ctx = L->ctx;
  CG_CUDA(cudaSetDevice(ctx->device));
  FrontBufs& fb = ctx->prep[slot];
  if (!ctx->prep_stream) CG_CUDA(cudaStreamCreateWithFlags(&ctx->prep_stream, cudaStreamNonBlocking));
  if (!ctx->prep_done[slot]) {
    CG_CUDA(cudaEventCreateWithFlags(&ctx->prep_done[slot], cudaEventDisableTiming));
    CG_CUDA(init_front_words(fb));
  }
  cg_context::PreparedJob& pj = ctx->prepared[slot];
  pj.valid = true;
  pj.front_queued = false;
  pj.cfg = *cfg;
  pj.poses.assign(poses, poses + 7 * F);
  pj.offs.resize(F + 1);
  for (size_t f = 0; f <= F; ++f) pj.offs[f] = offs[f] - offs[0];
  pj.d_points = d_pts ? d_pts + 3 * offs[0] : nullptr;
  pj.d_colors = d_cols ? d_cols + 4 * offs[0] : nullptr;
  pj.freespace = freespace;
  pj.voxel_size = L->v.voxel_size;
  const size_t total = pj.offs[F];
  const size_t max_group_points = env_size("CG_MAX_GROUP_POINTS", size_t(48) << 20);
  // the fast path: a valid merged / simple job that is one group; everything else is left to the
  // plain path inside cg_integrate_prepared (which also reports the errors)
  if ((cfg->method != CG_METHOD_MERGED && cfg->method != CG_METHOD_SIMPLE) ||
      !(cfg->default_truncation_distance > 0.0f) || !(cfg->max_ray_length_m > 0.0f) || total == 0 ||
      total > max_group_points || total > 0x7FFFFFF0ull || F > (1u << 20) || !d_pts || !d_cols)
    return CG_OK;
  const IntegratorParams P = make_params(L, cfg, freespace);
  cudaStream_t ps = ctx->prep_stream;
  // the inputs were produced on the context's stream (or by the staged copy): order behind them
  if (!ctx->wait_event) CG_CUDA(cudaEventCreateWithFlags(&ctx->wait_event, cudaEventDisableTiming));
  CG_CUDA(cudaEventRecord(ctx->wait_event, ctx->stream));
  CG_CUDA(cudaStreamWaitEvent(ps, ctx->wait_event, 0));
  if (inputs_ready) CG_CUDA(cudaStreamWaitEvent(ps, inputs_ready, 0));
  CG_CUDA(fill_bytes(fb.d_front_err, 0, sizeof(int32_t), ps));
  int32_t rc = upload_frame_tables(fb, F, pj.poses.data(), pj.offs.data(), ps);
  if (rc) return rc;
  bool need_split = false;
  rc = front_enqueue(ctx, fb, ps, fb.d_front_err, L, cfg, P, pj.d_points, pj.d_colors,
                     pj.offs.data(), 0, F, 0, &need_split);
  if (rc) return rc;
  if (need_split) {  // does not fit one group: drain and leave the job to the plain path
    CG_CUDA(cudaStreamSynchronize(ps));
    return CG_OK;
  }
  CG_CUDA(cudaEventRecord(ctx->prep_done[slot], ps));
  pj.front_queued = true;
  return CG_OK;
}

}  // namespace cg

using namespace cg;

extern "C" {

int32_t cg_prepare_batch_device(cg_layer* L, const cg_integrator_config* cfg, size_t F,
                                const float* poses, const float* d_pts, const uint8_t* d_cols,
                                const uint64_t* offs, int32_t freespace, int32_t slot) {
  return prepare_job(L, cfg, F, poses, d_pts, d_cols, offs, freespace, slot, nullptr);
}

int32_t cg_prepare_batch_staged(cg_layer* L, const cg_integrator_config* cfg, size_t F,
                                const float* poses, int32_t stage_slot, const uint64_t* offs,
                                int32_t freespace, int32_t slot) {
  if (!L || stage_slot < 0 || stage_slot > 1 || !offs || !L->ctx->stage_ready[stage_slot]) {
    set_error("cg_prepare_batch_staged: invalid argument (nothing staged in this slot?)");
    return CG_ERR_INVALID_ARG;
  }
  cg_context* ctx = L->ctx;
  if (offs[0] != 0 || offs[F] != ctx->stage_points[stage_slot]) {
    set_error("cg_prepare_batch_staged: frame_offsets must cover exactly the %zu staged points",
              ctx->stage_points[stage_slot]);
    return CG_ERR_INVALID_ARG;
  }
  return prepare_job(L, cfg, F, poses, ctx->stage_pts[stage_slot].as<float>(),
                     ctx->stage_cols[stage_slot].as<uint8_t>(), offs, freespace, slot,
                     ctx->stage_ready[stage_slot]);
}

int32_t cg_integrate_prepared(cg_layer* L, int32_t slot, cg_integrate_stats* stats) {
  if (!L || slot < 0 || slot > 1 || !L->ctx->prepared[slot].valid) {
    set_error("cg_integrate_prepared: nothing prepared in this slot");
    return CG_ERR_INVALID_ARG;
  }
  cg_context* ctx = L->ctx;
  CG_CUDA(cudaSetDevice(ctx->device));
  cg_context::PreparedJob& pj = ctx->prepared[slot];
  pj.valid = false;
  const size_t F = pj.offs.size() - 1;
  if (pj.front_queued && pj.voxel_size == L->v.voxel_size) {
    FrontBufs& fb = ctx->prep[slot];
    CG_CUDA(cudaEventSynchronize(ctx->prep_done[slot]));
    int32_t rc = CG_OK;
    const FrontVerdict v = front_digest(ctx, fb, pj.cfg.method == CG_METHOD_MERGED, F, 3, &rc);
    if (v == kFrontOk && !(fb.h_counters->err & kErrOutOfRange)) {
      const IntegratorParams P = make_params(L, &pj.cfg, pj.freespace);
      const int64_t blocks_before = L->num_blocks;
      if (stats) {
        memset(stats, 0, sizeof(*stats));
        stats->points_in = pj.offs[F];
        stats->points_beyond_reach = fb.h_counters->far_dropped;
      }
      const uint32_t num_rays = static_cast<uint32_t>(fb.h_counters->rays);
      const size_t num_pairs = fb.h_counters->pairs;
      if (num_rays > 0 && num_pairs > 0) {
        if (stats) {
          stats->rays = num_rays;
          stats->voxel_updates = num_pairs;
        }
        rc = run_back_half(ctx, fb, L, P, num_rays, num_pairs, fb.h_counters->segments, stats);
      }
      const int32_t rc2 = finish_call(L, nullptr);
      if (stats) stats->blocks_allocated = L->num_blocks - blocks_before;
      return rc ? rc : rc2;
    }
    // a point outside the key box, too many voxel visits for one group, ...: the plain path
    // handles it (regrouping, retries, the error report); the prepared front half is dropped
  }
  return cg_integrate_batch_device(L, &pj.cfg, F, pj.poses.data(), pj.d_points, pj.d_colors,
                                   pj.offs.data(), pj.freespace, stats);
}

void cg_integrator_config_default(cg_integrator_config* c) {
  if (!c) return;
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
  c->method = CG_METHOD_MERGED;
  c->integration_order_mode = CG_ORDER_MIXED;
  c->start_voxel_subsampling_factor = 2.0f;
  c->max_consecutive_ray_collisions = 2;
}

int32_t cg_integrate_batch_device(cg_layer* L, const cg_integrator_config* cfg, size_t F,
                                  const float* poses, const float* d_pts, const uint8_t* d_cols,
                                  const uint64_t* offs, int32_t freespace,
                                  cg_integrate_stats* stats) {
  if (!L || !cfg || !poses || !offs || (offs[F] > offs[0] && (!d_pts || !d_cols))) {
    set_error("cg_integrate: null argument");
    return CG_ERR_INVALID_ARG;
  }
  for (size_t f = 0; f < F; ++f)
    if (offs[f + 1] < offs[f]) {
      set_error("frame_offsets must be non-decreasing");
      return CG_ERR_INVALID_ARG;
    }
  return integrate_job(L, cfg, F, poses, d_pts, d_cols, offs, freespace, stats);
}

int32_t cg_integrate_batch(cg_layer* L, const cg_integrator_config* cfg, size_t F,
                           const float* poses, const float* pts, const uint8_t* cols,
                           const uint64_t* offs, int32_t freespace, cg_integrate_stats* stats) {
  if (!L || !cfg || !poses || !offs) {
    set_error("cg_integrate: null argument");
    return CG_ERR_INVALID_ARG;
  }
  const size_t first = offs[0], total = offs[F] - offs[0];
  if (total && (!pts || !cols)) {
    set_error("cg_integrate: null argument");
    return CG_ERR_INVALID_ARG;
  }
  std::vector<uint64_t> rel(F + 1);
  for (size_t f = 0; f <= F; ++f) rel[f] = offs[f] - first;
  cg_context* ctx = L->ctx;
  int32_t rc = stage_inputs(ctx, pts + 3 * first, cols + 4 * first, total);
  if (rc) return rc;
  return cg_integrate_batch_device(L, cfg, F, poses, ctx->points.as<float>(),
                                   ctx->colors.as<uint8_t>(), rel.data(), freespace, stats);
}

int32_t cg_stage_batch_async(cg_context* ctx, int32_t slot, const float* pts, const uint8_t* cols,
                             size_t n) {
  if (!ctx || slot < 0 || slot > 1 || (n && (!pts || !cols))) {
    set_error("cg_stage_batch_async: invalid argument");
    return CG_ERR_INVALID_ARG;
  }
  CG_CUDA(cudaSetDevice(ctx->device));
  if (!ctx->copy_stream)
    CG_CUDA(cudaStreamCreateWithFlags(&ctx->copy_stream, cudaStreamNonBlocking));
  if (!ctx->stage_ready[slot])
    CG_CUDA(cudaEventCreateWithFlags(&ctx->stage_ready[slot], cudaEventDisableTiming));
  CG_CUDA(ctx->stage_pts[slot].reserve(n * 3 * sizeof(float)));
  CG_CUDA(ctx->stage_cols[slot].reserve(n * 4));
  if (n) {
    CG_CUDA(cudaMemcpyAsync(ctx->stage_pts[slot].p, pts, n * 3 * sizeof(float),
                            cudaMemcpyHostToDevice, ctx->copy_stream));
    CG_CUDA(cudaMemcpyAsync(ctx->stage_cols[slot].p, cols, n * 4, cudaMemcpyHostToDevice,
                            ctx->copy_stream));
  }
  CG_CUDA(cudaEventRecord(ctx->stage_ready[slot], ctx->copy_stream));
  ctx->stage_points[slot] = n;
  return CG_OK;
}

int32_t cg_integrate_batch_staged(cg_layer* L, const cg_integrator_config* cfg, size_t F,
                                  const float* poses, int32_t slot, const uint64_t* offs,
                                  int32_t freespace, cg_integrate_stats* stats) {
  if (!L || !cfg || !poses || !offs || slot < 0 || slot > 1 || !L->ctx->stage_ready[slot]) {
    set_error("cg_integrate_batch_staged: invalid argument (nothing staged in this slot?)");
    return CG_ERR_INVALID_ARG;
  }
  cg_context* ctx = L->ctx;
  if (offs[0] != 0 || offs[F] != ctx->stage_points[slot]) {
    set_error("cg_integrate_batch_staged: frame_offsets must cover exactly the %zu staged points",
              ctx->stage_points[slot]);
    return CG_ERR_INVALID_ARG;
  }
  CG_CUDA(cudaStreamWaitEvent(ctx->stream, ctx->stage_ready[slot], 0));
  return cg_integrate_batch_device(L, cfg, F, poses, ctx->stage_pts[slot].as<float>(),
                                   ctx->stage_cols[slot].as<uint8_t>(), offs, freespace, stats);
}

int32_t cg_integrate_pointcloud_device(cg_layer* L, const cg_integrator_config* cfg,
                                       const float T[7], const float* d_pts, const uint8_t* d_cols,
                                       size_t n, int32_t freespace, cg_integrate_stats* stats) {
  const uint64_t offs[2] = {0, n};
  return cg_integrate_batch_device(L, cfg, 1, T, d_pts, d_cols, offs, freespace, stats);
}

int32_t cg_integrate_pointcloud(cg_layer* L, const cg_integrator_config* cfg, const float T[7],
                                const float* pts, const uint8_t* cols, size_t n, int32_t freespace,
                                cg_integrate_stats* stats) {
  const uint64_t offs[2] = {0, n};
  return cg_integrate_batch(L, cfg, 1, T, pts, cols, offs, freespace, stats);
}

}  // extern "C"
