// integrate_front.cu — front half of the TSDF integration: points to one ray per bundle (R1, R2,
// R6).  Nothing here touches the layer, so the front half of a later job can run beside the back
// half (integrate_back.cu) of the current one.
//   k_point_keys        validity, T_G_C * p, bundle key [frame | clearing | voxel of p_G relative
//                       to the sensor voxel | visit rank]
//   radix sort (keys)   on the bits above the rank: bundles in canonical order, their points in the
//                       order the reference visits them
//   select              bundle heads
//   k_gather_sorted     the sorted points next to each other
//   k_bundle_histogram / k_frame_scan / k_bundle_order   bundles by size class, longest first,
//                       and their ray ids
//   k_fold              the reference's *sequential* weighted mean and colour blend per bundle
//                       (bit-exact: the merged point decides which voxels and blocks the ray
//                       visits), long bundles and short ones in two parts of one launch -> one ray
//                       per bundle
//   k_grazing_build     (anti-grazing only) set of the scan's bundle voxels
//   k_bundle_rays       T_G_C * merged point, closed-form visit / block counts; k_scan_* offsets
// SIMPLE skips the bundles: k_simple_rays makes one ray per valid point.
#include <cub/cub.cuh>
#include <thrust/iterator/counting_iterator.h>
#include <string.h>

#include <algorithm>

#include "integrate.cuh"

namespace cg {

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
// entries are read), base = offs[0]; slots and point indices are relative to the group.  counts
// (depth jobs, else null): the group's entries of the job's kept-count table; frame f's points
// are then the first counts[f] of its slots, the others are holes.
struct FrameTable {
  const uint64_t* offs;
  uint64_t base;
  int F;
  const uint32_t* counts;
  __device__ __forceinline__ uint64_t start(int f) const { return offs[f] - base; }
  __device__ __forceinline__ int count(int f) const {
    return counts ? static_cast<int>(counts[f]) : static_cast<int>(start(f + 1) - start(f));
  }
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
    const int n = ft.count(f);
    const int i = static_cast<int>(g - base);
    // (a hole, i >= n, keeps its slot: visit_rank(i) = i there)
    const uint32_t k = static_cast<uint32_t>(visit_rank(i, n, P.order_mode));
    const V3 pc = i < n ? load_point(pts, g) : V3{0.0f, 0.0f, 0.0f};
    bool clearing = false;
    uint64_t key = kInvalidPointKey;
    if (i < n && point_valid(P, pc, &clearing)) {
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
  const int n = ft.count(f);
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
//   k_fold              bundles of 64 points or more 8 lanes each (fold_wide); the shorter ones one
//                       lane each, 32 consecutive bundles of the order per warp, every lane
//                       streaming its own run of `sorted` with a 4-deep register prefetch
//                       (fold_short).
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
    const int n = ft.count(f);
    if (static_cast<int>(g - base) >= n) return false;  // a hole of a depth job's slab
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
  const int n = ft.count(f);
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
// CTA 0 also sums a depth job's kept points of the group (kept_counts[0, F)) into
// c->points_kept (0 for a cloud job, whose count the host knows).  Merged depth jobs: when every
// dropped key of the group is a hole of a slab (the sentinel bundle starts at slot `kept`), the
// cloud of the same images has no dropped point and no sentinel ray; c->hole_sentinel = 1 tells
// the host to leave that ray out of the stats.
__global__ void __launch_bounds__(kScanThreads)
k_scan_partials(const uint32_t* __restrict__ num_rays, const unsigned long long* __restrict__ in,
                unsigned long long* __restrict__ partials, const uint32_t* __restrict__ kept_counts,
                int F, const uint64_t* __restrict__ sorted_keys, const uint32_t* __restrict__ heads,
                CallCounters* c) {
  typedef cub::BlockReduce<unsigned long long, kScanThreads> Reduce;
  __shared__ typename Reduce::TempStorage tmp;
  uint32_t lo, hi;
  scan_range(*num_rays, lo, hi);
  unsigned long long sum = 0;
  for (uint32_t i = lo + threadIdx.x; i < hi; i += kScanThreads) sum += in[i];
  sum = Reduce(tmp).Sum(sum);
  if (threadIdx.x == 0) partials[blockIdx.x] = sum;
  if (blockIdx.x != 0) return;
  unsigned long long kept = 0;
  if (kept_counts) {
    __syncthreads();  // tmp is reused
    for (int f = threadIdx.x; f < F; f += kScanThreads) kept += kept_counts[f];
    kept = Reduce(tmp).Sum(kept);
  }
  if (threadIdx.x == 0) {
    c->points_kept = kept;
    const uint32_t nb = *num_rays;
    c->hole_sentinel = kept_counts && sorted_keys && nb > 0 && heads[nb - 1] == kept &&
                       sorted_keys[heads[nb - 1]] == kInvalidPointKey;
  }
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

int32_t front_enqueue(cg_context* ctx, FrontBufs& fb, cudaStream_t s, int32_t* d_err,
                      const cg_layer* L, const cg_integrator_config* cfg, const IntegratorParams& P,
                      const float* d_points, const uint8_t* d_colors, const uint64_t* offs,
                      const uint32_t* d_counts, size_t f0, size_t f1, int attempt, bool* need_split) {
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
  const uint32_t* group_counts = d_counts ? d_counts + f0 : nullptr;
  const FrameTable ft{fb.frame_base.as<uint64_t>() + f0, offs[f0] - offs[0], static_cast<int>(F),
                      group_counts};
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
      constexpr unsigned wide_per_sm = 4, short_per_sm = 4;
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
                                                   fb.scan_partials.as<unsigned long long>(),
                                                   group_counts, static_cast<int>(F),
                                                   merged ? dk.Current() : nullptr,
                                                   fb.scan.as<uint32_t>(), fb.d_counters);
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

FrontVerdict front_digest(cg_context* ctx, const FrontBufs& fb, bool merged, size_t F, int attempt,
                          int32_t* rc) {
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

// The job's poses and frame offsets (relative to its first point) go up once per job, through a
// pinned, device-mapped host buffer and a copy KERNEL: an H2D memcpy would be queued on the copy
// engine behind the point data that the staging / pipelined paths have in flight.
__global__ void k_copy_words(uint32_t* __restrict__ dst, const uint32_t* __restrict__ src, size_t n) {
  const size_t i = blockIdx.x * static_cast<size_t>(blockDim.x) + threadIdx.x;
  if (i < n) dst[i] = src[i];
}
int32_t upload_frame_tables(FrontBufs& fb, size_t F, const float* h_poses, const uint64_t* offs,
                            cudaStream_t stream) {
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

}  // namespace cg
