// integrate_back.cu — back half of the TSDF integration: rays to voxels (R3, R4, R5).
//
// The voxels a job visits fall in two classes.  Nearly all of them (the carved free space) only
// ever see observations with sdf >= truncation while being fresh or already saturated at
// +truncation: for those updateTsdfVoxel degenerates to "D = trunc, W = min(max_weight, W + sum
// of the ray weights)", which needs no ordering — a fixed-point sum per voxel (deterministic, the
// adds commute exactly).  The rest ("general" voxels: any observation inside the truncation band
// or behind the surface, or a previous state that is not saturated) replay their updates in the
// reference's order.
//   k_walk_segments     3-D DDA per ray (voxblox::RayCaster); every visited block enters the GPU
//                       hash (allocation on first visit, R4); one record per (ray, block); voxels
//                       whose update order matters are flagged "general"
//   k_mark_existing     voxels of previously existing blocks whose state is not saturated
//   k_segment_hist / k_segment_scatter    segments grouped by block
//   k_block_accumulate  per block, in shared memory: commutative weight sums of the free-space
//                       visits; visits of general voxels go out as (voxel, ray) keys
//   radix sort (keys)   per-voxel update lists in canonical order
//   k_visit_precompute  the state-independent part of every ordered update
//   k_voxel_update / k_long_partials / k_long_finish   ordered replay of the general voxels
//   k_finalize_blocks   one CTA per touched block: coalesced read-modify-write of the remaining
//                       voxels from the accumulators; resets the per-call scratch.
#include <cub/cub.cuh>
#include <thrust/iterator/counting_iterator.h>

#include <algorithm>
#include <type_traits>

#include "integrate.cuh"

namespace cg {

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

int32_t run_back_half(cg_context* ctx, const FrontBufs& fb, cg_layer* L, const IntegratorParams& P,
                      uint32_t num_rays, size_t num_pairs, size_t num_segments,
                      cg_integrate_stats* stats) {
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
  uint32_t slack = P.anti_grazing ? 8 : 1;
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

}  // namespace cg
