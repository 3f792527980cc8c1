// esdf.cu — ESDF of the device-resident TSDF layer (SURVEY.md §8f N4, second half).
//
// Replaces voxblox::EsdfIntegrator::updateFromTsdfLayerBatch() as the client's MapServer calls it
// right after the merge (coxgraph/include/coxgraph/client/map_server.h:141-145, reached from
// coxgraph/src/client/map_server.cpp:99) and voxblox::createFreePointcloudFromEsdfLayer
// (coxgraph/src/client/map_server.cpp:112-113), so that neither the merged TSDF nor the ESDF has to
// leave the GPU to get the traversable cloud.
//
// Upstream ([EXT] integrator/esdf_integrator.cc) is a sequential label-correcting wavefront: voxels
// with |tsdf distance| < min_distance are copied and fixed, every other observed voxel starts at
// +-default_distance and processOpenSet lowers |distance| through the 26-neighbourhood
// (quasi-Euclidean: + voxel_size * {1, sqrt2, sqrt3} per hop) between voxels of equal sign, from
// voxels with |distance| < max_distance, taking an update when it improves by more than min_diff_m.
// The fixed point of that relaxation for min_diff_m = 0 is unique — the operator
//   d(n) <- min(d(n), min over eligible neighbours v of fl(d(v) + w))
// is monotone in every d(v), floats included — so ANY order of relaxations ends in the same
// bits.  That is what is computed here, block-parallel:
//   k_esdf_init   working plane per block (NaN = unobserved), bit plane of the fixed voxels
//   k_esdf_sweep  one CTA per dirty block: the block + a one-voxel halo of its 26 neighbours in
//                 shared memory, relaxed to the block-local fixed point (z-columns per thread,
//                 forward and backward); if a face changed, the neighbour blocks behind it are
//                 dirty in the next sweep.  Sweeps repeat until no block is dirty.
//   k_esdf_finish parent direction, flag byte, NaN -> the default-constructed voxel
// With min_diff_m > 0 upstream stops early and may stay above this fixed point by less than
// min_diff_m per hop (tests bound it); `parent` follows upstream's queue order there and a fixed
// neighbour order here (faces, edges, corners; first neighbour that attains the distance).
//
// cg_layer_esdf_update (updateFromTsdfLayer) starts from the retained result instead: it finds the
// voxels whose init state changed (k_esdf_compare), re-initialises every block within reach of them
// (k_esdf_dilate) and runs the same sweeps and finish over those blocks only; DESIGN §4.6 has the
// argument that this ends in the batch's bits.
#include <cub/cub.cuh>

#include <algorithm>
#include <cmath>
#include <cstring>
#include <utility>

#include "cg_internal.cuh"

namespace cg {

constexpr int kEsdfThreads = 256;
constexpr int kTileSide = kVps + 2;             // 18
constexpr int kTileRow = kTileSide;             // x stride 1, y stride 18
constexpr int kTilePlane = kTileSide * kTileSide;
constexpr int kTileVoxels = kTileSide * kTileSide * kTileSide;  // 5832 floats = 23,328 B

struct EsdfParams {
  float max_distance, default_distance, min_distance, min_weight;
  float w1, w2, w3;  // voxel_size * {1, sqrt2, sqrt3} (NeighborhoodLookupTables::kDistances)
  int crust;
};

__device__ __forceinline__ float quiet_nan() { return __int_as_float(0x7FC00000); }

// 26 neighbours: faces, edges, corners; dz / dy / dx ascending inside a class
struct NeighborTable {
  int8_t dx[26], dy[26], dz[26], cls[26];
};
__constant__ NeighborTable c_nb;

// the init state of a block's voxels; `list` (may be null: all n blocks) names the blocks,
// `counters` (may be null) receives the observed / fixed totals
__global__ void k_esdf_init(LayerView L, const uint32_t* __restrict__ slots,
                            const uint32_t* __restrict__ list, uint32_t n, EsdfParams P,
                            float* __restrict__ dist, uint32_t* __restrict__ fixed_bits,
                            int32_t* __restrict__ slot_to_b, uint8_t* __restrict__ dirty,
                            unsigned long long* __restrict__ counters) {
  unsigned long long n_obs = 0, n_fixed = 0;
  for (uint32_t item = blockIdx.x; item < n; item += gridDim.x) {
    const uint32_t b = list ? list[item] : item;
    const int slot = static_cast<int>(slots[b]);
    const float* td = L.dist_plane(slot);
    const float* tw = L.weight_plane(slot);
    if (threadIdx.x == 0) {
      slot_to_b[slot] = static_cast<int32_t>(b);
      dirty[b] = 1;
    }
    for (int i = threadIdx.x; i < kVoxelsPerBlock; i += kEsdfThreads) {
      const float d = td[i], w = tw[i];
      float out;
      bool fixed = false;
      if (w < P.min_weight) {
        out = P.crust ? -P.default_distance : quiet_nan();
      } else {
        fixed = fabsf(d) < P.min_distance;  // EsdfIntegrator::isFixed
        const float sgn = d == 0.0f ? 0.0f : (d < 0.0f ? -1.0f : 1.0f);
        out = fixed ? d : sgn * P.default_distance;
        ++n_obs;
        n_fixed += fixed ? 1 : 0;
      }
      dist[static_cast<size_t>(b) * kVoxelsPerBlock + i] = out;
      const uint32_t bits = __ballot_sync(0xFFFFFFFFu, fixed);
      if ((threadIdx.x & 31) == 0) fixed_bits[static_cast<size_t>(b) * 128 + (i >> 5)] = bits;
    }
  }
  if (!counters) return;
  n_obs = __reduce_add_sync(0xFFFFFFFFu, static_cast<unsigned>(n_obs));
  n_fixed = __reduce_add_sync(0xFFFFFFFFu, static_cast<unsigned>(n_fixed));
  if ((threadIdx.x & 31) == 0) {
    atomicAdd(&counters[0], n_obs);
    atomicAdd(&counters[1], n_fixed);
  }
}

__global__ void k_esdf_collect(uint8_t* __restrict__ dirty, uint32_t n, uint32_t* __restrict__ list,
                               uint32_t* __restrict__ count) {
  const uint32_t b = blockIdx.x * blockDim.x + threadIdx.x;
  if (b >= n || !dirty[b]) return;
  dirty[b] = 0;
  list[atomicAdd(count, 1u)] = b;
}

// neighbour blocks of block key `key` as positions in the sorted block list (-1: not allocated)
__device__ __forceinline__ void load_neighbor_table(const LayerView& L, uint64_t key,
                                                    const int32_t* __restrict__ slot_to_b,
                                                    int* table) {
  if (threadIdx.x < 27) {
    int bx, by, bz;
    unpack_block_key(key, bx, by, bz);
    const int t = threadIdx.x;
    const int dx = t % 3 - 1, dy = (t / 3) % 3 - 1, dz = t / 9 - 1;
    const int slot = L.find_slot(pack_block_key(bx + dx, by + dy, bz + dz));
    table[t] = slot < 0 ? -1 : slot_to_b[slot];
  }
}

// the block's 16^3 voxels and the one-voxel shell around them
__device__ __forceinline__ void load_tile(const float* __restrict__ dist, uint32_t b,
                                          const int* table, float* tile) {
  const float* own = dist + static_cast<size_t>(b) * kVoxelsPerBlock;
  for (int z = 0; z < kVps; ++z)
    tile[(z + 1) * kTilePlane + ((threadIdx.x >> 4) + 1) * kTileRow + (threadIdx.x & 15) + 1] =
        own[z * 256 + threadIdx.x];
  for (int i = threadIdx.x; i < kTileVoxels; i += kEsdfThreads) {
    const int hx = i % kTileSide - 1, hy = (i / kTileSide) % kTileSide - 1, hz = i / kTilePlane - 1;
    const int ox = hx < 0 ? 0 : (hx > 15 ? 2 : 1), oy = hy < 0 ? 0 : (hy > 15 ? 2 : 1),
              oz = hz < 0 ? 0 : (hz > 15 ? 2 : 1);
    if (ox == 1 && oy == 1 && oz == 1) continue;
    const int nb = table[ox + 3 * oy + 9 * oz];
    float v = quiet_nan();
    if (nb >= 0)
      v = __ldcg(dist + static_cast<size_t>(nb) * kVoxelsPerBlock + (hx & 15) + 16 * ((hy & 15) + 16 * (hz & 15)));
    tile[i] = v;
  }
}

// |distance| a voxel of sign s can take from its 26 neighbours (the current magnitude if none helps)
__device__ __forceinline__ float relax_voxel(const float* t, float s, float m, const EsdfParams& P) {
#define CG_ESDF_TAP(off, w)                         \
  {                                                 \
    const float a = s * t[off];                     \
    if (a > 0.0f && a < P.max_distance) m = fminf(m, a + (w)); \
  }
  CG_ESDF_TAP(-1, P.w1) CG_ESDF_TAP(1, P.w1) CG_ESDF_TAP(-kTileRow, P.w1) CG_ESDF_TAP(kTileRow, P.w1)
  CG_ESDF_TAP(-kTilePlane, P.w1) CG_ESDF_TAP(kTilePlane, P.w1)
  CG_ESDF_TAP(-kTileRow - 1, P.w2) CG_ESDF_TAP(-kTileRow + 1, P.w2) CG_ESDF_TAP(kTileRow - 1, P.w2)
  CG_ESDF_TAP(kTileRow + 1, P.w2) CG_ESDF_TAP(-kTilePlane - 1, P.w2) CG_ESDF_TAP(-kTilePlane + 1, P.w2)
  CG_ESDF_TAP(kTilePlane - 1, P.w2) CG_ESDF_TAP(kTilePlane + 1, P.w2)
  CG_ESDF_TAP(-kTilePlane - kTileRow, P.w2) CG_ESDF_TAP(-kTilePlane + kTileRow, P.w2)
  CG_ESDF_TAP(kTilePlane - kTileRow, P.w2) CG_ESDF_TAP(kTilePlane + kTileRow, P.w2)
  CG_ESDF_TAP(-kTilePlane - kTileRow - 1, P.w3) CG_ESDF_TAP(-kTilePlane - kTileRow + 1, P.w3)
  CG_ESDF_TAP(-kTilePlane + kTileRow - 1, P.w3) CG_ESDF_TAP(-kTilePlane + kTileRow + 1, P.w3)
  CG_ESDF_TAP(kTilePlane - kTileRow - 1, P.w3) CG_ESDF_TAP(kTilePlane - kTileRow + 1, P.w3)
  CG_ESDF_TAP(kTilePlane + kTileRow - 1, P.w3) CG_ESDF_TAP(kTilePlane + kTileRow + 1, P.w3)
#undef CG_ESDF_TAP
  return m;
}

__global__ void __launch_bounds__(kEsdfThreads)
k_esdf_sweep(LayerView L, const uint64_t* __restrict__ keys, const uint32_t* __restrict__ list,
             const uint32_t* __restrict__ count, EsdfParams P, float* __restrict__ dist,
             const uint32_t* __restrict__ fixed_bits, const int32_t* __restrict__ slot_to_b,
             const uint8_t* __restrict__ region, uint8_t* __restrict__ dirty) {
  __shared__ float tile[kTileVoxels];
  __shared__ int table[27];
  __shared__ uint32_t face_flags;
  const uint32_t n = *count;
  const int x = threadIdx.x & 15, y = threadIdx.x >> 4;
  const int col = (y + 1) * kTileRow + x + 1;  // this thread's z-column
  for (uint32_t item = blockIdx.x; item < n; item += gridDim.x) {
    const uint32_t b = list[item];
    __syncthreads();  // the previous item's tile is done with
    load_neighbor_table(L, keys[b], slot_to_b, table);
    if (threadIdx.x == 0) face_flags = 0;
    __syncthreads();
    load_tile(dist, b, table, tile);
    // voxels this thread may change: observed (not NaN) and not fixed
    uint32_t live = 0;
    {
      const uint32_t* fb = fixed_bits + static_cast<size_t>(b) * 128;
      for (int z = 0; z < kVps; ++z) {
        const uint32_t word = fb[z * 8 + (threadIdx.x >> 5)];
        const float own = dist[static_cast<size_t>(b) * kVoxelsPerBlock + z * 256 + threadIdx.x];
        if (!((word >> (threadIdx.x & 31)) & 1u) && own == own && own != 0.0f) live |= 1u << z;
      }
    }
    __syncthreads();
    // relax to the block-local fixed point; reads of values a neighbour thread is lowering at the
    // same time are merely stale (the relaxation is monotone), the round after the last change
    // reads settled values only
    for (;;) {
      bool changed = false;
      for (int pass = 0; pass < 2; ++pass) {
        for (int k = 0; k < kVps; ++k) {
          const int z = pass ? kVps - 1 - k : k;
          if (!((live >> z) & 1u)) continue;
          float* t = tile + (z + 1) * kTilePlane + col;
          const float cur = *t;
          const float s = cur < 0.0f ? -1.0f : 1.0f;
          const float m0 = fabsf(cur);
          const float m = relax_voxel(t, s, m0, P);
          if (m < m0) {
            *t = s * m;
            changed = true;
          }
        }
        __syncthreads();
      }
      if (!__syncthreads_or(changed)) break;
    }
    // write back what changed; a changed face wakes the blocks behind it (those of the region
    // only, when one is given: the values outside it are final)
    uint32_t faces = 0;
    float* own = dist + static_cast<size_t>(b) * kVoxelsPerBlock;
    for (int z = 0; z < kVps; ++z) {
      if (!((live >> z) & 1u)) continue;
      const float v = tile[(z + 1) * kTilePlane + col];
      if (v != own[z * 256 + threadIdx.x]) {
        own[z * 256 + threadIdx.x] = v;
        faces |= (x == 0 ? 1u : 0u) | (x == 15 ? 2u : 0u) | (y == 0 ? 4u : 0u) | (y == 15 ? 8u : 0u) |
                 (z == 0 ? 16u : 0u) | (z == 15 ? 32u : 0u);
      }
    }
    faces = __reduce_or_sync(0xFFFFFFFFu, faces);
    if ((threadIdx.x & 31) == 0 && faces) atomicOr(&face_flags, faces);
    __syncthreads();
    if (threadIdx.x < 27 && threadIdx.x != 13 && table[threadIdx.x] >= 0) {
      const int t = threadIdx.x;
      const int dx = t % 3 - 1, dy = (t / 3) % 3 - 1, dz = t / 9 - 1;
      const uint32_t need = (dx < 0 ? 1u : dx > 0 ? 2u : 0u) | (dy < 0 ? 4u : dy > 0 ? 8u : 0u) |
                            (dz < 0 ? 16u : dz > 0 ? 32u : 0u);
      if ((face_flags & need) == need && (!region || region[table[t]])) dirty[table[t]] = 1;
    }
  }
}

// flag byte + parent of every voxel; unobserved voxels become the default-constructed EsdfVoxel
// (distance 0) in the working plane itself, which then is the result plane.
// packed = parent.x << 24 | parent.y << 16 | parent.z << 8 | flags (Block<EsdfVoxel>::
// serializeToIntegers' second word); flags: 1 observed, 2 hallucinated, 4 in_queue, 8 fixed
__global__ void __launch_bounds__(kEsdfThreads)
k_esdf_finish(LayerView L, const uint64_t* __restrict__ keys, const uint32_t* __restrict__ slots,
              const uint32_t* __restrict__ list, uint32_t n, EsdfParams P, float* dist,
              const uint32_t* __restrict__ fixed_bits, const int32_t* __restrict__ slot_to_b,
              uint32_t* __restrict__ packed) {
  __shared__ float tile[kTileVoxels];
  __shared__ int table[27];
  const int x = threadIdx.x & 15, y = threadIdx.x >> 4;
  const int col = (y + 1) * kTileRow + x + 1;
  for (uint32_t item = blockIdx.x; item < n; item += gridDim.x) {
    const uint32_t b = list ? list[item] : item;
    __syncthreads();
    load_neighbor_table(L, keys[b], slot_to_b, table);
    __syncthreads();
    load_tile(dist, b, table, tile);
    __syncthreads();
    const float* tw = L.weight_plane(static_cast<int>(slots[b]));
    const uint32_t* fb = fixed_bits + static_cast<size_t>(b) * 128;
    for (int z = 0; z < kVps; ++z) {
      const int lin = z * 256 + threadIdx.x;
      const float* t = tile + (z + 1) * kTilePlane + col;
      const float cur = *t;
      const bool fixed = (fb[z * 8 + (threadIdx.x >> 5)] >> (threadIdx.x & 31)) & 1u;
      const bool observed = cur == cur;
      const bool hallucinated = observed && tw[lin] < P.min_weight;
      uint32_t word = (observed ? 1u : 0u) | (hallucinated ? 2u : 0u) | (fixed ? 8u : 0u);
      if (observed && !fixed && cur != 0.0f && fabsf(cur) < P.default_distance) {
        const float s = cur < 0.0f ? -1.0f : 1.0f, m = fabsf(cur);
        for (int k = 0; k < 26; ++k) {
          const int dx = c_nb.dx[k], dy = c_nb.dy[k], dz = c_nb.dz[k];
          const float a = s * t[dz * kTilePlane + dy * kTileRow + dx];
          const float w = c_nb.cls[k] == 1 ? P.w1 : (c_nb.cls[k] == 2 ? P.w2 : P.w3);
          if (a > 0.0f && a < P.max_distance && a + w == m) {
            word |= (static_cast<uint32_t>(dx & 0xFF) << 24) | (static_cast<uint32_t>(dy & 0xFF) << 16) |
                    (static_cast<uint32_t>(dz & 0xFF) << 8);
            break;
          }
        }
      }
      // in place: only NaNs are rewritten, and a 0 in a neighbour's halo is no source either
      // (sources need s * d > 0), so blocks finished earlier do not disturb later ones
      if (!observed) dist[static_cast<size_t>(b) * kVoxelsPerBlock + lin] = 0.0f;
      packed[static_cast<size_t>(b) * kVoxelsPerBlock + lin] = word;
    }
  }
}

// createFreePointcloudFromEsdfLayer: count, then write (x, y, z, distance) in block / linear order
template <bool kWrite>
__global__ void __launch_bounds__(kEsdfThreads)
k_esdf_free(const uint64_t* __restrict__ keys, uint32_t n, const float* __restrict__ dist,
            const uint32_t* __restrict__ packed, float min_distance, float voxel_size,
            float block_size, uint32_t* __restrict__ counts, const uint32_t* __restrict__ begin,
            float4* __restrict__ out) {
  __shared__ uint32_t warp_sum[kEsdfThreads / 32];
  __shared__ uint32_t running;
  for (uint32_t b = blockIdx.x; b < n; b += gridDim.x) {
    if (threadIdx.x == 0) running = 0;
    __syncthreads();
    int bx, by, bz;
    unpack_block_key(keys[b], bx, by, bz);
    for (int z = 0; z < kVps; ++z) {  // linear order: 256 voxels per round
      const int lin = z * 256 + threadIdx.x;
      const size_t o = static_cast<size_t>(b) * kVoxelsPerBlock + lin;
      const float d = dist[o];
      const bool take = (packed[o] & 1u) && d >= min_distance;
      const uint32_t ballot = __ballot_sync(0xFFFFFFFFu, take);
      const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
      if (lane == 0) warp_sum[warp] = __popc(ballot);
      __syncthreads();
      uint32_t before = running;
      for (int w = 0; w < warp; ++w) before += warp_sum[w];
      if (kWrite && take) {
        const uint32_t pos = begin[b] + before + __popc(ballot & ((1u << lane) - 1u));
        // Block::computeCoordinatesFromVoxelIndex: origin + (index + 0.5) * voxel_size, the
        // centre evaluated in double and rounded once (the 0.5 is a double literal upstream)
        const float cx = static_cast<float>((static_cast<double>(static_cast<float>(lin & 15)) + 0.5) * static_cast<double>(voxel_size));
        const float cy = static_cast<float>((static_cast<double>(static_cast<float>((lin >> 4) & 15)) + 0.5) * static_cast<double>(voxel_size));
        const float cz = static_cast<float>((static_cast<double>(static_cast<float>(z)) + 0.5) * static_cast<double>(voxel_size));
        out[pos] = make_float4(static_cast<float>(bx) * block_size + cx,
                               static_cast<float>(by) * block_size + cy,
                               static_cast<float>(bz) * block_size + cz, d);
      }
      __syncthreads();
      if (threadIdx.x == 0) {
        uint32_t total = 0;
        for (int w = 0; w < kEsdfThreads / 32; ++w) total += warp_sum[w];
        running += total;
      }
      __syncthreads();
    }
    if (!kWrite && threadIdx.x == 0) counts[b] = running;
  }
}

// ------------------------------------------------------------------ incremental update
// Counters of one update (uint32 words after the batch's counters): see cg_layer_esdf_update.
enum UpdateCount { kUcSources = 0, kUcRemoved, kUcMoved, kUcChanged, kUcRegion, kUcWords = 8 };

// position of `key` in the sorted `keys[0, n)`, or -1
__device__ __forceinline__ int32_t find_sorted(const uint64_t* __restrict__ keys, uint32_t n,
                                               uint64_t key) {
  uint32_t lo = 0, hi = n;
  while (lo < hi) {
    const uint32_t mid = (lo + hi) >> 1;
    if (keys[mid] < key) lo = mid + 1; else hi = mid;
  }
  return lo < n && keys[lo] == key ? static_cast<int32_t>(lo) : -1;
}

// Matches the new block list with the retained one by key (slots are not stable: removing blocks
// compacts the pool).  New block b -> old_b[b] (-1: new block); retained blocks the layer no
// longer has are sources of the region.
__global__ void k_esdf_match(const uint64_t* __restrict__ keys, const uint32_t* __restrict__ slots,
                             uint32_t n, const uint64_t* __restrict__ old_keys, uint32_t n_old,
                             int32_t* __restrict__ old_b, int32_t* __restrict__ slot_to_b,
                             uint64_t* __restrict__ sources, uint32_t* __restrict__ ucount) {
  const uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i < n) {
    const int32_t ob = find_sorted(old_keys, n_old, keys[i]);
    old_b[i] = ob;
    slot_to_b[slots[i]] = static_cast<int32_t>(i);
    if (ob != static_cast<int32_t>(i)) atomicAdd(&ucount[kUcMoved], 1u);
  }
  if (i < n_old && find_sorted(keys, n, old_keys[i]) < 0) {
    sources[atomicAdd(&ucount[kUcSources], 1u)] = old_keys[i];
    atomicAdd(&ucount[kUcRemoved], 1u);
  }
}

// One pass over every block: the new init state of each voxel (k_esdf_init's rule) against the
// one the retained result implies — fixed voxels kept their distance, other observed voxels
// started at sign(result) * default (0 stays 0), unobserved ones have packed & 1 == 0 and the
// hallucinated bit is packed & 2.  A block with any difference, or without a retained block, is a
// source of the region.  Also counts the observed / fixed voxels of the whole map.
__global__ void __launch_bounds__(kEsdfThreads)
k_esdf_compare(LayerView L, const uint64_t* __restrict__ keys, const uint32_t* __restrict__ slots,
               uint32_t n, EsdfParams P, const int32_t* __restrict__ old_b,
               const float* __restrict__ old_dist, const uint32_t* __restrict__ old_packed,
               uint64_t* __restrict__ sources, uint32_t* __restrict__ ucount,
               unsigned long long* __restrict__ counters) {
  unsigned long long n_obs = 0, n_fixed = 0;
  for (uint32_t b = blockIdx.x; b < n; b += gridDim.x) {
    const int slot = static_cast<int>(slots[b]);
    const int32_t ob = old_b[b];
    const float* td = L.dist_plane(slot);
    const float* tw = L.weight_plane(slot);
    bool changed = ob < 0;
    for (int i = threadIdx.x; i < kVoxelsPerBlock; i += kEsdfThreads) {
      const float d = td[i], w = tw[i];
      uint32_t flags;  // 1 observed, 2 hallucinated, 8 fixed
      float init = 0.0f;
      if (w < P.min_weight) {
        flags = P.crust ? 3u : 0u;
        init = -P.default_distance;
      } else {
        const bool fixed = fabsf(d) < P.min_distance;
        const float sgn = d == 0.0f ? 0.0f : (d < 0.0f ? -1.0f : 1.0f);
        init = fixed ? d : sgn * P.default_distance;
        flags = fixed ? 9u : 1u;
        ++n_obs;
        n_fixed += fixed ? 1 : 0;
      }
      if (ob >= 0) {
        const size_t o = static_cast<size_t>(ob) * kVoxelsPerBlock + i;
        const uint32_t op = __ldcs(old_packed + o) & 11u;
        const float od = __ldcs(old_dist + o);
        const float oinit = (op & 8u) ? od : (od == 0.0f ? 0.0f : (od < 0.0f ? -P.default_distance : P.default_distance));
        if (op != flags || ((flags & 1u) && __float_as_uint(oinit) != __float_as_uint(init))) changed = true;
      }
    }
    if (__syncthreads_or(changed) && threadIdx.x == 0) {
      sources[atomicAdd(&ucount[kUcSources], 1u)] = keys[b];
      atomicAdd(&ucount[kUcChanged], 1u);
    }
  }
  n_obs = __reduce_add_sync(0xFFFFFFFFu, static_cast<unsigned>(n_obs));
  n_fixed = __reduce_add_sync(0xFFFFFFFFu, static_cast<unsigned>(n_fixed));
  if ((threadIdx.x & 31) == 0) {
    atomicAdd(&counters[0], n_obs);
    atomicAdd(&counters[1], n_fixed);
  }
}

// region: every current block within block-Chebyshev distance r of a source key, probed in the
// layer's hash
__global__ void k_esdf_dilate(LayerView L, const uint64_t* __restrict__ sources,
                              const uint32_t* __restrict__ ucount, int r,
                              const int32_t* __restrict__ slot_to_b, uint8_t* __restrict__ region) {
  const uint32_t n = ucount[kUcSources];
  const int side = 2 * r + 1, cube = side * side * side;
  for (uint32_t s = blockIdx.x; s < n; s += gridDim.x) {
    int bx, by, bz;
    unpack_block_key(sources[s], bx, by, bz);
    for (int o = threadIdx.x; o < cube; o += blockDim.x) {
      const int slot = L.find_slot(pack_block_key(bx + o % side - r, by + (o / side) % side - r,
                                                  bz + o / (side * side) - r));
      if (slot >= 0) region[slot_to_b[slot]] = 1;
    }
  }
}

__global__ void k_esdf_region_list(const uint8_t* __restrict__ region, uint32_t n,
                                   uint32_t* __restrict__ list, uint32_t* __restrict__ ucount) {
  const uint32_t b = blockIdx.x * blockDim.x + threadIdx.x;
  if (b < n && region[b]) list[atomicAdd(&ucount[kUcRegion], 1u)] = b;
}

// the retained distance and packed planes of the blocks outside the region to their new positions
// (every block outside the region has a retained block: new blocks are sources)
__global__ void __launch_bounds__(kEsdfThreads)
k_esdf_remap(const uint8_t* __restrict__ region, const int32_t* __restrict__ old_b, uint32_t n,
             const float4* __restrict__ old_dist, const uint4* __restrict__ old_packed,
             float4* __restrict__ dist, uint4* __restrict__ packed) {
  constexpr int kVec = kVoxelsPerBlock / 4;
  for (uint32_t b = blockIdx.x; b < n; b += gridDim.x) {
    if (region[b]) continue;
    const size_t src = static_cast<size_t>(old_b[b]) * kVec, dst = static_cast<size_t>(b) * kVec;
    for (int i = threadIdx.x; i < kVec; i += kEsdfThreads) {
      dist[dst + i] = __ldcs(old_dist + src + i);
      packed[dst + i] = __ldcs(old_packed + src + i);
    }
  }
}

static float float_from_bits(uint32_t u) {
  float f;
  memcpy(&f, &u, sizeof(f));
  return f;
}

static cudaError_t upload_neighbor_table() {
  static bool done[64] = {};
  int dev = 0;
  cudaGetDevice(&dev);
  if (dev >= 0 && dev < 64 && done[dev]) return cudaSuccess;
  NeighborTable t;
  int k = 0;
  for (int order = 1; order <= 3; ++order)
    for (int dz = -1; dz <= 1; ++dz)
      for (int dy = -1; dy <= 1; ++dy)
        for (int dx = -1; dx <= 1; ++dx)
          if (abs(dx) + abs(dy) + abs(dz) == order) {
            t.dx[k] = static_cast<int8_t>(dx);
            t.dy[k] = static_cast<int8_t>(dy);
            t.dz[k] = static_cast<int8_t>(dz);
            t.cls[k] = static_cast<int8_t>(order);
            ++k;
          }
  cudaError_t e = cudaMemcpyToSymbol(c_nb, &t, sizeof(t));
  if (e == cudaSuccess && dev >= 0 && dev < 64) done[dev] = true;
  return e;
}

static int32_t check_config(const cg_esdf_config* cfg, const char* fn) {
  if (cfg->full_euclidean_distance) {
    set_error("%s: full_euclidean_distance is not implemented (upstream default: off)", fn);
    return CG_ERR_UNSUPPORTED;
  }
  if (!(cfg->max_distance_m > 0.0f) || !(cfg->default_distance_m >= cfg->max_distance_m) ||
      !(cfg->min_distance_m >= 0.0f)) {
    set_error("%s: need max_distance_m > 0, default_distance_m >= max_distance_m "
              "(as voxblox_ros' parameter loader enforces), min_distance_m >= 0", fn);
    return CG_ERR_INVALID_ARG;
  }
  return CG_OK;
}

static EsdfParams make_params(const cg_layer* L, const cg_esdf_config* cfg) {
  EsdfParams P;
  P.max_distance = cfg->max_distance_m;
  P.default_distance = cfg->default_distance_m;
  P.min_distance = cfg->min_distance_m;
  P.min_weight = cfg->min_weight;
  P.w1 = 1.0f * L->v.voxel_size;
  P.w2 = float_from_bits(0x3FB504F3) * L->v.voxel_size;  // float(sqrt(2))
  P.w3 = float_from_bits(0x3FDDB3D7) * L->v.voxel_size;  // float(sqrt(3))
  P.crust = cfg->add_occupied_crust ? 1 : 0;
  return P;
}

// the config fields the result depends on, compared bit for bit
static bool same_result_config(const cg_esdf_config& a, const cg_esdf_config& b) {
  return memcmp(&a.max_distance_m, &b.max_distance_m, sizeof(float)) == 0 &&
         memcmp(&a.default_distance_m, &b.default_distance_m, sizeof(float)) == 0 &&
         memcmp(&a.min_distance_m, &b.min_distance_m, sizeof(float)) == 0 &&
         memcmp(&a.min_weight, &b.min_weight, sizeof(float)) == 0 &&
         (a.add_occupied_crust != 0) == (b.add_occupied_crust != 0);
}

// Block radius R of the region around a changed block (DESIGN §4.6).  A voxel feeds a neighbour
// only while |d| < max_distance and every hop adds at least w1 = voxel_size, so a voxel's result
// depends on the init states within L = ceil(max / w1) + 1 hops; one more hop covers the rounding
// of fl(a + w) (k hops lose less than k * 2^-24 relative, under one hop while k < 4096), and the
// packed word also reads the 26 neighbours' results: L + 2 voxels, R = ceil((L + 2) / 16) blocks.
static int region_reach(const cg_layer* L, const cg_esdf_config* cfg) {
  const double hops = std::ceil(static_cast<double>(cfg->max_distance_m) /
                                static_cast<double>(L->v.voxel_size)) + 2.0;
  return static_cast<int>(std::ceil((hops + 1.0) / kVps));
}

// the retained ESDF is now that of `L` under `cfg`
static int32_t retain(cg_context* ctx, const cg_layer* L, const cg_esdf_config* cfg, size_t n) {
  ctx->esdf_blocks = n;
  ctx->esdf_serial = L->serial;
  ctx->esdf_cfg = *cfg;
  ctx->esdf_voxel_size = L->v.voxel_size;
  ctx->esdf_block_size = L->v.block_size;
  return CG_OK;
}

// Sweeps over the dirty blocks until none is left.  With `region`, only region blocks are woken.
static int32_t run_sweeps(cg_context* ctx, const cg_layer* L, const uint64_t* keys, size_t n,
                          const EsdfParams& P, const uint8_t* region, uint64_t* sweeps,
                          uint64_t* passes, const char* fn) {
  cudaStream_t s = ctx->stream;
  uint32_t* d_count = reinterpret_cast<uint32_t*>(ctx->esdf_counters.as<unsigned long long>() + 2);
  for (;;) {
    CG_CUDA(cudaMemsetAsync(d_count, 0, sizeof(uint32_t), s));
    k_esdf_collect<<<grid_for(n, 256), 256, 0, s>>>(ctx->esdf_dirty.as<uint8_t>(),
                                                    static_cast<uint32_t>(n),
                                                    ctx->esdf_list.as<uint32_t>(), d_count);
    uint32_t h_count = 0;
    CG_CUDA(cudaMemcpyAsync(&h_count, d_count, sizeof(uint32_t), cudaMemcpyDeviceToHost, s));
    CG_CUDA(cudaStreamSynchronize(s));
    ctx->own_launches += 1;
    if (h_count == 0) break;
    if (++*sweeps > 100000) {
      set_error("%s: no convergence", fn);
      return CG_ERR_CUDA;
    }
    *passes += h_count;
    const unsigned grid = std::min<unsigned>(h_count, static_cast<unsigned>(ctx->num_sms) * 8u);
    ctx->own_launches += 1;
    k_esdf_sweep<<<grid, kEsdfThreads, 0, s>>>(L->v, keys, ctx->esdf_list.as<uint32_t>(), d_count, P,
                                               ctx->esdf_dist.as<float>(),
                                               ctx->esdf_fixed.as<uint32_t>(),
                                               ctx->esdf_slot_to_b.as<int32_t>(), region,
                                               ctx->esdf_dirty.as<uint8_t>());
  }
  return CG_OK;
}

}  // namespace cg

using namespace cg;

extern "C" {

void cg_esdf_config_default(cg_esdf_config* c) {
  if (!c) return;
  c->max_distance_m = 2.0f;
  c->default_distance_m = 2.0f;
  c->min_distance_m = 0.2f;
  c->min_diff_m = 0.001f;
  c->min_weight = 1e-6f;
  c->num_buckets = 20;
  c->multi_queue = 0;
  c->add_occupied_crust = 0;
  c->full_euclidean_distance = 0;
}

int32_t cg_layer_esdf_batch(const cg_layer* L, const cg_esdf_config* cfg, cg_esdf_stats* stats) {
  if (!L || !cfg) return CG_ERR_INVALID_ARG;
  cg_context* ctx = L->ctx;
  CG_CUDA(cudaSetDevice(ctx->device));
  if (stats) memset(stats, 0, sizeof(*stats));
  int32_t rc = check_config(cfg, "cg_layer_esdf_batch");
  if (rc) return rc;
  cudaStream_t s = ctx->stream;
  const size_t n = static_cast<size_t>(L->num_blocks);
  ctx->esdf_blocks = 0;
  ctx->esdf_serial = 0;
  ctx->esdf_voxel_size = L->v.voxel_size;
  ctx->esdf_block_size = L->v.block_size;
  if (n == 0) return retain(ctx, L, cfg, 0);
  CG_CUDA(upload_neighbor_table());
  const uint64_t* keys;
  const uint32_t* slots;
  rc = sort_blocks(L, &keys, &slots);
  if (rc) return rc;
  // sort_blocks leaves its result in scratch other calls reuse: keep our own copy
  CG_CUDA(ctx->esdf_keys.reserve(n * sizeof(uint64_t)));
  CG_CUDA(ctx->esdf_slots.reserve(n * sizeof(uint32_t)));
  CG_CUDA(cudaMemcpyAsync(ctx->esdf_keys.p, keys, n * sizeof(uint64_t), cudaMemcpyDeviceToDevice, s));
  CG_CUDA(cudaMemcpyAsync(ctx->esdf_slots.p, slots, n * sizeof(uint32_t), cudaMemcpyDeviceToDevice, s));
  keys = ctx->esdf_keys.as<uint64_t>();
  slots = ctx->esdf_slots.as<uint32_t>();
  CG_CUDA(ctx->esdf_dist.reserve(n * kVoxelsPerBlock * sizeof(float)));
  CG_CUDA(ctx->esdf_packed.reserve(n * kVoxelsPerBlock * sizeof(uint32_t)));
  CG_CUDA(ctx->esdf_fixed.reserve(n * 128 * sizeof(uint32_t)));
  CG_CUDA(ctx->esdf_slot_to_b.reserve(n * sizeof(int32_t)));
  CG_CUDA(ctx->esdf_dirty.reserve(n));
  CG_CUDA(ctx->esdf_list.reserve(n * sizeof(uint32_t)));
  CG_CUDA(ctx->esdf_index.reserve(n * 3 * sizeof(int32_t)));
  CG_CUDA(ctx->esdf_counters.reserve(4 * sizeof(unsigned long long)));
  const EsdfParams P = make_params(L, cfg);
  unsigned long long* counters = ctx->esdf_counters.as<unsigned long long>();
  CG_CUDA(cudaMemsetAsync(counters, 0, 4 * sizeof(unsigned long long), s));
  const unsigned wide = static_cast<unsigned>(std::min<size_t>(n, static_cast<size_t>(ctx->num_sms) * 16));
  ctx->own_launches += 2;
  k_esdf_init<<<wide, kEsdfThreads, 0, s>>>(L->v, slots, nullptr, static_cast<uint32_t>(n), P,
                                            ctx->esdf_dist.as<float>(), ctx->esdf_fixed.as<uint32_t>(),
                                            ctx->esdf_slot_to_b.as<int32_t>(),
                                            ctx->esdf_dirty.as<uint8_t>(), counters);
  k_unpack_idx<<<grid_for(n, 256), 256, 0, s>>>(keys, static_cast<uint32_t>(n),
                                                ctx->esdf_index.as<int32_t>());
  uint64_t sweeps = 0, passes = 0;
  rc = run_sweeps(ctx, L, keys, n, P, nullptr, &sweeps, &passes, "cg_layer_esdf_batch");
  if (rc) return rc;
  ctx->own_launches += 1;
  k_esdf_finish<<<wide, kEsdfThreads, 0, s>>>(L->v, keys, slots, nullptr, static_cast<uint32_t>(n), P,
                                              ctx->esdf_dist.as<float>(),
                                              ctx->esdf_fixed.as<uint32_t>(),
                                              ctx->esdf_slot_to_b.as<int32_t>(),
                                              ctx->esdf_packed.as<uint32_t>());
  unsigned long long h_counters[2] = {0, 0};
  CG_CUDA(cudaMemcpyAsync(h_counters, counters, sizeof(h_counters), cudaMemcpyDeviceToHost, s));
  CG_CUDA(cudaStreamSynchronize(s));
  CG_CUDA(cudaGetLastError());
  if (stats) {
    stats->blocks = n;
    stats->observed_voxels = h_counters[0];
    stats->fixed_voxels = h_counters[1];
    stats->sweeps = sweeps;
    stats->block_passes = passes;
  }
  return retain(ctx, L, cfg, n);
}

int32_t cg_layer_esdf_update(const cg_layer* L, const cg_esdf_config* cfg, cg_esdf_stats* stats,
                             cg_esdf_update_stats* ust) {
  if (!L || !cfg) return CG_ERR_INVALID_ARG;
  cg_context* ctx = L->ctx;
  CG_CUDA(cudaSetDevice(ctx->device));
  if (stats) memset(stats, 0, sizeof(*stats));
  if (ust) memset(ust, 0, sizeof(*ust));
  int32_t rc = check_config(cfg, "cg_layer_esdf_update");
  if (rc) return rc;
  const size_t n = static_cast<size_t>(L->num_blocks), n_old = ctx->esdf_blocks;
  if (ctx->esdf_serial != L->serial || n_old == 0 || n == 0 || !same_result_config(ctx->esdf_cfg, *cfg)) {
    rc = cg_layer_esdf_batch(L, cfg, stats);
    if (rc == CG_OK && ust) {
      ust->blocks_changed = ust->blocks_region = n;
      ust->full_rebuild = 1;
    }
    return rc;
  }
  cudaStream_t s = ctx->stream;
  ctx->esdf_blocks = 0;  // until the update is complete
  ctx->esdf_serial = 0;
  CG_CUDA(upload_neighbor_table());
  const uint64_t* keys;
  const uint32_t* slots;
  rc = sort_blocks(L, &keys, &slots);
  if (rc) return rc;
  CG_CUDA(ctx->esdf_old_b.reserve(n * sizeof(int32_t)));
  CG_CUDA(ctx->esdf_sources.reserve((n + n_old) * sizeof(uint64_t)));
  CG_CUDA(ctx->esdf_region.reserve(n));
  CG_CUDA(ctx->esdf_region_list.reserve(n * sizeof(uint32_t)));
  CG_CUDA(ctx->esdf_fixed.reserve(n * 128 * sizeof(uint32_t)));  // read for region blocks only
  CG_CUDA(ctx->esdf_slot_to_b.reserve(n * sizeof(int32_t)));
  CG_CUDA(ctx->esdf_dirty.reserve(n));
  CG_CUDA(ctx->esdf_list.reserve(n * sizeof(uint32_t)));
  CG_CUDA(ctx->esdf_counters.reserve((4 + kUcWords / 2) * sizeof(unsigned long long)));
  const EsdfParams P = make_params(L, cfg);
  unsigned long long* counters = ctx->esdf_counters.as<unsigned long long>();
  uint32_t* ucount = reinterpret_cast<uint32_t*>(counters + 4);
  uint8_t* region = ctx->esdf_region.as<uint8_t>();
  int32_t* old_b = ctx->esdf_old_b.as<int32_t>();
  uint64_t* sources = ctx->esdf_sources.as<uint64_t>();
  uint32_t* region_list = ctx->esdf_region_list.as<uint32_t>();
  int32_t* slot_to_b = ctx->esdf_slot_to_b.as<int32_t>();
  CG_CUDA(cudaMemsetAsync(counters, 0, (4 + kUcWords / 2) * sizeof(unsigned long long), s));
  CG_CUDA(cudaMemsetAsync(region, 0, n, s));
  CG_CUDA(cudaMemsetAsync(ctx->esdf_dirty.p, 0, n, s));
  const unsigned wide = static_cast<unsigned>(std::min<size_t>(n, static_cast<size_t>(ctx->num_sms) * 16));
  ctx->own_launches += 4;
  k_esdf_match<<<grid_for(std::max(n, n_old), 256), 256, 0, s>>>(
      keys, slots, static_cast<uint32_t>(n), ctx->esdf_keys.as<uint64_t>(),
      static_cast<uint32_t>(n_old), old_b, slot_to_b, sources, ucount);
  k_esdf_compare<<<wide, kEsdfThreads, 0, s>>>(L->v, keys, slots, static_cast<uint32_t>(n), P, old_b,
                                               ctx->esdf_dist.as<float>(), ctx->esdf_packed.as<uint32_t>(),
                                               sources, ucount, counters);
  k_esdf_dilate<<<static_cast<unsigned>(std::min<size_t>(n + n_old, static_cast<size_t>(ctx->num_sms) * 8)),
                  kEsdfThreads, 0, s>>>(L->v, sources, ucount, region_reach(L, cfg), slot_to_b, region);
  k_esdf_region_list<<<grid_for(n, 256), 256, 0, s>>>(region, static_cast<uint32_t>(n), region_list, ucount);
  unsigned long long h_counters[4 + kUcWords / 2];
  CG_CUDA(cudaMemcpyAsync(h_counters, counters, sizeof(h_counters), cudaMemcpyDeviceToHost, s));
  CG_CUDA(cudaStreamSynchronize(s));
  uint32_t h_ucount[kUcWords];
  memcpy(h_ucount, h_counters + 4, sizeof(h_ucount));
  const uint32_t n_region = h_ucount[kUcRegion];
  if (h_ucount[kUcMoved] != 0 || n != n_old) {
    // the block list changed: the blocks outside the region move to their new positions in a
    // second pair of planes, which then becomes the retained one
    CG_CUDA(ctx->esdf_dist_next.reserve(n * kVoxelsPerBlock * sizeof(float)));
    CG_CUDA(ctx->esdf_packed_next.reserve(n * kVoxelsPerBlock * sizeof(uint32_t)));
    if (n_region < n) {
      ctx->own_launches += 1;
      k_esdf_remap<<<wide, kEsdfThreads, 0, s>>>(region, old_b, static_cast<uint32_t>(n),
                                                 ctx->esdf_dist.as<float4>(), ctx->esdf_packed.as<uint4>(),
                                                 ctx->esdf_dist_next.as<float4>(),
                                                 ctx->esdf_packed_next.as<uint4>());
    }
    std::swap(ctx->esdf_dist, ctx->esdf_dist_next);
    std::swap(ctx->esdf_packed, ctx->esdf_packed_next);
    // k_esdf_match has read the retained keys (stream order) before they are replaced
    CG_CUDA(ctx->esdf_keys.reserve(n * sizeof(uint64_t)));
    CG_CUDA(ctx->esdf_index.reserve(n * 3 * sizeof(int32_t)));
    CG_CUDA(cudaMemcpyAsync(ctx->esdf_keys.p, keys, n * sizeof(uint64_t), cudaMemcpyDeviceToDevice, s));
    ctx->own_launches += 1;
    k_unpack_idx<<<grid_for(n, 256), 256, 0, s>>>(ctx->esdf_keys.as<uint64_t>(),
                                                  static_cast<uint32_t>(n),
                                                  ctx->esdf_index.as<int32_t>());
  }
  // the sweeps read the layer's hash and these keys; the slots stay sort_blocks' (this call only)
  keys = ctx->esdf_keys.as<uint64_t>();
  uint64_t sweeps = 0, passes = 0;
  if (n_region) {
    const unsigned grid = std::min<unsigned>(n_region, static_cast<unsigned>(ctx->num_sms) * 16u);
    ctx->own_launches += 1;
    k_esdf_init<<<grid, kEsdfThreads, 0, s>>>(L->v, slots, region_list, n_region, P,
                                              ctx->esdf_dist.as<float>(), ctx->esdf_fixed.as<uint32_t>(),
                                              slot_to_b, ctx->esdf_dirty.as<uint8_t>(), nullptr);
    rc = run_sweeps(ctx, L, keys, n, P, region, &sweeps, &passes, "cg_layer_esdf_update");
    if (rc) return rc;
    ctx->own_launches += 1;
    k_esdf_finish<<<grid, kEsdfThreads, 0, s>>>(L->v, keys, slots, region_list, n_region, P,
                                                ctx->esdf_dist.as<float>(), ctx->esdf_fixed.as<uint32_t>(),
                                                slot_to_b, ctx->esdf_packed.as<uint32_t>());
    CG_CUDA(cudaStreamSynchronize(s));
  }
  CG_CUDA(cudaGetLastError());
  if (stats) {
    stats->blocks = n;
    stats->observed_voxels = h_counters[0];
    stats->fixed_voxels = h_counters[1];
    stats->sweeps = sweeps;
    stats->block_passes = passes;
  }
  if (ust) {
    ust->blocks_changed = h_ucount[kUcChanged];
    ust->blocks_removed = h_ucount[kUcRemoved];
    ust->blocks_region = n_region;
  }
  return retain(ctx, L, cfg, n);
}

int32_t cg_esdf_fetch(cg_context* ctx, size_t capacity_blocks, int32_t* block_idx, float* distance,
                      uint32_t* packed, size_t* num_blocks_out) {
  if (!ctx) return CG_ERR_INVALID_ARG;
  CG_CUDA(cudaSetDevice(ctx->device));
  const size_t n = ctx->esdf_blocks;
  if (num_blocks_out) *num_blocks_out = n;
  if (!block_idx && !distance && !packed) return CG_OK;
  if (capacity_blocks < n) {
    set_error("cg_esdf_fetch: capacity %zu < %zu blocks", capacity_blocks, n);
    return CG_ERR_INVALID_ARG;
  }
  if (n == 0) return CG_OK;
  cudaStream_t s = ctx->stream;
  if (block_idx)
    CG_CUDA(cudaMemcpyAsync(block_idx, ctx->esdf_index.p, n * 3 * sizeof(int32_t),
                            cudaMemcpyDeviceToHost, s));
  if (distance)
    CG_CUDA(cudaMemcpyAsync(distance, ctx->esdf_dist.p, n * kVoxelsPerBlock * sizeof(float),
                            cudaMemcpyDeviceToHost, s));
  if (packed)
    CG_CUDA(cudaMemcpyAsync(packed, ctx->esdf_packed.p, n * kVoxelsPerBlock * sizeof(uint32_t),
                            cudaMemcpyDeviceToHost, s));
  CG_CUDA(cudaStreamSynchronize(s));
  return CG_OK;
}

int32_t cg_esdf_free_points(cg_context* ctx, float min_distance, size_t capacity_points,
                            float* xyzi, size_t* num_points_out) {
  if (!ctx) return CG_ERR_INVALID_ARG;
  CG_CUDA(cudaSetDevice(ctx->device));
  const size_t n = ctx->esdf_blocks;
  if (num_points_out) *num_points_out = 0;
  if (n == 0) return CG_OK;
  if (n > (0xFFFFFFFFull / kVoxelsPerBlock)) {  // the per-block ranges are 32-bit
    set_error("cg_esdf_free_points: %zu blocks hold more than 2^32 voxels", n);
    return CG_ERR_UNSUPPORTED;
  }
  cudaStream_t s = ctx->stream;
  ctx->mc_kind = kMeshReused;
  CG_CUDA(ctx->mc_counts.reserve(2 * (n + 1) * sizeof(uint32_t)));
  uint32_t* counts = ctx->mc_counts.as<uint32_t>();
  uint32_t* begin = counts + (n + 1);
  ctx->mc_blocks = 0;  // the marching-cubes result kept in these buffers is gone
  ctx->mc_total = 0;
  size_t tmp = 0;
  CG_CUDA(cub::DeviceScan::ExclusiveSum(nullptr, tmp, counts, begin, static_cast<int>(n + 1), s));
  CG_CUDA(ctx->cub_tmp.reserve(tmp));
  const unsigned grid = static_cast<unsigned>(std::min<size_t>(n, static_cast<size_t>(ctx->num_sms) * 16));
  const uint64_t* keys = ctx->esdf_keys.as<uint64_t>();
  CG_CUDA(cudaMemsetAsync(counts + n, 0, sizeof(uint32_t), s));
  ctx->own_launches += 1;
  k_esdf_free<false><<<grid, kEsdfThreads, 0, s>>>(keys, static_cast<uint32_t>(n),
                                                   ctx->esdf_dist.as<float>(),
                                                   ctx->esdf_packed.as<uint32_t>(), min_distance,
                                                   ctx->esdf_voxel_size, ctx->esdf_block_size, counts,
                                                   nullptr, nullptr);
  CG_CUDA(cub::DeviceScan::ExclusiveSum(ctx->cub_tmp.p, tmp, counts, begin, static_cast<int>(n + 1), s));
  uint32_t total = 0;
  CG_CUDA(cudaMemcpyAsync(&total, begin + n, sizeof(uint32_t), cudaMemcpyDeviceToHost, s));
  CG_CUDA(cudaStreamSynchronize(s));
  if (num_points_out) *num_points_out = total;
  if (!xyzi || total == 0) return CG_OK;
  if (capacity_points < total) {
    set_error("cg_esdf_free_points: capacity %zu < %u points", capacity_points, total);
    return CG_ERR_INVALID_ARG;
  }
  CG_CUDA(ctx->mc_vertices.reserve(static_cast<size_t>(total) * sizeof(float4)));
  ctx->own_launches += 1;
  k_esdf_free<true><<<grid, kEsdfThreads, 0, s>>>(keys, static_cast<uint32_t>(n),
                                                  ctx->esdf_dist.as<float>(),
                                                  ctx->esdf_packed.as<uint32_t>(), min_distance,
                                                  ctx->esdf_voxel_size, ctx->esdf_block_size, counts,
                                                  begin, ctx->mc_vertices.as<float4>());
  CG_CUDA(cudaMemcpyAsync(xyzi, ctx->mc_vertices.p, static_cast<size_t>(total) * sizeof(float4),
                          cudaMemcpyDeviceToHost, s));
  CG_CUDA(cudaStreamSynchronize(s));
  CG_CUDA(cudaGetLastError());
  return CG_OK;
}

}  // extern "C"
