// merge.cu — submap -> global TSDF resampling and merge.
//
// Replaces voxblox::mergeLayerAintoLayerB(layer_A, T_B_A, layer_B) = transformLayer +
// Interpolator<TsdfVoxel> + Block::mergeBlock (R7-R10 of SURVEY.md §8a); reference call sites
// coxgraph/src/client/map_server.cpp:67-69 and, through cblox getProjectedMap(),
// coxgraph/src/server/visualizer/server_visualizer.cpp:123-126.
//
//   k_mark_candidates   forward pass: every source block marks the output blocks its bounding
//                       sphere can reach (deduplicated in a scratch hash set)
//   k_resample_merge    one CTA per candidate output block: inverse-transform each voxel centre,
//                       8-tap trilinear gather (nearest fallback) from the source layer, and —
//                       only if any voxel succeeded — claim / find the destination block and fold
//                       the 4096 resampled voxels into it (mergeVoxelAIntoVoxelB).  The temporary
//                       transformed layer of the reference never exists in memory.
#include <cub/cub.cuh>
#include <stdlib.h>
#include <string.h>

#include <vector>

#include <algorithm>
#include <cmath>

#include "cg_internal.cuh"

namespace cg {

constexpr int kTab = 4;  // cached neighbourhood of source block slots: kTab^3

// transformLayer's forward pass for one source block (`key`, blocks of block_size_in): visit(k)
// for every destination block k (blocks of block_size_out) the block's bounding sphere can reach
// under T_B_A, one grid sample at a time (a block may come more than once); a sample outside the
// key range raises kErrOutOfRange instead
template <class Visit>
__device__ __forceinline__ void forward_pass(uint64_t key, float block_size_in, const Xform& T_B_A,
                                             float block_size_out, int32_t* err, Visit visit) {
  int bx, by, bz;
  unpack_block_key(key, bx, by, bz);
  const V3 c_in = V3{center_coord(bx, block_size_in), center_coord(by, block_size_in),
                     center_coord(bz, block_size_in)};
  const V3 c = apply(T_B_A, c_in);
  const float kDiag = 1.7320508075688772f;  // kUnitCubeDiagonalLength
  const float offset = kDiag * block_size_in * 0.5f;
  const float inv_out = 1.0f / block_size_out;
  constexpr int lim = kVoxIdxOffset / kVps;
  for (float x = c.x - offset; x < c.x + offset; x += block_size_out)
    for (float y = c.y - offset; y < c.y + offset; y += block_size_out)
      for (float z = c.z - offset; z < c.z + offset; z += block_size_out) {
        const int ix = grid_index(x, inv_out), iy = grid_index(y, inv_out),
                  iz = grid_index(z, inv_out);
        if (ix < -lim || ix >= lim || iy < -lim || iy >= lim || iz < -lim || iz >= lim) {
          atomicOr(err, kErrOutOfRange);
          continue;
        }
        visit(pack_block_key(ix, iy, iz));
      }
}

__global__ void k_mark_candidates(LayerView A, int num_a, Xform T_B_A, float block_size_out,
                                  KeySet set, uint64_t* list, CallCounters* counters, int32_t* err) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= num_a) return;
  forward_pass(A.block_keys[i], A.block_size, T_B_A, block_size_out, err, [&](uint64_t key) {
    bool inserted;
    set.insert(key, &inserted);
    if (inserted) list[atomicAdd(&counters->candidates, 1ull)] = key;
  });
}

struct SlotTable {
  int ax, ay, az;          // anchor block index
  int slot[kTab * kTab * kTab];
};

__device__ __forceinline__ int lookup_block(const LayerView& A, const SlotTable& tab, int bx, int by,
                                            int bz) {
  const unsigned dx = bx - tab.ax, dy = by - tab.ay, dz = bz - tab.az;
  if (dx < kTab && dy < kTab && dz < kTab) return tab.slot[dx + kTab * (dy + kTab * dz)];
  return A.find_slot(pack_block_key(bx, by, bz));
}

// 8x8 table of the SPIE PM159 trilinear formulation used by voxblox's Interpolator, applied as
// q . (M . data) with rows and the dot product accumulated left to right.
__device__ __forceinline__ float interp_member(const float q[8], const float d[8]) {
  float acc = q[0] * d[0];
  acc = acc + q[1] * (-d[0] + d[4]);
  acc = acc + q[2] * (-d[0] + d[2]);
  acc = acc + q[3] * (-d[0] + d[1]);
  acc = acc + q[4] * (((d[0] + -d[2]) + -d[4]) + d[6]);
  acc = acc + q[5] * (((d[0] + -d[1]) + -d[2]) + d[3]);
  acc = acc + q[6] * (((d[0] + -d[1]) + -d[4]) + d[5]);
  acc = acc + q[7] * (((((((-d[0] + d[1]) + d[2]) + -d[3]) + d[4]) + -d[5]) + -d[6]) + d[7]);
  return acc;
}
// Same value, fewer instructions where the eight taps agree (carved free space: every distance is
// +truncation, every colour the default): all differences of the table are then exactly 0, so
// q . (M . data) = 1 * d0 + q1 * 0 + ... = d0 bit for bit.  (A zero d0 takes the long way: the sign
// of a zero result depends on the signs of q.)
__device__ __forceinline__ float interp_member_fast(const float q[8], const float d[8]) {
  bool same = true;
#pragma unroll
  for (int i = 1; i < 8; ++i) same = same && (d[i] == d[0]);
  if (same && d[0] != 0.0f) return d[0];
  return interp_member(q, d);
}
__device__ __forceinline__ uint32_t trunc_u8(float v) {
  if (!(v > 0.0f)) return 0u;
  if (v >= 255.0f) return 255u;
  return static_cast<uint32_t>(static_cast<int>(v));
}

// Interpolator<TsdfVoxel>::getVoxel(pos, voxel, true) then (.., false); returns success and
// leaves in `out` what the reference's temporary voxel would hold.
__device__ __forceinline__ bool resample_voxel(const LayerView& A, const SlotTable& tab, V3 p,
                                               VoxelState& out) {
  out.d = 0.0f;
  out.w = 0.0f;
  out.c = kDefaultColor;
  int b[3] = {grid_index(p.x, A.block_size_inv), grid_index(p.y, A.block_size_inv),
              grid_index(p.z, A.block_size_inv)};
  const int slot0 = lookup_block(A, tab, b[0], b[1], b[2]);
  if (slot0 < 0) return false;  // neither trilinear nor nearest can succeed
  const V3 org = V3{static_cast<float>(b[0]) * A.block_size, static_cast<float>(b[1]) * A.block_size,
                    static_cast<float>(b[2]) * A.block_size};
  const V3 rel = p - org;
  const int v0[3] = {grid_index(rel.x, A.voxel_size_inv), grid_index(rel.y, A.voxel_size_inv),
                     grid_index(rel.z, A.voxel_size_inv)};
  // ---- trilinear (R8).  All eight taps are addressed first and their loads issued together
  // (weights, then distances and colours): two memory round trips per voxel instead of one per
  // tap — the gather is latency-bound, not bandwidth-bound.
  {
    int v[3] = {v0[0], v0[1], v0[2]};
    const V3 vc = org + V3{center_coord(v[0], A.voxel_size), center_coord(v[1], A.voxel_size),
                           center_coord(v[2], A.voxel_size)};
    const float off[3] = {p.x - vc.x, p.y - vc.y, p.z - vc.z};
    bool moved = false;
#pragma unroll
    for (int a = 0; a < 3; ++a) {
      if (off[a] < 0.0f) {
        v[a]--;
        if (v[a] < 0) {
          b[a]--;
          v[a] += kVps;
          moved = true;
        }
      }
    }
    int base_slot = slot0;
    if (moved) base_slot = lookup_block(A, tab, b[0], b[1], b[2]);
    bool ok = base_slot >= 0;
    const float* tap[8];  // distance plane address of every tap (weight / colour at fixed offsets)
    // Tap addresses.  Common case (every base index in [0, 15]): a tap leaves the base block only
    // on axes where the base index is 15, so at most the 7 upper neighbour blocks are looked up —
    // none at all for most voxels — and the offsets come from two values per axis.
    const bool common = static_cast<unsigned>(v[0]) < kVps && static_cast<unsigned>(v[1]) < kVps &&
                        static_cast<unsigned>(v[2]) < kVps;
    if (ok && common) {
      const bool cx = v[0] == kVps - 1, cy = v[1] == kVps - 1, cz = v[2] == kVps - 1;
      const int s000 = base_slot;
      int s100 = -1, s010 = -1, s001 = -1, s110 = -1, s101 = -1, s011 = -1, s111 = -1;
      if (cx) s100 = lookup_block(A, tab, b[0] + 1, b[1], b[2]);
      if (cy) s010 = lookup_block(A, tab, b[0], b[1] + 1, b[2]);
      if (cz) s001 = lookup_block(A, tab, b[0], b[1], b[2] + 1);
      if (cx && cy) s110 = lookup_block(A, tab, b[0] + 1, b[1] + 1, b[2]);
      if (cx && cz) s101 = lookup_block(A, tab, b[0] + 1, b[1], b[2] + 1);
      if (cy && cz) s011 = lookup_block(A, tab, b[0], b[1] + 1, b[2] + 1);
      if (cx && cy && cz) s111 = lookup_block(A, tab, b[0] + 1, b[1] + 1, b[2] + 1);
      ok = !((cx && s100 < 0) || (cy && s010 < 0) || (cz && s001 < 0) || (cx && cy && s110 < 0) ||
             (cx && cz && s101 < 0) || (cy && cz && s011 < 0) || (cx && cy && cz && s111 < 0));
      const int xo[2] = {v[0], cx ? 0 : v[0] + 1};
      const int yo[2] = {kVps * v[1], cy ? 0 : kVps * (v[1] + 1)};
      const int zo[2] = {kVps * kVps * v[2], cz ? 0 : kVps * kVps * (v[2] + 1)};
#pragma unroll
      for (int i = 0; i < 8; ++i) {
        const int tx = (i >> 2) & 1, ty = (i >> 1) & 1, tz = i & 1;  // compile-time after unrolling
        const bool kx = tx && cx, ky = ty && cy, kz = tz && cz;
        const int slot = kz ? (ky ? (kx ? s111 : s011) : (kx ? s101 : s001))
                            : (ky ? (kx ? s110 : s010) : (kx ? s100 : s000));
        tap[i] = A.dist_plane(slot < 0 ? 0 : slot) + (xo[tx] + yo[ty] + zo[tz]);
      }
    } else if (ok) {
      // a base index of -1 or 16 left by the epsilon of the grid index: the general walk
#pragma unroll
      for (int i = 0; i < 8; ++i) {
        int nv[3] = {v[0] + ((i >> 2) & 1), v[1] + ((i >> 1) & 1), v[2] + (i & 1)};
        int nb[3] = {b[0], b[1], b[2]};
        int slot = base_slot;
        if (nv[0] >= kVps || nv[1] >= kVps || nv[2] >= kVps) {
#pragma unroll
          for (int a = 0; a < 3; ++a)
            if (nv[a] >= kVps) {
              nb[a]++;
              nv[a] -= kVps;
            }
          slot = lookup_block(A, tab, nb[0], nb[1], nb[2]);
          if (slot < 0) ok = false;
        }
        // a voxel index of -1 left by the epsilon of the grid index (see the oracle's
        // interp_trilinear): inside the block's array upstream's linear index is a definite voxel;
        // outside it (undefined behaviour upstream) the trilinear attempt fails
        int lin = nv[0] + kVps * (nv[1] + kVps * nv[2]);
        if (lin < 0 || lin >= kVoxelsPerBlock) {
          ok = false;
          lin = 0;
        }
        tap[i] = A.dist_plane(slot < 0 ? 0 : slot) + lin;
      }
    }
    if (ok) {
      float ww[8];
#pragma unroll
      for (int i = 0; i < 8; ++i) ww[i] = tap[i][kVoxelsPerBlock];
#pragma unroll
      for (int i = 0; i < 8; ++i) ok = ok && (ww[i] > kEps);  // utils::isObservedVoxel
      if (ok) {
        float dd[8];
        uint32_t cc[8];
#pragma unroll
        for (int i = 0; i < 8; ++i) {
          dd[i] = tap[i][0];
          cc[i] = __float_as_uint(tap[i][2 * kVoxelsPerBlock]);
        }
        // offset inside the cell of tap 0 (always inside base block b / voxel v)
        const V3 no = V3{static_cast<float>(b[0]) * A.block_size,
                         static_cast<float>(b[1]) * A.block_size,
                         static_cast<float>(b[2]) * A.block_size};
        const V3 vpos = no + V3{center_coord(v[0], A.voxel_size), center_coord(v[1], A.voxel_size),
                                center_coord(v[2], A.voxel_size)};
        const V3 o = (p - vpos) * A.voxel_size_inv;
        const float q[8] = {1.0f, o.x, o.y, o.z, o.x * o.y, o.y * o.z, o.z * o.x, o.x * o.y * o.z};
        out.d = interp_member_fast(q, dd);
        out.w = interp_member_fast(q, ww);
        bool same_colour = true;
#pragma unroll
        for (int i = 1; i < 8; ++i) same_colour = same_colour && (cc[i] == cc[0]);
        uint32_t rgba = cc[0];  // eight equal colours interpolate to themselves, channel by channel
        if (!same_colour) {
          float ch[8];
          rgba = 0;
#pragma unroll
          for (int s = 0; s < 4; ++s) {
#pragma unroll
            for (int i = 0; i < 8; ++i) ch[i] = static_cast<float>((cc[i] >> (8 * s)) & 255u);
            rgba |= trunc_u8(interp_member(q, ch)) << (8 * s);
          }
        }
        out.c = rgba;
        return true;
      }
    }
  }
  // ---- nearest (R9): clamped voxel index in the block containing p
  const int nx = max(min(v0[0], kVps - 1), 0), ny = max(min(v0[1], kVps - 1), 0),
            nz = max(min(v0[2], kVps - 1), 0);
  const int lin = nx + kVps * (ny + kVps * nz);
  out.d = A.dist_plane(slot0)[lin];
  out.w = A.weight_plane(slot0)[lin];
  out.c = A.color_plane(slot0)[lin];
  return out.w > kEps;
}

constexpr int kMergeThreads = 512;
constexpr int kVoxPerThread = kVoxelsPerBlock / kMergeThreads;

// dynamic shared memory of k_resample_merge / k_project_batch: one resampled block, planar
struct ResampleTile {
  float d[kVoxelsPerBlock];
  float w[kVoxelsPerBlock];
  uint32_t c[kVoxelsPerBlock];
  SlotTable tab;
};

// Resamples destination block `key` of B from A (R8 / R9; T_A_B: B's frame -> A's) into t; every
// thread of the CTA calls it after a barrier that ends the previous use of t.  Returns, on every
// thread, whether any voxel carried data (transformLayer keeps only such blocks).
__device__ __forceinline__ bool resample_block(const LayerView& A, const LayerView& B,
                                               const Xform& T_A_B, uint64_t key, ResampleTile& t) {
  int bx, by, bz;
  unpack_block_key(key, bx, by, bz);
  const V3 org_out = V3{static_cast<float>(bx) * B.block_size, static_cast<float>(by) * B.block_size,
                        static_cast<float>(bz) * B.block_size};
  // the source blocks around the destination block's reach
  if (threadIdx.x < kTab * kTab * kTab) {
    const V3 ctr = V3{center_coord(bx, B.block_size), center_coord(by, B.block_size),
                      center_coord(bz, B.block_size)};
    const V3 pc = apply(T_A_B, ctr);
    const float reach = 0.8660254f * B.block_size + A.voxel_size;
    const int ax = __float2int_rd((pc.x - reach) * A.block_size_inv);
    const int ay = __float2int_rd((pc.y - reach) * A.block_size_inv);
    const int az = __float2int_rd((pc.z - reach) * A.block_size_inv);
    const int i = threadIdx.x;
    const int dx = i % kTab, dy = (i / kTab) % kTab, dz = i / (kTab * kTab);
    t.tab.slot[i] = A.find_slot(pack_block_key(ax + dx, ay + dy, az + dz));
    if (i == 0) {
      t.tab.ax = ax;
      t.tab.ay = ay;
      t.tab.az = az;
    }
  }
  __syncthreads();
  bool any = false;
#pragma unroll 1
  for (int j = 0; j < kVoxPerThread; ++j) {
    const int lin = threadIdx.x + j * kMergeThreads;
    const int vx = lin & 15, vy = (lin >> 4) & 15, vz = lin >> 8;
    const V3 center_out =
        org_out + V3{center_coord(vx, B.voxel_size), center_coord(vy, B.voxel_size),
                     center_coord(vz, B.voxel_size)};
    const V3 p = apply(T_A_B, center_out);
    VoxelState v;
    any |= resample_voxel(A, t.tab, p, v);
    t.d[lin] = v.d;
    t.w[lin] = v.w;
    t.c[lin] = v.c;
  }
  return __syncthreads_or(any ? 1 : 0) != 0;
}

__global__ void __launch_bounds__(kMergeThreads)
k_resample_merge(LayerView A, LayerView B, Xform T_A_B, const uint64_t* __restrict__ cand,
                 CallCounters* counters) {
  extern __shared__ __align__(16) unsigned char smem_raw[];
  ResampleTile& t = *reinterpret_cast<ResampleTile*>(smem_raw);
  __shared__ int s_slot;
  const unsigned long long num_cand = counters->candidates;
  for (unsigned long long c = blockIdx.x; c < num_cand; c += gridDim.x) {
    __syncthreads();  // previous iteration done with t / s_slot
    if (!resample_block(A, B, T_A_B, cand[c], t)) continue;  // dropped: nothing merged
    if (threadIdx.x == 0) {
      const int e = B.insert_entry(cand[c]);
      s_slot = B.hash_vals[e];  // written by this thread or by an earlier kernel
      atomicAdd(&counters->blocks_out, 1ull);
      if (s_slot >= 0) {
        B.has_data[s_slot] = 1;
        B.updated[s_slot] = 1;
      }
    }
    __syncthreads();
    const int slot = s_slot;
    if (slot < 0) continue;
    float* dp = B.dist_plane(slot);
    float* wp = B.weight_plane(slot);
    uint32_t* cp = B.color_plane(slot);
#pragma unroll
    for (int j = 0; j < kVoxPerThread; ++j) {
      const int lin = threadIdx.x + j * kMergeThreads;
      VoxelState b{dp[lin], wp[lin], cp[lin]};
      merge_voxel(t.d[lin], t.w[lin], t.c[lin], b);
      dp[lin] = b.d;
      wp[lin] = b.w;
      cp[lin] = b.c;
    }
  }
}

__global__ void k_reset_merge_counters(CallCounters* c) {
  c->candidates = 0;
  c->blocks_out = 0;
}

// transformLayer's forward pass marks at most this many destination blocks for `blocks` source
// blocks: per axis the grid x in [c - r, c + r) step block_size_out with r = sqrt(3)/2 block_size_in
// has at most floor(sqrt(3) block_in / block_out) + 2 samples
static size_t mark_bound(const cg_layer* A, const cg_layer* G, size_t blocks) {
  const double per_axis = std::floor(1.7320508075688772 * A->v.block_size / G->v.block_size) + 2.0;
  return blocks * static_cast<size_t>(per_axis * per_axis * per_axis);
}

static int32_t enqueue_merge(const cg_layer* A, const float T_B_A[7], cg_layer* B) {
  cg_context* ctx = B->ctx;
  cudaStream_t s = ctx->stream;
  const size_t nA = static_cast<size_t>(A->num_blocks);
  if (nA == 0) return CG_OK;
  // candidate set / list sized from the forward pass's own bound (a coarse source layer merged
  // into a fine one marks more than 27 destination blocks per source block)
  const size_t cand_bound = mark_bound(A, B, nA);
  const size_t cap = key_set_capacity(cand_bound, 1024);
  CG_CUDA(ctx->cand_keys.reserve(cap * sizeof(uint64_t)));
  CG_CUDA(ctx->cand_list.reserve(cand_bound * sizeof(uint64_t)));
  const Xform T = make_xform(T_B_A);
  {
    StageScope sc(ctx, kStageMergeMark, 2);
    CG_CUDA(cudaMemsetAsync(ctx->cand_keys.p, 0xFF, cap * sizeof(uint64_t), s));
    k_reset_merge_counters<<<1, 1, 0, s>>>(ctx->d_counters);
    k_mark_candidates<<<grid_for(nA, 128), 128, 0, s>>>(
        A->v, static_cast<int>(nA), T, B->v.block_size,
        KeySet{ctx->cand_keys.as<unsigned long long>(), static_cast<uint32_t>(cap - 1)},
        ctx->cand_list.as<uint64_t>(), ctx->d_counters, B->v.err);
  }
  const Xform Ti = inverse_xform_host(T);
  const unsigned grid = static_cast<unsigned>(
      std::min<size_t>(cand_bound, static_cast<size_t>(ctx->num_sms) * 4));
  constexpr size_t smem = sizeof(ResampleTile);
  CG_CUDA(allow_dynamic_smem<k_resample_merge>(ctx->device, smem));
  {
    StageScope sc(ctx, kStageMergeResample, 1);
    k_resample_merge<<<grid, kMergeThreads, smem, s>>>(A->v, B->v, Ti,
                                                       ctx->cand_list.as<uint64_t>(),
                                                       ctx->d_counters);
  }
  CG_CUDA(cudaGetLastError());
  return CG_OK;
}

// ------------------------------------------------------------------ batched projection
// cblox getProjectedMap() merges every submap into one layer.  Doing that submap by submap leaves
// the GPU idle (a 5 cm submap has ~100 blocks), so up to 64 submaps go through the three kernels
// below together:
//   k_mark_batch      transformLayer's forward pass for all source blocks of the batch; a scratch
//                     hash map destination block -> 64-bit mask of the submaps that may reach it
//   (scan)            candidate (block, submap) pairs numbered by a prefix sum of the mask
//                     population counts
//   k_list_candidates the explicit (destination block, submap, rank) list
//   k_project_batch   one CTA per candidate: resamples the block (R8 / R9) into shared memory and,
//                     if it carries data, claims the destination block (bit-exact block set) and
//                     folds it in (R10) when its turn comes — candidates of one destination block
//                     fold in ascending submap order, the order of the reference's loop, so the
//                     result is bit-identical to merging the submaps one after the other.
struct BatchSubmap {
  LayerView A;
  Xform T_B_A, T_A_B;
  uint32_t first_block;  // prefix sum of the source block counts
  uint32_t num_blocks;
};
constexpr int kBatchMax = 64;

// `filter_keys` (optional): a key set of filter_mask + 1 entries; the destination blocks outside it
// are not marked (incremental re-projection).  `map_mask` may be null: plain set insertion.
__global__ void k_mark_batch(const BatchSubmap* __restrict__ desc, int n, uint32_t total_blocks,
                             float block_size_out, KeySet map, unsigned long long* map_mask,
                             int32_t* err, const unsigned long long* __restrict__ filter_keys,
                             uint32_t filter_mask) {
  const KeyLookup filter{filter_keys, filter_mask};
  const uint32_t g = blockIdx.x * blockDim.x + threadIdx.x;
  if (g >= total_blocks) return;
  int lo = 0, hi = n;  // desc[lo].first_block <= g
  while (hi - lo > 1) {
    const int mid = (lo + hi) >> 1;
    if (desc[mid].first_block <= g) lo = mid; else hi = mid;
  }
  const BatchSubmap& d = desc[lo];
  forward_pass(d.A.block_keys[g - d.first_block], d.A.block_size, d.T_B_A, block_size_out, err,
               [&](uint64_t key) {
                 if (filter.keys && !filter.contains(key)) return;
                 const int e = map.insert(key);
                 if (map_mask && e >= 0) atomicOr(&map_mask[e], 1ull << lo);
               });
}

// Candidates are listed rank-major: first the lowest-numbered submap of every destination block,
// then the second, ... so that the candidates of one block are handed out far apart in time and a
// candidate rarely has to wait for its predecessor (block-major order made ~12 CTAs resample the
// same block side by side and then queue up for the fold).  rank_count[k] = number of blocks with
// more than k candidates; the position inside a rank comes from an atomic cursor — the list order
// inside a rank is arbitrary, the result is not: the fold order per block is fixed by the ranks.
struct BatchCand {
  uint32_t entry;     // scratch map entry = destination block
  uint32_t sub_rank;  // submap | rank << 8
};
struct RankTable {
  uint32_t count[kBatchMax];
  uint32_t cursor[kBatchMax];
  uint32_t total;
};
__global__ void k_rank_hist(const unsigned long long* __restrict__ map_mask, uint32_t cap,
                            RankTable* table) {
  __shared__ uint32_t s_cnt[kBatchMax];
  if (threadIdx.x < kBatchMax) s_cnt[threadIdx.x] = 0;
  __syncthreads();
  const uint32_t h = blockIdx.x * blockDim.x + threadIdx.x;
  const int p = h < cap ? __popcll(map_mask[h]) : 0;
  for (int k = 0; k < p; ++k) atomicAdd(&s_cnt[k], 1u);
  __syncthreads();
  if (threadIdx.x < kBatchMax && s_cnt[threadIdx.x]) atomicAdd(&table->count[threadIdx.x], s_cnt[threadIdx.x]);
}
__global__ void k_list_candidates(const unsigned long long* __restrict__ map_mask, uint32_t cap,
                                  RankTable* table, BatchCand* __restrict__ list,
                                  CallCounters* counters) {
  __shared__ uint32_t s_base[kBatchMax + 1];
  if (threadIdx.x == 0) {
    uint32_t run = 0;
    for (int k = 0; k < kBatchMax; ++k) {
      s_base[k] = run;
      run += table->count[k];
    }
    s_base[kBatchMax] = run;
    if (blockIdx.x == 0) {
      table->total = run;
      atomicAdd(&counters->candidates, 1ull * run);
    }
  }
  __syncthreads();
  const uint32_t h = blockIdx.x * blockDim.x + threadIdx.x;
  if (h >= cap) return;
  unsigned long long m = map_mask[h];
  for (uint32_t k = 0; m; ++k, m &= m - 1) {
    const uint32_t pos = s_base[k] + atomicAdd(&table->cursor[k], 1u);
    list[pos] = BatchCand{h, static_cast<uint32_t>(__ffsll(static_cast<long long>(m)) - 1) | (k << 8)};
  }
}

// One CTA per candidate, handed out in ascending order by an atomic counter.  The resampled block
// (R8 / R9) stays in shared memory; if it carries data the CTA waits until the lower-ranked
// candidates of the same destination block are done, claims the block (bit-exact block set: only
// candidates with data claim) and folds its 4096 voxels in (R10).  Ranks follow the submap order,
// so the result is bit-identical to merging the submaps one after the other, and nothing but the
// destination block itself (L2-resident) is written.  A waiting CTA only waits on candidates with
// a smaller number; those were handed out earlier to CTAs that are running, so the smallest
// unfinished candidate never waits: no deadlock whatever the grid size or residency.
__global__ void __launch_bounds__(kMergeThreads)
k_project_batch(const BatchSubmap* __restrict__ desc, LayerView B,
                const unsigned long long* __restrict__ map_keys, const BatchCand* __restrict__ list,
                const RankTable* __restrict__ table, unsigned long long* done,
                uint32_t* work_counter, CallCounters* counters) {
  extern __shared__ __align__(16) unsigned char smem_raw[];
  ResampleTile& t = *reinterpret_cast<ResampleTile*>(smem_raw);
  __shared__ uint32_t s_cand;
  __shared__ int s_slot;
  const uint32_t num_cand = table->total;
  for (;;) {
    __syncthreads();  // previous iteration done with the shared state
    if (threadIdx.x == 0) s_cand = atomicAdd(work_counter, 1u);
    __syncthreads();
    const uint32_t c = s_cand;
    if (c >= num_cand) break;
    const BatchCand cd = list[c];
    const uint32_t rank = cd.sub_rank >> 8;
    const BatchSubmap& d = desc[cd.sub_rank & 0xFFu];
    const unsigned long long key = map_keys[cd.entry];
    const bool has_data = resample_block(d.A, B, d.T_A_B, key, t);
    unsigned long long* turn = done + cd.entry;
    if (!has_data) {  // dropped from its transformed layer: nothing merged, nobody waits for it
      if (threadIdx.x == 0) atomicOr(turn, 1ull << rank);
      continue;
    }
    if (threadIdx.x == 0) {
      const unsigned long long need = (1ull << rank) - 1ull;
      while ((*reinterpret_cast<volatile unsigned long long*>(turn) & need) != need) __nanosleep(64);
      __threadfence();  // acquire: the earlier folds (and the block claim) are visible
      const int e = B.insert_entry(key);
      const int slot = *reinterpret_cast<volatile int32_t*>(B.hash_vals + e);
      s_slot = slot;
      atomicAdd(&counters->blocks_out, 1ull);
      if (slot >= 0) {
        B.has_data[slot] = 1;
        B.updated[slot] = 1;
      }
    }
    __syncthreads();
    const int slot = s_slot;
    if (slot >= 0) {
      // the block may have been written by another SM a moment ago: bypass L1 both ways
      float* dp = B.dist_plane(slot);
      float* wp = B.weight_plane(slot);
      uint32_t* cp = B.color_plane(slot);
      VoxelState st[kVoxPerThread];
#pragma unroll
      for (int j = 0; j < kVoxPerThread; ++j) {
        const int lin = threadIdx.x + j * kMergeThreads;
        st[j] = VoxelState{__ldcg(dp + lin), __ldcg(wp + lin), __ldcg(cp + lin)};
      }
#pragma unroll
      for (int j = 0; j < kVoxPerThread; ++j) {
        const int lin = threadIdx.x + j * kMergeThreads;
        merge_voxel(t.d[lin], t.w[lin], t.c[lin], st[j]);
        __stcg(dp + lin, st[j].d);
        __stcg(wp + lin, st[j].w);
        __stcg(cp + lin, st[j].c);
      }
      __threadfence();  // release: every thread's stores before the turn is passed on
    }
    __syncthreads();
    if (threadIdx.x == 0) atomicOr(turn, 1ull << rank);
  }
}

__global__ void k_copy_desc(uint32_t* __restrict__ dst, const uint32_t* __restrict__ src, size_t n) {
  const size_t i = blockIdx.x * static_cast<size_t>(blockDim.x) + threadIdx.x;
  if (i < n) dst[i] = src[i];
}

// submaps [i0, i1) as one batch (descriptors already on the device); everything is enqueued on the
// context's stream, nothing is read back
static int32_t project_batch(const cg_layer* const* submaps, const BatchSubmap* h_desc,
                             const BatchSubmap* d_desc, size_t i0, size_t i1, cg_layer* G,
                             KeyLookup filter = KeyLookup{}) {
  cg_context* ctx = G->ctx;
  cudaStream_t s = ctx->stream;
  const int n = static_cast<int>(i1 - i0);
  uint32_t total = 0;
  size_t cand_bound = 0;  // transformLayer marks at most this many destination blocks
  for (int k = 0; k < n; ++k) {
    const cg_layer* A = submaps[i0 + k];
    total += h_desc[i0 + k].num_blocks;
    cand_bound += mark_bound(A, G, h_desc[i0 + k].num_blocks);
  }
  if (total == 0) return CG_OK;
  const size_t cap = key_set_capacity(cand_bound, 4096);
  CG_CUDA(ctx->cand_keys.reserve(cap * sizeof(uint64_t)));
  // masks, then the per-entry "done" masks of the fused fold, then the rank table (one memset
  // clears all)
  const size_t scratch_bytes = 2 * cap * sizeof(unsigned long long) + sizeof(RankTable);
  CG_CUDA(ctx->cand_list.reserve(scratch_bytes));
  CG_CUDA(ctx->merge_cands.reserve(cand_bound * sizeof(BatchCand)));
  unsigned long long* masks = ctx->cand_list.as<unsigned long long>();
  unsigned long long* done = masks + cap;
  RankTable* table = reinterpret_cast<RankTable*>(done + cap);
  {
    StageScope sc(ctx, kStageMergeMark, 3);
    CG_CUDA(cudaMemsetAsync(ctx->cand_keys.p, 0xFF, cap * sizeof(uint64_t), s));
    CG_CUDA(cudaMemsetAsync(masks, 0, scratch_bytes, s));
    CG_CUDA(cudaMemsetAsync(ctx->d_work_counter, 0, sizeof(uint32_t), s));
    k_mark_batch<<<grid_for(total, 128), 128, 0, s>>>(
        d_desc + i0, n, total, G->v.block_size,
        KeySet{ctx->cand_keys.as<unsigned long long>(), static_cast<uint32_t>(cap - 1)}, masks,
        G->v.err, filter.keys, filter.mask);
    k_rank_hist<<<grid_for(cap, 256), 256, 0, s>>>(masks, static_cast<uint32_t>(cap), table);
    k_list_candidates<<<grid_for(cap, 256), 256, 0, s>>>(masks, static_cast<uint32_t>(cap), table,
                                                         ctx->merge_cands.as<BatchCand>(),
                                                         ctx->d_counters);
  }
  constexpr size_t smem = sizeof(ResampleTile);
  CG_CUDA(allow_dynamic_smem<k_project_batch>(ctx->device, smem));
  {
    StageScope sc(ctx, kStageMergeResample, 1);
    const unsigned grid = static_cast<unsigned>(
        std::min<size_t>(cand_bound, static_cast<size_t>(ctx->num_sms) * 2));
    k_project_batch<<<grid, kMergeThreads, smem, s>>>(
        d_desc + i0, G->v, ctx->cand_keys.as<unsigned long long>(), ctx->merge_cands.as<BatchCand>(), table,
        done, ctx->d_work_counter, ctx->d_counters);
  }
  CG_CUDA(cudaGetLastError());
  return CG_OK;
}

// ------------------------------------------------------------------ incremental re-projection
// (SURVEY §8f N1)  The server rebuilds the whole global map whenever poses change
// (coxgraph/include/coxgraph/server/coxgraph_server.h:275-283 -> server_visualizer.cpp:123-126).
// Here only the destination blocks a moved submap can reach — under its old or its new pose — are
// rebuilt: they are reset, every submap (moved or not) whose forward pass marks them is resampled
// and folded into them in submap order, and those left without data are removed.  Every other
// block holds exactly what a full rebuild would produce, so the result is bit-identical to
// clearing the layer and projecting all submaps again.
// Lists the slots of the dirty blocks G holds (counts[0] of them; counts[1]: dirty keys).  With
// `out_keys` (cg_reproject_submaps_sharded) the keys of those blocks are also appended there
// (cursor *out_count, at most out_cap stored); `slots` / `counts` may then be null.
__global__ void k_dirty_slots(LayerView G, const uint64_t* __restrict__ dirty_keys, uint32_t cap,
                              uint32_t* __restrict__ slots, uint32_t* __restrict__ counts,
                              uint64_t* __restrict__ out_keys, uint32_t* out_count, uint32_t out_cap) {
  const uint32_t h = blockIdx.x * blockDim.x + threadIdx.x;
  if (h >= cap) return;
  const uint64_t key = dirty_keys[h];
  if (key == kEmptyKey) return;
  if (counts) atomicAdd(&counts[1], 1u);  // dirty destination blocks
  const int slot = G.find_slot(key);
  if (slot < 0) return;
  if (slots) slots[atomicAdd(&counts[0], 1u)] = static_cast<uint32_t>(slot);
  if (out_keys) {
    const uint32_t at = atomicAdd(out_count, 1u);
    if (at < out_cap) out_keys[at] = key;
  }
}
__global__ void __launch_bounds__(256)
k_reset_blocks(LayerView G, const uint32_t* __restrict__ slots, const uint32_t* __restrict__ counts) {
  const uint32_t n = counts[0];
  for (uint32_t i = blockIdx.x; i < n; i += gridDim.x) {
    const uint32_t slot = slots[i];
    uint4* p = reinterpret_cast<uint4*>(G.dist_plane(slot));
    for (int w = threadIdx.x; w < 3 * kVoxelsPerBlock / 4; w += blockDim.x) {
      const uint32_t v = w >= 2 * kVoxelsPerBlock / 4 ? kDefaultColor : 0u;
      p[w] = make_uint4(v, v, v, v);
    }
    if (threadIdx.x == 0) G.has_data[slot] = 0;
  }
}
__global__ void k_flag_dead(LayerView G, const uint32_t* __restrict__ slots,
                            const uint32_t* __restrict__ counts, uint8_t* __restrict__ remove) {
  const uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i < counts[0] && !G.has_data[slots[i]]) remove[slots[i]] = 1;
}

static void fill_desc(BatchSubmap& d, const cg_layer* A, const float* pose, uint32_t first) {
  d.A = A->v;
  d.T_B_A = make_xform(pose);
  d.T_A_B = inverse_xform_host(d.T_B_A);
  d.first_block = first;
  d.num_blocks = static_cast<uint32_t>(A->num_blocks);
}

// Puts `count` descriptors into ctx->batch_desc (pinned, device-mapped staging + a copy kernel)
// and resets the merge counters of the call behind them.  The host writes ctx->h_tables only while
// no queued kernel reads it: every call that stages through it (the projections here and
// integrate_front.cu's upload_frame_tables) ends, on success, in finish_call's stream
// synchronise.  An error return may leave the copy queued; the CUDA errors that end a call early
// are sticky, so no later call gets as far as writing the table.
static int32_t upload_descs(cg_context* ctx, const BatchSubmap* descs, size_t count) {
  const size_t desc_bytes = count * sizeof(BatchSubmap);
  if (desc_bytes > ctx->h_tables_cap) {
    if (ctx->h_tables) cudaFreeHost(ctx->h_tables);
    ctx->h_tables = nullptr;
    ctx->h_tables_cap = 0;
    CG_CUDA(cudaHostAlloc(&ctx->h_tables, desc_bytes * 2, cudaHostAllocMapped));
    ctx->h_tables_cap = desc_bytes * 2;
  }
  memcpy(ctx->h_tables, descs, desc_bytes);
  void* d_alias = nullptr;
  CG_CUDA(cudaHostGetDevicePointer(&d_alias, ctx->h_tables, 0));
  CG_CUDA(ctx->batch_desc.reserve(desc_bytes));
  ctx->own_launches += 2;
  k_copy_desc<<<grid_for(desc_bytes / 4, 256), 256, 0, ctx->stream>>>(
      ctx->batch_desc.as<uint32_t>(), static_cast<const uint32_t*>(d_alias), desc_bytes / 4);
  k_reset_merge_counters<<<1, 1, 0, ctx->stream>>>(ctx->d_counters);
  return CG_OK;
}

static bool pose_changed(const float* a, const float* b, float eps_t, float eps_rot) {
  if (memcmp(a, b, 7 * sizeof(float)) == 0) return false;
  const double dx = double(a[4]) - b[4], dy = double(a[5]) - b[5], dz = double(a[6]) - b[6];
  if (std::sqrt(dx * dx + dy * dy + dz * dz) > eps_t) return true;
  double dot = std::fabs(double(a[0]) * b[0] + double(a[1]) * b[1] + double(a[2]) * b[2] +
                         double(a[3]) * b[3]);
  const double na = std::sqrt(double(a[0]) * a[0] + double(a[1]) * a[1] + double(a[2]) * a[2] +
                              double(a[3]) * a[3]);
  const double nb = std::sqrt(double(b[0]) * b[0] + double(b[1]) * b[1] + double(b[2]) * b[2] +
                              double(b[3]) * b[3]);
  if (na > 0 && nb > 0) dot /= na * nb;
  return 2.0 * std::acos(std::min(1.0, dot)) > eps_rot;
}

// dirty blocks / blocks of the map above which the re-projections rebuild the whole map
// (CG_REPROJECT_FULL_FRACTION overrides it; the tests use 2 to force the block-by-block path)
double full_rebuild_fraction() {
  const char* e = getenv("CG_REPROJECT_FULL_FRACTION");
  return (e && *e) ? atof(e) : 0.3;
}

int32_t reset_dirty_blocks(cg_layer* G, const uint64_t* dirty_keys, uint32_t cap, uint32_t* slots,
                           uint32_t* counts) {
  cg_context* ctx = G->ctx;
  cudaStream_t s = ctx->stream;
  CG_CUDA(cudaMemsetAsync(counts, 0, 2 * sizeof(uint32_t), s));
  StageScope sc(ctx, kStageMergeMark, 2);
  k_dirty_slots<<<grid_for(cap, 256), 256, 0, s>>>(G->v, dirty_keys, cap, slots, counts, nullptr,
                                                   nullptr, 0);
  k_reset_blocks<<<ctx->num_sms * 8, 256, 0, s>>>(G->v, slots, counts);
  CG_CUDA(cudaGetLastError());
  return CG_OK;
}

int32_t remove_dead_blocks(cg_layer* G, const uint32_t* slots, const uint32_t* counts,
                           uint32_t listed, uint64_t* removed) {
  cg_context* ctx = G->ctx;
  cudaStream_t s = ctx->stream;
  CG_CUDA(ctx->flags.reserve(static_cast<size_t>(G->num_blocks) + 1));
  CG_CUDA(cudaMemsetAsync(ctx->flags.p, 0, static_cast<size_t>(G->num_blocks), s));
  ctx->own_launches += 1;
  k_flag_dead<<<grid_for(listed, 256), 256, 0, s>>>(G->v, slots, counts, ctx->flags.as<uint8_t>());
  const int32_t rc = remove_flagged_blocks(G, ctx->flags.as<uint8_t>(), removed);
  if (rc) return rc;
  return finish_call(G, nullptr);
}

// cg_reproject_submaps, and the local step of cg_reproject_submaps_sharded: submaps [0, num_known)
// are re-projected (moved ones under poses_new), submaps [num_known, n) are new and projected under
// poses_new behind them.  The dirty set is every destination block a moved submap marks under
// either pose and every block a new submap marks.  With `dirty`, the keys of the dirty blocks G
// holds before the call and those it holds after it are appended to dirty->keys (a key may appear
// twice).
int32_t reproject_local(const cg_layer* const* submaps, size_t n, size_t num_known,
                        const float* poses_old, const float* poses_new, float eps_translation,
                        float eps_rotation, cg_layer* G, uint8_t* changed_out,
                        cg_reproject_stats* stats, const DirtyKeysOut* dirty, const char* who) {
  cg_context* ctx = G->ctx;
  cudaStream_t s = ctx->stream;
  if (stats) memset(stats, 0, sizeof(*stats));
  std::vector<size_t> moved;
  for (size_t i = 0; i < n; ++i) {
    const cg_layer* A = submaps[i];
    if (!A || A == G || A->ctx != ctx) {
      set_error("%s: submap %zu invalid", who, i);
      return CG_ERR_INVALID_ARG;
    }
    const bool ch = i >= num_known ||
                    pose_changed(poses_old + 7 * i, poses_new + 7 * i, eps_translation, eps_rotation);
    if (changed_out) changed_out[i] = ch ? 1 : 0;
    if (ch && i < num_known) moved.push_back(i);
  }
  if (stats) stats->submaps_moved = moved.size();
  if (moved.empty() && num_known == n) return CG_OK;
  // descriptor table: [0, num_known) the known submaps under their effective pose and
  // [num_known, n) the new ones (batch-relative block prefixes, batches start at 0 and at
  // num_known), then every moved submap under its old and under its new pose and every new submap
  // (one prefix over the list)
  const size_t num_new = n - num_known;
  std::vector<BatchSubmap> h(n + 2 * moved.size() + num_new);
  {
    size_t mi = 0;
    const size_t ranges[2][2] = {{0, num_known}, {num_known, n}};
    for (const auto& r : ranges) {
      const size_t end = r[1];
      for (size_t i0 = r[0]; i0 < end; i0 += kBatchMax) {
        uint32_t total = 0;
        for (size_t i = i0; i < std::min(end, i0 + static_cast<size_t>(kBatchMax)); ++i) {
          const bool ch = i >= num_known || (mi < moved.size() && moved[mi] == i);
          if (ch && i < num_known) ++mi;
          fill_desc(h[i], submaps[i], (ch ? poses_new : poses_old) + 7 * i, total);
          total += h[i].num_blocks;
        }
      }
    }
  }
  uint32_t dirty_src = 0;
  size_t dirty_bound = 0;
  for (size_t k = 0; k < moved.size(); ++k) {
    const size_t i = moved[k];
    fill_desc(h[n + 2 * k], submaps[i], poses_old + 7 * i, dirty_src);
    dirty_src += h[n + 2 * k].num_blocks;
    fill_desc(h[n + 2 * k + 1], submaps[i], poses_new + 7 * i, dirty_src);
    dirty_src += h[n + 2 * k + 1].num_blocks;
    dirty_bound += 2 * mark_bound(submaps[i], G, h[n + 2 * k].num_blocks);
  }
  for (size_t i = num_known; i < n; ++i) {
    BatchSubmap& d = h[n + 2 * moved.size() + (i - num_known)];
    fill_desc(d, submaps[i], poses_new + 7 * i, dirty_src);
    dirty_src += d.num_blocks;
    dirty_bound += mark_bound(submaps[i], G, d.num_blocks);
  }
  int32_t urc = upload_descs(ctx, h.data(), h.size());
  if (urc) return urc;
  const BatchSubmap* d_desc = ctx->batch_desc.as<BatchSubmap>();
  uint32_t dirty_total = 0, dirty_existing = 0;
  uint64_t removed = 0;
  if (dirty_src > 0) {
    // the dirty set: destination blocks a moved submap marks under either pose, or a new one marks
    const size_t cap = key_set_capacity(dirty_bound, 4096);
    const size_t g_blocks = static_cast<size_t>(G->num_blocks);
    CG_CUDA(ctx->stage_a.reserve(cap * sizeof(uint64_t)));
    CG_CUDA(ctx->stage_b.reserve((g_blocks + 2) * sizeof(uint32_t)));
    uint32_t* counts = ctx->stage_b.as<uint32_t>();  // [0] dirty blocks present in G, [1] dirty blocks
    uint32_t* slots = counts + 2;
    const KeySet dirty_set{ctx->stage_a.as<unsigned long long>(), static_cast<uint32_t>(cap - 1)};
    const uint64_t* dirty_keys = ctx->stage_a.as<uint64_t>();
    {
      StageScope sc(ctx, kStageMergeMark, 3);
      CG_CUDA(cudaMemsetAsync(ctx->stage_a.p, 0xFF, cap * sizeof(uint64_t), s));
      CG_CUDA(cudaMemsetAsync(counts, 0, 2 * sizeof(uint32_t), s));
      k_mark_batch<<<grid_for(dirty_src, 128), 128, 0, s>>>(
          d_desc + n, static_cast<int>(2 * moved.size() + num_new), dirty_src, G->v.block_size,
          dirty_set, nullptr, G->v.err, nullptr, 0);
      k_dirty_slots<<<grid_for(cap, 256), 256, 0, s>>>(
          G->v, dirty_keys, static_cast<uint32_t>(cap), slots, counts,
          dirty ? dirty->keys : nullptr, dirty ? dirty->count : nullptr, dirty ? dirty->cap : 0);
    }
    // the dirty blocks G holds once the call is done
    auto publish_after = [&]() -> int32_t {
      if (!dirty) return CG_OK;
      ctx->own_launches += 1;
      k_dirty_slots<<<grid_for(cap, 256), 256, 0, s>>>(G->v, dirty_keys, static_cast<uint32_t>(cap),
                                                       nullptr, nullptr, dirty->keys, dirty->count,
                                                       dirty->cap);
      CG_CUDA(cudaGetLastError());
      return CG_OK;
    };
    // When the moved submaps dirty a large part of the map (a corridor map where every block is
    // shared by a few submaps: a tenth of the poses dirties more than half of the blocks),
    // rebuilding the dirty blocks from ALL submaps that reach them plus the block removal costs
    // more than the full rebuild, which gives the same layer by definition: take that instead.
    {
      uint32_t h_dirty[2] = {0, 0};
      CG_CUDA(cudaMemcpyAsync(h_dirty, counts, sizeof(h_dirty), cudaMemcpyDeviceToHost, s));
      CG_CUDA(cudaStreamSynchronize(s));
      if (static_cast<double>(h_dirty[0]) > full_rebuild_fraction() * static_cast<double>(g_blocks)) {
        std::vector<float> eff(7 * n);
        size_t mi = 0;
        for (size_t i = 0; i < n; ++i) {
          const bool ch = i >= num_known || (mi < moved.size() && moved[mi] == i);
          if (ch && i < num_known) ++mi;
          memcpy(&eff[7 * i], (ch ? poses_new : poses_old) + 7 * i, 7 * sizeof(float));
        }
        int32_t rc = cg_layer_clear(G);
        if (rc) return rc;
        cg_merge_stats ms;
        rc = cg_project_submaps(submaps, eff.data(), n, G, &ms);
        if (stats) {
          stats->blocks_dirty = h_dirty[1];
          stats->candidates = ms.blocks_candidate;
          stats->blocks_folded = ms.blocks_out;
          stats->full_rebuild = 1;
        }
        return rc ? rc : publish_after();
      }
    }
    {
      StageScope sc(ctx, kStageMergeMark, 1);
      k_reset_blocks<<<ctx->num_sms * 8, 256, 0, s>>>(G->v, slots, counts);
    }
    // every known submap that reaches a dirty block is folded into it again, in submap order; the
    // new submaps follow as plain batches
    for (size_t i0 = 0; i0 < num_known; i0 += kBatchMax) {
      int32_t rc = project_batch(submaps, h.data(), d_desc, i0,
                                 std::min(num_known, i0 + static_cast<size_t>(kBatchMax)), G,
                                 KeyLookup{dirty_set.keys, dirty_set.mask});
      if (rc) return rc;
    }
    for (size_t i0 = num_known; i0 < n; i0 += kBatchMax) {
      int32_t rc = project_batch(submaps, h.data(), d_desc, i0,
                                 std::min(n, i0 + static_cast<size_t>(kBatchMax)), G);
      if (rc) return rc;
    }
    // dirty blocks that ended up without data leave the layer (a fresh projection would not
    // have allocated them)
    uint32_t h_counts[2] = {0, 0};
    CG_CUDA(cudaMemcpyAsync(h_counts, counts, sizeof(h_counts), cudaMemcpyDeviceToHost, s));
    CG_CUDA(cudaStreamSynchronize(s));
    dirty_existing = h_counts[0];
    dirty_total = h_counts[1];
    if (dirty_existing > 0) {
      // new blocks were claimed behind the old ones: flags cover the current block count
      CallCounters c0;
      int32_t rc = finish_call(G, &c0);
      if (rc) return rc;
      const CallCounters keep = c0;
      rc = remove_dead_blocks(G, slots, counts, dirty_existing, &removed);
      if (rc) return rc;
      if (stats) {
        stats->candidates = keep.candidates;
        stats->blocks_folded = keep.blocks_out;
      }
    }
    const int32_t rc = publish_after();
    if (rc) return rc;
  }
  if (dirty_existing == 0) {
    CallCounters c;
    const int32_t rc = finish_call(G, &c);
    if (rc) return rc;
    if (stats) {
      stats->candidates = c.candidates;
      stats->blocks_folded = c.blocks_out;
    }
  }
  if (stats) {
    stats->blocks_dirty = dirty_total;
    stats->blocks_removed = removed;
  }
  return CG_OK;
}

}  // namespace cg

using namespace cg;

extern "C" {

int32_t cg_merge_layer_into_layer(const cg_layer* A, const float T_B_A[7], cg_layer* B,
                                  cg_merge_stats* stats) {
  if (!A || !B || !T_B_A || A == B || A->ctx != B->ctx) {
    set_error("cg_merge_layer_into_layer: invalid argument (layers must differ and share a context)");
    return CG_ERR_INVALID_ARG;
  }
  CG_CUDA(cudaSetDevice(B->ctx->device));
  int32_t rc = enqueue_merge(A, T_B_A, B);
  if (rc) return rc;
  CallCounters c;
  rc = finish_call(B, &c);
  if (stats) {
    stats->blocks_in = static_cast<uint64_t>(A->num_blocks);
    stats->blocks_candidate = A->num_blocks ? c.candidates : 0;
    stats->blocks_out = A->num_blocks ? c.blocks_out : 0;
  }
  return rc;
}

int32_t cg_project_submaps(const cg_layer* const* submaps, const float* poses, size_t n,
                           cg_layer* G, cg_merge_stats* stats) {
  if (!G || (n && (!submaps || !poses))) return CG_ERR_INVALID_ARG;
  CG_CUDA(cudaSetDevice(G->ctx->device));
  cg_context* ctx = G->ctx;
  if (stats) memset(stats, 0, sizeof(*stats));
  for (size_t i = 0; i < n; ++i) {
    const cg_layer* A = submaps[i];
    if (!A || A == G || A->ctx != ctx) {
      set_error("cg_project_submaps: submap %zu invalid", i);
      return CG_ERR_INVALID_ARG;
    }
  }
  if (n == 0) return finish_call(G, nullptr);
  // descriptors of all submaps go up once
  std::vector<BatchSubmap> h(n);
  uint64_t blocks_in = 0;
  for (size_t i0 = 0; i0 < n; i0 += kBatchMax) {
    uint32_t total = 0;
    for (size_t i = i0; i < std::min(n, i0 + static_cast<size_t>(kBatchMax)); ++i) {
      fill_desc(h[i], submaps[i], poses + 7 * i, total);  // prefix sum inside the submap's batch
      total += h[i].num_blocks;
    }
    blocks_in += total;
  }
  int32_t urc = upload_descs(ctx, h.data(), n);
  if (urc) return urc;
  // batches of up to 64 submaps, in submap order (the mask of a destination block has one bit per
  // submap of the batch)
  for (size_t i0 = 0; i0 < n; i0 += kBatchMax) {
    int32_t rc = project_batch(submaps, h.data(), ctx->batch_desc.as<BatchSubmap>(), i0,
                               std::min(n, i0 + static_cast<size_t>(kBatchMax)), G);
    if (rc) return rc;
  }
  CallCounters c;
  const int32_t rc = finish_call(G, &c);
  if (stats) {
    stats->blocks_in = blocks_in;
    stats->blocks_candidate = c.candidates;
    stats->blocks_out = c.blocks_out;
  }
  return rc;
}

int32_t cg_reproject_submaps(const cg_layer* const* submaps, const float* poses_old,
                             const float* poses_new, size_t n, float eps_translation,
                             float eps_rotation, cg_layer* G, uint8_t* changed_out,
                             cg_reproject_stats* stats) {
  if (!G || (n && (!submaps || !poses_old || !poses_new))) return CG_ERR_INVALID_ARG;
  CG_CUDA(cudaSetDevice(G->ctx->device));
  return reproject_local(submaps, n, n, poses_old, poses_new, eps_translation, eps_rotation, G,
                         changed_out, stats, nullptr, "cg_reproject_submaps");
}

}  // extern "C"
