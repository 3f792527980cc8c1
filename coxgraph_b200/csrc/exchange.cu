// exchange.cu — multi-GPU plumbing for the global merge (SURVEY.md §8e).
//
// Submaps are sharded over ranks; every rank projects its submaps into a *partial* global layer.
// A global block is owned by rank cg_block_owner(idx).  cg_layer_pack_by_owner serialises a
// partial layer into fixed-size records grouped by owner (the host exchanges them with one
// all-to-all), and cg_layer_merge_packed folds received records into the owner's layer with the
// 2-argument voxblox::mergeLayerAintoLayerB semantics (Block::mergeBlock / mergeVoxelAIntoVoxelB,
// R10; reference call site of that overload: coxgraph/src/server/submap_collection.cpp:31-33).
// Records of the same block are applied in record order, so concatenating the buffers in
// ascending source-rank order gives a deterministic result.
#include <cub/cub.cuh>

#include <vector>

#include "cg_internal.cuh"

namespace cg {

struct PackedHeader {
  int32_t x, y, z;
  uint32_t flags;
};
static_assert(sizeof(PackedHeader) == 16, "record header");
constexpr size_t kRecordWords = CG_PACKED_BLOCK_BYTES / 4;

__global__ void k_owner_keys(const uint64_t* sorted_keys, int n, uint32_t nranks, uint32_t* owners,
                             unsigned long long* counts) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  const uint32_t o = owner_pick(sorted_keys[i], nranks);
  owners[i] = o;
  atomicAdd(&counts[o], 1ull);
}

__global__ void k_pack_records(LayerView L, const uint32_t* order, const uint32_t* slots_sorted,
                               int n, uint32_t* out) {
  const int b = blockIdx.x;
  if (b >= n) return;
  const int slot = slots_sorted[order[b]];
  uint32_t* rec = out + static_cast<size_t>(b) * kRecordWords;
  if (threadIdx.x == 0) {
    int x, y, z;
    unpack_block_key(L.block_keys[slot], x, y, z);
    rec[0] = static_cast<uint32_t>(x);
    rec[1] = static_cast<uint32_t>(y);
    rec[2] = static_cast<uint32_t>(z);
    rec[3] = (L.has_data[slot] ? 1u : 0u) | (L.updated[slot] ? 2u : 0u);
  }
  const uint4* src = reinterpret_cast<const uint4*>(L.dist_plane(slot));
  uint4* dst = reinterpret_cast<uint4*>(rec + 4);
  for (int i = threadIdx.x; i < 3 * kVoxelsPerBlock / 4; i += blockDim.x) dst[i] = src[i];
}

__global__ void k_record_keys(const uint32_t* recs, int n, uint64_t* keys, uint32_t* idx,
                              int32_t* err) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  const uint32_t* rec = recs + static_cast<size_t>(i) * kRecordWords;
  const int x = static_cast<int>(rec[0]), y = static_cast<int>(rec[1]), z = static_cast<int>(rec[2]);
  constexpr int lim = kVoxIdxOffset / kVps;
  idx[i] = i;
  if (x < -lim || x >= lim || y < -lim || y >= lim || z < -lim || z >= lim) {
    atomicOr(err, kErrOutOfRange);
    keys[i] = kEmptyKey;
    return;
  }
  keys[i] = pack_block_key(x, y, z);
}

// one CTA per distinct destination block: fold its records in record order
__global__ void k_merge_records(LayerView B, const uint32_t* recs, const uint64_t* keys,
                                const uint32_t* idx, int n) {
  const int i = blockIdx.x;
  if (i >= n) return;
  const uint64_t key = keys[i];
  if (key == kEmptyKey || (i > 0 && keys[i - 1] == key)) return;
  __shared__ int s_slot;
  if (threadIdx.x == 0) {
    const int e = B.insert_entry(key);
    s_slot = B.hash_vals[e];
  }
  __syncthreads();
  const int slot = s_slot;
  if (slot < 0) return;
  float* dp = B.dist_plane(slot);
  float* wp = B.weight_plane(slot);
  uint32_t* cp = B.color_plane(slot);
  for (int j = i; j < n && keys[j] == key; ++j) {
    const uint32_t* rec = recs + static_cast<size_t>(idx[j]) * kRecordWords;
    if (!(rec[3] & 1u)) continue;  // Block::mergeBlock: source without data is skipped
    const uint32_t* sd = rec + 4;
    const uint32_t* sw = sd + kVoxelsPerBlock;
    const uint32_t* sc = sw + kVoxelsPerBlock;
    for (int v = threadIdx.x; v < kVoxelsPerBlock; v += blockDim.x) {
      VoxelState b{dp[v], wp[v], cp[v]};
      merge_voxel(__uint_as_float(sd[v]), __uint_as_float(sw[v]), sc[v], b);
      dp[v] = b.d;
      wp[v] = b.w;
      cp[v] = b.c;
    }
    if (threadIdx.x == 0) {
      B.has_data[slot] = 1;
      B.updated[slot] = 1;
    }
  }
}

}  // namespace cg

using namespace cg;

extern "C" {

int32_t cg_block_owner(int32_t bx, int32_t by, int32_t bz, int32_t nranks) {
  if (nranks <= 0) return -1;
  return static_cast<int32_t>(owner_pick(pack_block_key(bx, by, bz), static_cast<uint32_t>(nranks)));
}

int32_t cg_layer_pack_by_owner(const cg_layer* L, int32_t nranks, void* d_packed, size_t capacity,
                               uint64_t* counts_out) {
  if (!L || nranks <= 0 || nranks > 4096 || !counts_out) return CG_ERR_INVALID_ARG;
  cg_context* ctx = L->ctx;
  cudaStream_t s = ctx->stream;
  CG_CUDA(cudaSetDevice(ctx->device));
  const int n = static_cast<int>(L->num_blocks);
  for (int r = 0; r < nranks; ++r) counts_out[r] = 0;
  if (n == 0) return CG_OK;
  if (!d_packed || capacity < static_cast<size_t>(n)) {
    set_error("cg_layer_pack_by_owner: capacity %zu < %d blocks", capacity, n);
    return CG_ERR_INVALID_ARG;
  }
  // 1. blocks sorted by (z,y,x) key  2. stable sort by owner  3. gather records
  CG_CUDA(ctx->key_a.reserve(n * sizeof(uint64_t)));
  CG_CUDA(ctx->key_b.reserve(n * sizeof(uint64_t)));
  CG_CUDA(ctx->val_a.reserve(n * sizeof(uint32_t)));
  CG_CUDA(ctx->val_b.reserve(n * sizeof(uint32_t)));
  CG_CUDA(ctx->flags.reserve(n * sizeof(uint32_t)));
  CG_CUDA(ctx->scan.reserve(n * sizeof(uint32_t)));
  const size_t counts_off = ((2 * n * sizeof(uint32_t) + 7) / 8) * 8;
  CG_CUDA(ctx->stage_b.reserve(counts_off + nranks * sizeof(unsigned long long)));
  uint32_t* iota = ctx->val_a.as<uint32_t>();
  uint32_t* slots_sorted = ctx->val_b.as<uint32_t>();
  k_iota<<<grid_for(n, 256), 256, 0, s>>>(iota, n);
  size_t tmp1 = 0, tmp2 = 0;
  cub::DeviceRadixSort::SortPairs(nullptr, tmp1, L->v.block_keys, ctx->key_b.as<uint64_t>(), iota,
                                  slots_sorted, n, 0, 63, s);
  cub::DeviceRadixSort::SortPairs(nullptr, tmp2, ctx->flags.as<uint32_t>(),
                                  ctx->scan.as<uint32_t>(), iota, iota, n, 0, 12, s);
  CG_CUDA(ctx->cub_tmp.reserve(std::max(tmp1, tmp2)));
  CG_CUDA(cub::DeviceRadixSort::SortPairs(ctx->cub_tmp.p, tmp1, L->v.block_keys,
                                          ctx->key_b.as<uint64_t>(), iota, slots_sorted, n, 0, 63,
                                          s));
  uint32_t* owners = ctx->flags.as<uint32_t>();
  uint32_t* owners_sorted = ctx->scan.as<uint32_t>();
  uint32_t* pos_in = ctx->stage_b.as<uint32_t>();
  uint32_t* order = pos_in + n;
  unsigned long long* d_counts =
      reinterpret_cast<unsigned long long*>(reinterpret_cast<char*>(ctx->stage_b.p) + counts_off);
  CG_CUDA(cudaMemsetAsync(d_counts, 0, nranks * sizeof(unsigned long long), s));
  k_owner_keys<<<grid_for(n, 256), 256, 0, s>>>(ctx->key_b.as<uint64_t>(), n,
                                                static_cast<uint32_t>(nranks), owners, d_counts);
  k_iota<<<grid_for(n, 256), 256, 0, s>>>(pos_in, n);
  CG_CUDA(cub::DeviceRadixSort::SortPairs(ctx->cub_tmp.p, tmp2, owners, owners_sorted, pos_in,
                                          order, n, 0, 12, s));
  k_pack_records<<<n, 256, 0, s>>>(L->v, order, slots_sorted, n, static_cast<uint32_t*>(d_packed));
  std::vector<unsigned long long> h(nranks);
  CG_CUDA(cudaMemcpyAsync(h.data(), d_counts, nranks * sizeof(unsigned long long),
                          cudaMemcpyDeviceToHost, s));
  CG_CUDA(cudaStreamSynchronize(s));
  CG_CUDA(cudaGetLastError());
  for (int r = 0; r < nranks; ++r) counts_out[r] = h[r];
  return CG_OK;
}

int32_t cg_layer_merge_packed(cg_layer* L, const void* d_packed, size_t num_blocks) {
  if (!L || (num_blocks && !d_packed) || num_blocks > 0x7FFFFFFF) return CG_ERR_INVALID_ARG;
  if (num_blocks == 0) return CG_OK;
  cg_context* ctx = L->ctx;
  cudaStream_t s = ctx->stream;
  CG_CUDA(cudaSetDevice(ctx->device));
  const int n = static_cast<int>(num_blocks);
  CG_CUDA(ctx->key_a.reserve(n * sizeof(uint64_t)));
  CG_CUDA(ctx->key_b.reserve(n * sizeof(uint64_t)));
  CG_CUDA(ctx->val_a.reserve(n * sizeof(uint32_t)));
  CG_CUDA(ctx->val_b.reserve(n * sizeof(uint32_t)));
  const uint32_t* recs = static_cast<const uint32_t*>(d_packed);
  k_record_keys<<<grid_for(n, 256), 256, 0, s>>>(recs, n, ctx->key_a.as<uint64_t>(),
                                                 ctx->val_a.as<uint32_t>(), L->v.err);
  size_t tmp = 0;
  cub::DeviceRadixSort::SortPairs(nullptr, tmp, ctx->key_a.as<uint64_t>(),
                                  ctx->key_b.as<uint64_t>(), ctx->val_a.as<uint32_t>(),
                                  ctx->val_b.as<uint32_t>(), n, 0, 64, s);
  CG_CUDA(ctx->cub_tmp.reserve(tmp));
  CG_CUDA(cub::DeviceRadixSort::SortPairs(ctx->cub_tmp.p, tmp, ctx->key_a.as<uint64_t>(),
                                          ctx->key_b.as<uint64_t>(), ctx->val_a.as<uint32_t>(),
                                          ctx->val_b.as<uint32_t>(), n, 0, 64, s));
  k_merge_records<<<n, 256, 0, s>>>(L->v, recs, ctx->key_b.as<uint64_t>(),
                                    ctx->val_b.as<uint32_t>(), n);
  return finish_call(L, nullptr);
}

}  // extern "C"
