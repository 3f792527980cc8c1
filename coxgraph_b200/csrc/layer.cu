// layer.cu — context and Layer<TsdfVoxel> replacement: creation, clear, upload, download.
// Boundary: include/coxgraph_b200.h.  Reference data contract: voxblox Layer / Block /
// TsdfVoxel as consumed at coxgraph/include/coxgraph/utils/msg_converter.h:49-50,107-109.
#include <cub/cub.cuh>
#include <stdarg.h>
#include <string.h>
#include <thrust/iterator/counting_iterator.h>

#include <algorithm>
#include <atomic>

#include "cg_internal.cuh"
#include "host_stage.cuh"

namespace cg {

static thread_local char g_err[512] = "";

void set_error(const char* fmt, ...) {
  va_list ap;
  va_start(ap, fmt);
  vsnprintf(g_err, sizeof(g_err), fmt, ap);
  va_end(ap);
}
int32_t cuda_fail(cudaError_t e, const char* what) {
  set_error("CUDA error %d (%s) at %s", static_cast<int>(e), cudaGetErrorString(e), what);
  return CG_ERR_CUDA;
}

const char* stage_name(int s) {
  static const char* names[kNumStages] = {
      "point_keys",    "bundle_sort",  "bundle_scan",      "gather_sorted", "bundle_order",
      "fold_wide",     "fold_bundles", "bundle_rays",      "ray_scan",      "walk_segments",
      "segment_sort",  "block_accumulate", "pair_sort",    "segments",   "visits",   "voxel_update",
      "replay_wide",   "finalize",     "merge_mark",       "merge_resample", "transfer",
      "depth_points"};
  return (s >= 0 && s < kNumStages) ? names[s] : "?";
}

static void drain_events(cg_context* ctx) {
  for (const PendingEvent& pe : ctx->pending) {
    float ms = 0.0f;
    if (cudaEventElapsedTime(&ms, pe.start, pe.stop) == cudaSuccess) ctx->stage_ms[pe.stage] += ms;
    ctx->event_pool.push_back(pe.start);
    ctx->event_pool.push_back(pe.stop);
  }
  ctx->pending.clear();
}

// ------------------------------------------------------------------ kernels
__global__ void k_fill_default(float* pool, size_t first_block, size_t num_blocks) {
  // one block plane triple = 3 * 4096 words; words [8192, 12288) are the colour plane
  const size_t words = num_blocks * (3 * kVoxelsPerBlock);
  uint32_t* p = reinterpret_cast<uint32_t*>(pool + first_block * (3 * kVoxelsPerBlock));
  for (size_t i = (blockIdx.x * static_cast<size_t>(blockDim.x) + threadIdx.x) * 4; i < words;
       i += static_cast<size_t>(gridDim.x) * blockDim.x * 4) {
    const uint32_t in_block = static_cast<uint32_t>(i % (3 * kVoxelsPerBlock));
    const uint32_t val = in_block >= 2 * kVoxelsPerBlock ? kDefaultColor : 0u;
    *reinterpret_cast<uint4*>(p + i) = make_uint4(val, val, val, val);
  }
}

__global__ void k_read_counters(LayerView L, CallCounters* c) {
  int n = *L.num_blocks;
  if (n > L.max_blocks) {
    n = L.max_blocks;
    *L.num_blocks = n;
  }
  c->num_blocks = n;
  c->err = *L.err;
  *L.err = 0;
}

__global__ void k_iota(uint32_t* v, int n) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i < n) v[i] = i;
}

// planar pool block -> voxblox AoS (one CTA per output block)
__global__ void k_gather_aos(LayerView L, const uint32_t* slots, int first, int count,
                             uint32_t* out_words, int32_t* out_idx, uint8_t* out_flags,
                             const uint64_t* sorted_keys) {
  const int b = blockIdx.x;
  if (b >= count) return;
  const int slot = slots[first + b];
  const float* d = L.dist_plane(slot);
  const float* w = L.weight_plane(slot);
  const uint32_t* c = L.color_plane(slot);
  uint32_t* o = out_words + static_cast<size_t>(b) * (3 * kVoxelsPerBlock);
  for (int i = threadIdx.x; i < kVoxelsPerBlock; i += blockDim.x) {
    o[3 * i + 0] = __float_as_uint(d[i]);
    o[3 * i + 1] = __float_as_uint(w[i]);
    o[3 * i + 2] = c[i];
  }
  if (threadIdx.x == 0) {
    int x, y, z;
    unpack_block_key(sorted_keys[first + b], x, y, z);
    if (out_idx) {
      out_idx[3 * b + 0] = x;
      out_idx[3 * b + 1] = y;
      out_idx[3 * b + 2] = z;
    }
    if (out_flags) out_flags[b] = (L.has_data[slot] ? 1 : 0) | (L.updated[slot] ? 2 : 0);
  }
}

// voxblox::Block<TsdfVoxel>::serializeToIntegers: three words per voxel — float bits of the
// distance, float bits of the weight, colour packed a | b << 8 | g << 16 | r << 24
__device__ __forceinline__ uint32_t msg_color(uint32_t rgba) {  // rgba: r | g << 8 | b << 16 | a << 24
  return __byte_perm(rgba, 0, 0x0123);
}
__global__ void k_serialize_blocks(LayerView L, const uint32_t* slots, int count,
                                   uint32_t* out_words, int32_t* out_idx,
                                   const uint64_t* sorted_keys, const uint32_t* order) {
  const int b = blockIdx.x;
  if (b >= count) return;
  const int src = order ? static_cast<int>(order[b]) : b;
  const int slot = slots[src];
  const float* d = L.dist_plane(slot);
  const float* w = L.weight_plane(slot);
  const uint32_t* c = L.color_plane(slot);
  uint32_t* o = out_words + static_cast<size_t>(b) * (3 * kVoxelsPerBlock);
  for (int i = threadIdx.x; i < kVoxelsPerBlock; i += blockDim.x) {
    o[3 * i + 0] = __float_as_uint(d[i]);
    o[3 * i + 1] = __float_as_uint(w[i]);
    o[3 * i + 2] = msg_color(c[i]);
  }
  if (threadIdx.x == 0) {
    int x, y, z;
    unpack_block_key(sorted_keys[src], x, y, z);
    out_idx[3 * b + 0] = x;
    out_idx[3 * b + 1] = y;
    out_idx[3 * b + 2] = z;
  }
}
__global__ void k_compact_blocks(const uint64_t* __restrict__ keys, const uint32_t* __restrict__ slots,
                                 const uint32_t* __restrict__ order, uint32_t n,
                                 uint64_t* __restrict__ keys_out, uint32_t* __restrict__ slots_out) {
  const uint32_t j = blockIdx.x * blockDim.x + threadIdx.x;
  if (j >= n) return;
  keys_out[j] = keys[order[j]];
  slots_out[j] = slots[order[j]];
}
__global__ void k_select_updated(LayerView L, const uint32_t* slots, int n, uint32_t* order,
                                 uint32_t* count) {
  // sorted position i -> kept, in order (single CTA, n is a few thousand blocks at most per call)
  __shared__ uint32_t s_run;
  if (threadIdx.x == 0) s_run = 0;
  __syncthreads();
  for (int i0 = 0; i0 < n; i0 += blockDim.x) {
    const int i = i0 + threadIdx.x;
    const bool keep = i < n && L.updated[slots[i]];
    // ordered compaction: ballot within warps, warp offsets through shared memory
    __shared__ uint32_t s_warp[32];
    const unsigned m = __ballot_sync(0xFFFFFFFFu, keep);
    const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5;
    if (lane == 0) s_warp[wid] = __popc(m);
    __syncthreads();
    uint32_t before = 0;
    for (int k = 0; k < wid; ++k) before += s_warp[k];
    if (keep) order[s_run + before + __popc(m & ((1u << lane) - 1u))] = i;
    __syncthreads();
    if (threadIdx.x == 0) {
      uint32_t tot = 0;
      for (int k = 0; k < static_cast<int>(blockDim.x >> 5); ++k) tot += s_warp[k];
      s_run += tot;
    }
    __syncthreads();
  }
  if (threadIdx.x == 0) *count = s_run;
}
__global__ void k_deserialize_write(LayerView L, const int32_t* entries, const uint32_t* in_words,
                                    int n) {
  const int b = blockIdx.x;
  if (b >= n) return;
  const int e = entries[b];
  if (e < 0) return;
  const int slot = L.hash_vals[e];
  if (slot < 0) return;
  float* d = L.dist_plane(slot);
  float* w = L.weight_plane(slot);
  uint32_t* c = L.color_plane(slot);
  const uint32_t* in = in_words + static_cast<size_t>(b) * (3 * kVoxelsPerBlock);
  for (int i = threadIdx.x; i < kVoxelsPerBlock; i += blockDim.x) {
    d[i] = __uint_as_float(in[3 * i + 0]);
    w[i] = __uint_as_float(in[3 * i + 1]);
    c[i] = msg_color(in[3 * i + 2]);  // the byte reversal is its own inverse
  }
  if (threadIdx.x == 0) {
    L.has_data[slot] = 1;  // Block::deserializeFromIntegers
    L.updated[slot] = 1;
  }
}

// listed block indices -> pool slots (-1: not allocated) and packed keys, for k_gather_aos
__global__ void k_lookup_listed(LayerView L, const int32_t* __restrict__ idx, int n,
                                uint32_t* __restrict__ slots, uint64_t* __restrict__ keys,
                                uint8_t* __restrict__ found) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  const int x = idx[3 * i], y = idx[3 * i + 1], z = idx[3 * i + 2];
  constexpr int lim = kVoxIdxOffset / kVps;
  int slot = -1;
  uint64_t key = 0;
  if (x >= -lim && x < lim && y >= -lim && y < lim && z >= -lim && z < lim) {
    key = pack_block_key(x, y, z);
    slot = L.find_slot(key);
  }
  slots[i] = slot < 0 ? 0u : static_cast<uint32_t>(slot);
  keys[i] = key;
  found[i] = slot >= 0 ? 1 : 0;
}

// probe lengths of the block hash: [0] sum over the allocated blocks, [1] maximum
__global__ void k_probe_lengths(LayerView L, int n, unsigned long long* out) {
  const int slot = blockIdx.x * blockDim.x + threadIdx.x;
  unsigned len = 0;
  if (slot < n) {
    const uint64_t key = L.block_keys[slot];
    uint32_t h = hash_key(key) & L.hash_mask;
    len = 1;
    while (L.hash_keys[h] != key) {
      h = (h + 1) & L.hash_mask;
      ++len;
    }
  }
  const unsigned sum = __reduce_add_sync(0xFFFFFFFFu, len);
  const unsigned mx = __reduce_max_sync(0xFFFFFFFFu, len);
  if ((threadIdx.x & 31) == 0 && sum) {
    atomicAdd(&out[0], static_cast<unsigned long long>(sum));
    atomicMax(&out[1], static_cast<unsigned long long>(mx));
  }
}

__global__ void k_unpack_idx(const uint64_t* sorted_keys, int n, int32_t* out_idx) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  int x, y, z;
  unpack_block_key(sorted_keys[i], x, y, z);
  out_idx[3 * i] = x;
  out_idx[3 * i + 1] = y;
  out_idx[3 * i + 2] = z;
}

__global__ void k_upload_insert(LayerView L, const int32_t* idx, int n, int32_t* entries) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  const int x = idx[3 * i], y = idx[3 * i + 1], z = idx[3 * i + 2];
  constexpr int lim = kVoxIdxOffset / kVps;  // keeps every voxel index inside +-2^19
  if (x < -lim || x >= lim || y < -lim || y >= lim || z < -lim || z >= lim) {
    atomicOr(L.err, kErrOutOfRange);
    entries[i] = -1;
    return;
  }
  entries[i] = L.insert_entry(pack_block_key(x, y, z));
}

__global__ void k_upload_write(LayerView L, const int32_t* entries, const uint32_t* in_words,
                               const uint8_t* flags, int n) {
  const int b = blockIdx.x;
  if (b >= n) return;
  const int e = entries[b];
  if (e < 0) return;
  const int slot = L.hash_vals[e];
  if (slot < 0) return;
  float* d = L.dist_plane(slot);
  float* w = L.weight_plane(slot);
  uint32_t* c = L.color_plane(slot);
  const uint32_t* in = in_words + static_cast<size_t>(b) * (3 * kVoxelsPerBlock);
  for (int i = threadIdx.x; i < kVoxelsPerBlock; i += blockDim.x) {
    d[i] = __uint_as_float(in[3 * i + 0]);
    w[i] = __uint_as_float(in[3 * i + 1]);
    c[i] = in[3 * i + 2];
  }
  if (threadIdx.x == 0) {
    const uint8_t f = flags ? flags[b] : 1;
    L.has_data[slot] = f & 1;
    L.updated[slot] = (f >> 1) & 1;
  }
}

// ------------------------------------------------------------------ block removal
// Layer::removeBlock for a set of blocks: the pool stays dense (claimed slots are [0, num_blocks)),
// so the survivors of the tail fill the holes, the freed tail returns to the default-constructed
// state and the hash is rebuilt from block_keys.
struct HoleSlot {
  const uint8_t* remove;
  uint32_t keep;  // blocks that survive
  __device__ __forceinline__ bool operator()(uint32_t slot) const {
    return slot < keep && remove[slot] != 0;
  }
};
struct FillerSlot {
  const uint8_t* remove;
  uint32_t keep;
  __device__ __forceinline__ bool operator()(uint32_t slot) const {
    return slot >= keep && remove[slot] == 0;
  }
};
__global__ void k_count_flags(const uint8_t* __restrict__ flags, uint32_t n, uint32_t* count) {
  uint32_t c = 0;
  for (uint32_t i = blockIdx.x * blockDim.x + threadIdx.x; i < n; i += gridDim.x * blockDim.x)
    c += flags[i] != 0;
  c = __reduce_add_sync(0xFFFFFFFFu, c);
  if ((threadIdx.x & 31) == 0 && c) atomicAdd(count, c);
}
__global__ void __launch_bounds__(256)
k_move_blocks(LayerView L, const uint32_t* __restrict__ holes, const uint32_t* __restrict__ fillers,
              uint32_t m) {
  for (uint32_t i = blockIdx.x; i < m; i += gridDim.x) {
    const uint32_t dst = holes[i], src = fillers[i];
    const uint4* from = reinterpret_cast<const uint4*>(L.dist_plane(src));
    uint4* to = reinterpret_cast<uint4*>(L.dist_plane(dst));
    for (int w = threadIdx.x; w < 3 * kVoxelsPerBlock / 4; w += blockDim.x) to[w] = from[w];
    if (threadIdx.x == 0) {
      L.block_keys[dst] = L.block_keys[src];
      L.has_data[dst] = L.has_data[src];
      L.updated[dst] = L.updated[src];
    }
  }
}
__global__ void k_rehash(LayerView L, uint32_t n) {
  const uint32_t slot = blockIdx.x * blockDim.x + threadIdx.x;
  if (slot >= n) return;
  const uint64_t key = L.block_keys[slot];
  uint32_t h = hash_key(key) & L.hash_mask;
  for (;;) {
    if (L.hash_keys[h] == kEmptyKey &&
        atomicCAS(reinterpret_cast<unsigned long long*>(&L.hash_keys[h]), kEmptyKey, key) == kEmptyKey) {
      L.hash_vals[h] = static_cast<int32_t>(slot);
      return;
    }
    h = (h + 1) & L.hash_mask;
  }
}
__global__ void k_set_num_blocks(LayerView L, int32_t n) { *L.num_blocks = n; }

int32_t remove_flagged_blocks(cg_layer* L, const uint8_t* d_remove, uint64_t* removed_out) {
  cg_context* ctx = L->ctx;
  cudaStream_t s = ctx->stream;
  const uint32_t n = static_cast<uint32_t>(L->num_blocks);
  if (removed_out) *removed_out = 0;
  if (n == 0) return CG_OK;
  uint32_t* d_cnt = ctx->d_select_count;
  CG_CUDA(cudaMemsetAsync(d_cnt, 0, sizeof(uint32_t), s));
  ctx->own_launches += 1;
  k_count_flags<<<std::min<unsigned>(grid_for(n, 256), ctx->num_sms * 8u), 256, 0, s>>>(d_remove, n,
                                                                                         d_cnt);
  uint32_t r = 0;
  CG_CUDA(cudaMemcpyAsync(&r, d_cnt, sizeof(uint32_t), cudaMemcpyDeviceToHost, s));
  CG_CUDA(cudaStreamSynchronize(s));
  if (r == 0) return CG_OK;
  const uint32_t keep = n - r;
  LayerView& v = L->v;
  if (keep > 0) {
    CG_CUDA(ctx->val_a.reserve(sizeof(uint32_t) * r));
    CG_CUDA(ctx->val_b.reserve(sizeof(uint32_t) * r));
    thrust::counting_iterator<uint32_t> iota(0);
    size_t tmp = 0;
    CG_CUDA(cub::DeviceSelect::If(nullptr, tmp, iota, ctx->val_a.as<uint32_t>(), d_cnt,
                                  static_cast<int>(n), HoleSlot{d_remove, keep}, s));
    CG_CUDA(ctx->cub_tmp.reserve(tmp));
    CG_CUDA(cub::DeviceSelect::If(ctx->cub_tmp.p, tmp, iota, ctx->val_a.as<uint32_t>(), d_cnt,
                                  static_cast<int>(n), HoleSlot{d_remove, keep}, s));
    CG_CUDA(cub::DeviceSelect::If(ctx->cub_tmp.p, tmp, iota, ctx->val_b.as<uint32_t>(), d_cnt,
                                  static_cast<int>(n), FillerSlot{d_remove, keep}, s));
    uint32_t m = 0;  // holes below `keep` == survivors at or above it
    CG_CUDA(cudaMemcpyAsync(&m, d_cnt, sizeof(uint32_t), cudaMemcpyDeviceToHost, s));
    CG_CUDA(cudaStreamSynchronize(s));
    if (m > 0) {
      ctx->own_launches += 1;
      k_move_blocks<<<std::min<unsigned>(m, ctx->num_sms * 8u), 256, 0, s>>>(
          v, ctx->val_a.as<uint32_t>(), ctx->val_b.as<uint32_t>(), m);
    }
  }
  ctx->own_launches += 3;
  k_fill_default<<<ctx->num_sms * 8, 256, 0, s>>>(v.pool, keep, r);
  CG_CUDA(cudaMemsetAsync(v.has_data + keep, 0, r, s));
  CG_CUDA(cudaMemsetAsync(v.updated + keep, 0, r, s));
  CG_CUDA(cudaMemsetAsync(v.hash_keys, 0xFF, L->hash_cap * sizeof(uint64_t), s));
  CG_CUDA(cudaMemsetAsync(v.hash_vals, 0xFF, L->hash_cap * sizeof(int32_t), s));
  if (keep > 0) k_rehash<<<grid_for(keep, 256), 256, 0, s>>>(v, keep);
  k_set_num_blocks<<<1, 1, 0, s>>>(v, static_cast<int32_t>(keep));
  CG_CUDA(cudaGetLastError());
  L->num_blocks = keep;
  if (removed_out) *removed_out = r;
  return CG_OK;
}

__global__ void k_flag_listed(LayerView L, const int32_t* __restrict__ idx, int n,
                              uint8_t* __restrict__ remove) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  const int x = idx[3 * i], y = idx[3 * i + 1], z = idx[3 * i + 2];
  constexpr int lim = kVoxIdxOffset / kVps;
  if (x < -lim || x >= lim || y < -lim || y >= lim || z < -lim || z >= lim) return;
  const int slot = L.find_slot(pack_block_key(x, y, z));
  if (slot >= 0) remove[slot] = 1;
}

cudaError_t init_front_words(FrontBufs& fb) {
  cudaError_t e;
  if ((e = cudaMallocHost(&fb.h_counters, sizeof(CallCounters))) != cudaSuccess) return e;
  if ((e = cudaMalloc(&fb.d_counters, sizeof(CallCounters))) != cudaSuccess) return e;
  if ((e = cudaMemset(fb.d_counters, 0, sizeof(CallCounters))) != cudaSuccess) return e;
  if ((e = cudaMalloc(&fb.d_select_count, sizeof(uint32_t))) != cudaSuccess) return e;
  if ((e = cudaMemset(fb.d_select_count, 0, sizeof(uint32_t))) != cudaSuccess) return e;
  if ((e = cudaMalloc(&fb.d_key_bounds, 6 * sizeof(int))) != cudaSuccess) return e;
  const int init[6] = {0x3FFFFFFF, 0x3FFFFFFF, 0x3FFFFFFF, -0x3FFFFFFF, -0x3FFFFFFF, -0x3FFFFFFF};
  if ((e = cudaMemcpy(fb.d_key_bounds, init, sizeof(init), cudaMemcpyHostToDevice)) != cudaSuccess) return e;
  if ((e = cudaMalloc(&fb.d_class_count, 128 * sizeof(uint32_t))) != cudaSuccess) return e;
  if ((e = cudaMalloc(&fb.d_front_err, sizeof(int32_t))) != cudaSuccess) return e;
  return cudaMemset(fb.d_front_err, 0, sizeof(int32_t));
}
bool side_stream(FrontBufs& fb, cudaStream_t like) {
  if (fb.side) return true;
  int prio = 0;
  if (cudaStreamGetPriority(like, &prio) != cudaSuccess) prio = 0;
  if (cudaStreamCreateWithPriority(&fb.side, cudaStreamNonBlocking, prio) != cudaSuccess ||
      cudaEventCreateWithFlags(&fb.ev_fork, cudaEventDisableTiming) != cudaSuccess ||
      cudaEventCreateWithFlags(&fb.ev_join, cudaEventDisableTiming) != cudaSuccess) {
    cudaGetLastError();
    if (fb.side) cudaStreamDestroy(fb.side);
    if (fb.ev_fork) cudaEventDestroy(fb.ev_fork);
    if (fb.ev_join) cudaEventDestroy(fb.ev_join);
    fb.side = nullptr;
    fb.ev_fork = fb.ev_join = nullptr;
    return false;
  }
  return true;
}

void release_front(FrontBufs& fb) {
  DevBuf* bufs[] = {&fb.poses, &fb.frame_base, &fb.key_a, &fb.key_b, &fb.scan, &fb.cub_tmp, &fb.rays,
                    &fb.ray_count, &fb.ray_offset, &fb.sorted_pts, &fb.scan_partials, &fb.ray_id,
                    &fb.frame_count,
                    &fb.grazing_keys, &fb.grazing_ray_key, &fb.depth_pts, &fb.depth_cols,
                    &fb.depth_counts, &fb.depth_tiles};
  for (DevBuf* b : bufs) b->release();
  if (fb.h_counters) cudaFreeHost(fb.h_counters);
  if (fb.d_counters) cudaFree(fb.d_counters);
  if (fb.d_select_count) cudaFree(fb.d_select_count);
  if (fb.d_key_bounds) cudaFree(fb.d_key_bounds);
  if (fb.d_class_count) cudaFree(fb.d_class_count);
  if (fb.d_front_err) cudaFree(fb.d_front_err);
  if (fb.h_tables) cudaFreeHost(fb.h_tables);
  if (fb.side) cudaStreamDestroy(fb.side);
  if (fb.ev_fork) cudaEventDestroy(fb.ev_fork);
  if (fb.ev_join) cudaEventDestroy(fb.ev_join);
  fb = FrontBufs();
}

int32_t finish_call(cg_layer* layer, CallCounters* out) {
  cg_context* ctx = layer->ctx;
  k_read_counters<<<1, 1, 0, ctx->stream>>>(layer->v, ctx->d_counters);
  CG_CUDA(cudaMemcpyAsync(ctx->h_counters, ctx->d_counters, sizeof(CallCounters),
                          cudaMemcpyDeviceToHost, ctx->stream));
  CG_CUDA(cudaStreamSynchronize(ctx->stream));
  CG_CUDA(cudaGetLastError());
  layer->num_blocks = ctx->h_counters->num_blocks;
  if (out) *out = *ctx->h_counters;
  const int err = ctx->h_counters->err;
  if (err & kErrPoolFull) {
    // the keys that found no slot are still in the hash (value -1): rebuild it from block_keys
    // so that later calls do not find them and silently skip those blocks
    const LayerView& v = layer->v;
    const uint32_t keep = static_cast<uint32_t>(layer->num_blocks);
    cudaMemsetAsync(v.hash_keys, 0xFF, layer->hash_cap * sizeof(uint64_t), ctx->stream);
    cudaMemsetAsync(v.hash_vals, 0xFF, layer->hash_cap * sizeof(int32_t), ctx->stream);
    if (keep > 0) k_rehash<<<grid_for(keep, 256), 256, 0, ctx->stream>>>(v, keep);
    cudaStreamSynchronize(ctx->stream);
    set_error("block pool exhausted (max_blocks = %zu)", layer->max_blocks);
    return CG_ERR_POOL_FULL;
  }
  if (err & kErrOutOfRange) {
    set_error("voxel / block index outside the addressable range");
    return CG_ERR_OUT_OF_RANGE;
  }
  return CG_OK;
}

// sorted (z,y,x) view of the allocated blocks: keys in ctx->key_b, slots in ctx->val_b
int32_t sort_blocks(const cg_layer* layer, const uint64_t** keys, const uint32_t** slots) {
  cg_context* ctx = layer->ctx;
  const int n = static_cast<int>(layer->num_blocks);
  CG_CUDA(ctx->key_b.reserve(sizeof(uint64_t) * n));
  CG_CUDA(ctx->val_a.reserve(sizeof(uint32_t) * n));
  CG_CUDA(ctx->val_b.reserve(sizeof(uint32_t) * n));
  k_iota<<<grid_for(n, 256), 256, 0, ctx->stream>>>(ctx->val_a.as<uint32_t>(), n);
  size_t tmp = 0;
  cub::DeviceRadixSort::SortPairs(nullptr, tmp, layer->v.block_keys, ctx->key_b.as<uint64_t>(),
                                  ctx->val_a.as<uint32_t>(), ctx->val_b.as<uint32_t>(), n, 0, 63,
                                  ctx->stream);
  CG_CUDA(ctx->cub_tmp.reserve(tmp));
  CG_CUDA(cub::DeviceRadixSort::SortPairs(ctx->cub_tmp.p, tmp, layer->v.block_keys,
                                          ctx->key_b.as<uint64_t>(), ctx->val_a.as<uint32_t>(),
                                          ctx->val_b.as<uint32_t>(), n, 0, 63, ctx->stream));
  *keys = ctx->key_b.as<uint64_t>();
  *slots = ctx->val_b.as<uint32_t>();
  return CG_OK;
}

}  // namespace cg

using namespace cg;

extern "C" {

const char* cg_last_error(void) { return g_err; }
const char* cg_version(void) { return "coxgraph_b200 0.1 (sm_100a)"; }

int32_t cg_context_create(int32_t device, void* stream, cg_context** out) {
  if (!out) return CG_ERR_INVALID_ARG;
  *out = nullptr;
  int count = 0;
  cudaError_t e = cudaGetDeviceCount(&count);
  if (e != cudaSuccess || count == 0) {
    set_error("no CUDA device available (%s); this library has no CPU fallback",
              e == cudaSuccess ? "device count is 0" : cudaGetErrorString(e));
    return CG_ERR_CUDA;
  }
  if (device < 0 || device >= count) {
    set_error("device %d out of range (%d devices)", device, count);
    return CG_ERR_INVALID_ARG;
  }
  CG_CUDA(cudaSetDevice(device));
  cg_context* ctx = new cg_context();
  ctx->device = device;
  if (stream) {
    ctx->stream = static_cast<cudaStream_t>(stream);
  } else {
    CG_CUDA(cudaStreamCreateWithFlags(&ctx->stream, cudaStreamNonBlocking));
    ctx->own_stream = true;
  }
  cudaDeviceGetAttribute(&ctx->num_sms, cudaDevAttrMultiProcessorCount, device);
  CG_CUDA(init_front_words(*ctx));
  CG_CUDA(cudaMalloc(&ctx->d_work_counter, sizeof(uint32_t)));
  CG_CUDA(cudaMalloc(&ctx->d_long_counter, sizeof(unsigned long long)));
  CG_CUDA(cudaMalloc(&ctx->d_touch_count, 2 * sizeof(uint32_t)));
  CG_CUDA(cudaMalloc(&ctx->d_walk_counters, 4 * sizeof(uint32_t)));
  CG_CUDA(cudaMemsetAsync(ctx->d_walk_counters, 0, 4 * sizeof(uint32_t), ctx->stream));
  *out = ctx;
  return CG_OK;
}

int32_t cg_context_destroy(cg_context* ctx) {
  if (!ctx) return CG_ERR_INVALID_ARG;
  cudaSetDevice(ctx->device);
  cudaStreamSynchronize(ctx->stream);
  cg_comm_destroy(ctx);
  DevBuf* bufs[] = {&ctx->points, &ctx->colors, &ctx->val_a, &ctx->val_b, &ctx->flags,
                    &ctx->pkey_a, &ctx->pkey_b, &ctx->seg_keys_a, &ctx->seg_keys_b, &ctx->seg_idx_a,
                    &ctx->seg_idx_b, &ctx->seg_recs, &ctx->seg_order, &ctx->seg_bins,
                    &ctx->touch_ord, &ctx->touch_entry, &ctx->touch_acc, &ctx->touch_bits,
                    &ctx->seg_start, &ctx->long_list, &ctx->long_partials, &ctx->visits, &ctx->cand_keys,
                    &ctx->cand_list, &ctx->stage_a, &ctx->stage_b, &ctx->stage_c, &ctx->batch_desc,
                    &ctx->merge_cands, &ctx->mc_counts, &ctx->mc_index, &ctx->mc_vertices,
                    &ctx->mc_normals, &ctx->mc_colors, &ctx->mesh_in, &ctx->mesh_tri,
                    &ctx->mesh_pairs, &ctx->mesh_pts_g, &ctx->mesh_cols_g, &ctx->mesh_pts_c,
                    &ctx->mesh_cols_c, &ctx->mesh_frames, &ctx->esdf_keys, &ctx->esdf_slots,
                    &ctx->esdf_dist, &ctx->esdf_packed, &ctx->esdf_fixed,
                    &ctx->esdf_slot_to_b, &ctx->esdf_dirty, &ctx->esdf_list, &ctx->esdf_index,
                    &ctx->esdf_counters, &ctx->esdf_dist_next, &ctx->esdf_packed_next,
                    &ctx->esdf_old_b, &ctx->esdf_sources, &ctx->esdf_region,
                    &ctx->esdf_region_list, &ctx->weld_keys, &ctx->weld_words, &ctx->weld_out};
  for (DevBuf* b : bufs) b->release();
  drain_events(ctx);
  for (cudaEvent_t e : ctx->event_pool) cudaEventDestroy(e);
  release_front(*ctx);
  for (int i = 0; i < 2; ++i) {
    release_front(ctx->prep[i]);
    if (ctx->prep_done[i]) cudaEventDestroy(ctx->prep_done[i]);
  }
  if (ctx->prep_stream) cudaStreamDestroy(ctx->prep_stream);
  if (ctx->d_touch_count) cudaFree(ctx->d_touch_count);
  if (ctx->d_walk_counters) cudaFree(ctx->d_walk_counters);
  if (ctx->d_work_counter) cudaFree(ctx->d_work_counter);
  if (ctx->d_long_counter) cudaFree(ctx->d_long_counter);
  for (int i = 0; i < 2; ++i) {
    ctx->stage_pts[i].release();
    ctx->stage_cols[i].release();
    if (ctx->stage_ready[i]) cudaEventDestroy(ctx->stage_ready[i]);
  }
  if (ctx->wait_event) cudaEventDestroy(ctx->wait_event);
  cg::destroy_stager(ctx->stager);
  ctx->stager = nullptr;
  if (ctx->copy_stream) cudaStreamDestroy(ctx->copy_stream);
  if (ctx->own_stream) cudaStreamDestroy(ctx->stream);
  delete ctx;
  return CG_OK;
}

int32_t cg_context_set_profiling(cg_context* ctx, int32_t enable) {
  if (!ctx) return CG_ERR_INVALID_ARG;
  ctx->profiling = enable != 0;
  return CG_OK;
}

int32_t cg_context_reset_profile(cg_context* ctx) {
  if (!ctx) return CG_ERR_INVALID_ARG;
  CG_CUDA(cudaStreamSynchronize(ctx->stream));
  drain_events(ctx);
  for (int i = 0; i < kNumStages; ++i) {
    ctx->stage_ms[i] = 0.0;
    ctx->stage_launches[i] = 0;
  }
  return CG_OK;
}

int32_t cg_context_get_profile(cg_context* ctx, cg_stage_profile* out, size_t capacity,
                               size_t* num_out) {
  if (!ctx) return CG_ERR_INVALID_ARG;
  CG_CUDA(cudaStreamSynchronize(ctx->stream));
  drain_events(ctx);
  if (num_out) *num_out = kNumStages;
  for (size_t i = 0; out && i < capacity && i < kNumStages; ++i) {
    snprintf(out[i].name, sizeof(out[i].name), "%s", stage_name(static_cast<int>(i)));
    out[i].ms = ctx->stage_ms[i];
    out[i].launches = ctx->stage_launches[i];
  }
  return CG_OK;
}

uint64_t cg_context_kernel_launches(const cg_context* ctx) { return ctx ? ctx->own_launches : 0; }

int32_t cg_context_synchronize(cg_context* ctx) {
  if (!ctx) return CG_ERR_INVALID_ARG;
  CG_CUDA(cudaStreamSynchronize(ctx->stream));
  return CG_OK;
}

int32_t cg_context_wait_stream(cg_context* ctx, void* producer_stream) {
  if (!ctx) return CG_ERR_INVALID_ARG;
  cudaStream_t ps = static_cast<cudaStream_t>(producer_stream);
  if (ps == ctx->stream) return CG_OK;
  CG_CUDA(cudaSetDevice(ctx->device));
  if (!ctx->wait_event) CG_CUDA(cudaEventCreateWithFlags(&ctx->wait_event, cudaEventDisableTiming));
  CG_CUDA(cudaEventRecord(ctx->wait_event, ps));
  CG_CUDA(cudaStreamWaitEvent(ctx->stream, ctx->wait_event, 0));
  return CG_OK;
}

int32_t cg_layer_create(cg_context* ctx, float voxel_size, int32_t vps, size_t max_blocks,
                        cg_layer** out) {
  if (!ctx || !out || !(voxel_size > 0.0f) || max_blocks == 0 || max_blocks > (1u << 30)) {
    set_error("cg_layer_create: invalid argument");
    return CG_ERR_INVALID_ARG;
  }
  if (vps != kVps) {
    set_error("voxels_per_side must be 16");
    return CG_ERR_UNSUPPORTED;
  }
  *out = nullptr;
  CG_CUDA(cudaSetDevice(ctx->device));
  cg_layer* L = new cg_layer();
  static std::atomic<uint64_t> next_serial{1};
  L->serial = next_serial.fetch_add(1);
  L->ctx = ctx;
  L->max_blocks = max_blocks;
  size_t cap = 1024;
  while (cap < 2 * max_blocks) cap <<= 1;
  L->hash_cap = cap;
  LayerView& v = L->v;
  v.hash_mask = static_cast<uint32_t>(cap - 1);
  v.max_blocks = static_cast<int32_t>(max_blocks);
  v.voxel_size = voxel_size;
  v.voxel_size_inv = 1.0f / voxel_size;
  v.block_size = voxel_size * static_cast<float>(kVps);
  v.block_size_inv = 1.0f / v.block_size;
  cudaError_t e = cudaSuccess;
  auto alloc = [&](void** p, size_t bytes) {
    if (e == cudaSuccess) e = cudaMalloc(p, bytes);
  };
  alloc(reinterpret_cast<void**>(&v.hash_keys), cap * sizeof(uint64_t));
  alloc(reinterpret_cast<void**>(&v.hash_vals), cap * sizeof(int32_t));
  alloc(reinterpret_cast<void**>(&v.block_keys), max_blocks * sizeof(uint64_t));
  alloc(reinterpret_cast<void**>(&v.has_data), max_blocks);
  alloc(reinterpret_cast<void**>(&v.updated), max_blocks);
  alloc(reinterpret_cast<void**>(&v.pool), max_blocks * static_cast<size_t>(CG_BLOCK_BYTES));
  alloc(reinterpret_cast<void**>(&v.num_blocks), sizeof(int32_t));
  alloc(reinterpret_cast<void**>(&v.err), sizeof(int32_t));
  if (e != cudaSuccess) {
    cg_layer_destroy(L);
    return cuda_fail(e, "cg_layer_create allocation");
  }
  cudaStream_t s = ctx->stream;
  CG_CUDA(cudaMemsetAsync(v.hash_keys, 0xFF, cap * sizeof(uint64_t), s));
  CG_CUDA(cudaMemsetAsync(v.hash_vals, 0xFF, cap * sizeof(int32_t), s));
  CG_CUDA(cudaMemsetAsync(v.has_data, 0, max_blocks, s));
  CG_CUDA(cudaMemsetAsync(v.updated, 0, max_blocks, s));
  CG_CUDA(cudaMemsetAsync(v.num_blocks, 0, sizeof(int32_t), s));
  CG_CUDA(cudaMemsetAsync(v.err, 0, sizeof(int32_t), s));
  k_fill_default<<<ctx->num_sms * 8, 256, 0, s>>>(v.pool, 0, max_blocks);
  CG_CUDA(cudaStreamSynchronize(s));
  CG_CUDA(cudaGetLastError());
  *out = L;
  return CG_OK;
}

int32_t cg_layer_destroy(cg_layer* L) {
  if (!L) return CG_ERR_INVALID_ARG;
  cudaSetDevice(L->ctx->device);
  cudaStreamSynchronize(L->ctx->stream);
  LayerView& v = L->v;
  cudaFree(v.hash_keys);
  cudaFree(v.hash_vals);
  cudaFree(v.block_keys);
  cudaFree(v.has_data);
  cudaFree(v.updated);
  cudaFree(v.pool);
  cudaFree(v.num_blocks);
  cudaFree(v.err);
  delete L;
  return CG_OK;
}

int32_t cg_layer_clear(cg_layer* L) {
  if (!L) return CG_ERR_INVALID_ARG;
  cudaStream_t s = L->ctx->stream;
  LayerView& v = L->v;
  CG_CUDA(cudaMemsetAsync(v.hash_keys, 0xFF, L->hash_cap * sizeof(uint64_t), s));
  CG_CUDA(cudaMemsetAsync(v.hash_vals, 0xFF, L->hash_cap * sizeof(int32_t), s));
  if (L->num_blocks > 0) {
    CG_CUDA(cudaMemsetAsync(v.has_data, 0, L->num_blocks, s));
    CG_CUDA(cudaMemsetAsync(v.updated, 0, L->num_blocks, s));
    k_fill_default<<<L->ctx->num_sms * 8, 256, 0, s>>>(v.pool, 0, L->num_blocks);
  }
  CG_CUDA(cudaMemsetAsync(v.num_blocks, 0, sizeof(int32_t), s));
  L->num_blocks = 0;
  // no host synchronisation: everything that touches the layer afterwards is ordered behind these
  // fills on the context's stream, and a round trip to the host costs more than the fills
  CG_CUDA(cudaGetLastError());
  return CG_OK;
}

int32_t cg_layer_remove_blocks(cg_layer* L, size_t n, const int32_t* idx, uint64_t* removed_out) {
  if (!L || (n && !idx)) return CG_ERR_INVALID_ARG;
  if (removed_out) *removed_out = 0;
  if (n == 0 || L->num_blocks == 0) return CG_OK;
  cg_context* ctx = L->ctx;
  cudaStream_t s = ctx->stream;
  CG_CUDA(cudaSetDevice(ctx->device));
  CG_CUDA(ctx->stage_b.reserve(n * 3 * sizeof(int32_t)));
  CG_CUDA(ctx->stage_c.reserve(static_cast<size_t>(L->num_blocks)));
  CG_CUDA(cudaMemcpyAsync(ctx->stage_b.p, idx, n * 3 * sizeof(int32_t), cudaMemcpyHostToDevice, s));
  CG_CUDA(cudaMemsetAsync(ctx->stage_c.p, 0, static_cast<size_t>(L->num_blocks), s));
  ctx->own_launches += 1;
  k_flag_listed<<<grid_for(n, 128), 128, 0, s>>>(L->v, ctx->stage_b.as<int32_t>(),
                                                 static_cast<int>(n), ctx->stage_c.as<uint8_t>());
  int32_t rc = remove_flagged_blocks(L, ctx->stage_c.as<uint8_t>(), removed_out);
  if (rc) return rc;
  return finish_call(L, nullptr);
}

int64_t cg_layer_num_blocks(const cg_layer* L) { return L ? L->num_blocks : -1; }
float cg_layer_voxel_size(const cg_layer* L) { return L ? L->v.voxel_size : 0.0f; }

int32_t cg_layer_block_indices(const cg_layer* L, size_t capacity, int32_t* idx, size_t* n_out) {
  if (!L) return CG_ERR_INVALID_ARG;
  const size_t n = static_cast<size_t>(L->num_blocks);
  if (n_out) *n_out = n;
  if (!idx || n == 0) return CG_OK;
  if (capacity < n) {
    set_error("cg_layer_block_indices: capacity %zu < %zu blocks", capacity, n);
    return CG_ERR_INVALID_ARG;
  }
  cg_context* ctx = L->ctx;
  const uint64_t* keys;
  const uint32_t* slots;
  int32_t rc = sort_blocks(L, &keys, &slots);
  if (rc) return rc;
  CG_CUDA(ctx->stage_b.reserve(n * 3 * sizeof(int32_t)));
  k_unpack_idx<<<grid_for(n, 256), 256, 0, ctx->stream>>>(keys, static_cast<int>(n),
                                                          ctx->stage_b.as<int32_t>());
  CG_CUDA(cudaMemcpyAsync(idx, ctx->stage_b.p, n * 3 * sizeof(int32_t), cudaMemcpyDeviceToHost,
                          ctx->stream));
  CG_CUDA(cudaStreamSynchronize(ctx->stream));
  return CG_OK;
}

int32_t cg_layer_download(const cg_layer* L, size_t capacity, int32_t* idx, cg_tsdf_voxel* voxels,
                          uint8_t* flags, size_t* n_out) {
  if (!L) return CG_ERR_INVALID_ARG;
  const size_t n = static_cast<size_t>(L->num_blocks);
  if (n_out) *n_out = n;
  if (n == 0 || (!idx && !voxels && !flags)) return CG_OK;
  if (capacity < n) {
    set_error("cg_layer_download: capacity %zu < %zu blocks", capacity, n);
    return CG_ERR_INVALID_ARG;
  }
  cg_context* ctx = L->ctx;
  cudaStream_t s = ctx->stream;
  const uint64_t* keys;
  const uint32_t* slots;
  int32_t rc = sort_blocks(L, &keys, &slots);
  if (rc) return rc;
  const size_t chunk = 2048;  // 96 MB staging
  CG_CUDA(ctx->stage_a.reserve(std::min(chunk, n) * CG_BLOCK_BYTES));
  CG_CUDA(ctx->stage_b.reserve(std::min(chunk, n) * 3 * sizeof(int32_t)));
  CG_CUDA(ctx->stage_c.reserve(std::min(chunk, n)));
  for (size_t first = 0; first < n; first += chunk) {
    const size_t cnt = std::min(chunk, n - first);
    k_gather_aos<<<static_cast<unsigned>(cnt), 256, 0, s>>>(
        L->v, slots, static_cast<int>(first), static_cast<int>(cnt), ctx->stage_a.as<uint32_t>(),
        ctx->stage_b.as<int32_t>(), ctx->stage_c.as<uint8_t>(), keys);
    if (voxels)
      CG_CUDA(cudaMemcpyAsync(voxels + first * kVoxelsPerBlock, ctx->stage_a.p,
                              cnt * CG_BLOCK_BYTES, cudaMemcpyDeviceToHost, s));
    if (idx)
      CG_CUDA(cudaMemcpyAsync(idx + first * 3, ctx->stage_b.p, cnt * 3 * sizeof(int32_t),
                              cudaMemcpyDeviceToHost, s));
    if (flags)
      CG_CUDA(cudaMemcpyAsync(flags + first, ctx->stage_c.p, cnt, cudaMemcpyDeviceToHost, s));
    CG_CUDA(cudaStreamSynchronize(s));
  }
  CG_CUDA(cudaGetLastError());
  return CG_OK;
}

int32_t cg_layer_download_updated(const cg_layer* L, size_t capacity, int32_t* idx,
                                  cg_tsdf_voxel* voxels, uint8_t* flags, size_t* n_out) {
  if (!L) return CG_ERR_INVALID_ARG;
  cg_context* ctx = L->ctx;
  cudaStream_t s = ctx->stream;
  const size_t n_all = static_cast<size_t>(L->num_blocks);
  if (n_out) *n_out = 0;
  if (n_all == 0) return CG_OK;
  const uint64_t* keys;
  const uint32_t* slots;
  int32_t rc = sort_blocks(L, &keys, &slots);
  if (rc) return rc;
  // Layer::getAllUpdatedBlocks, in (z, y, x) order
  CG_CUDA(ctx->val_a.reserve(sizeof(uint32_t) * (2 * n_all + 1)));  // val_a is free after the sort
  CG_CUDA(ctx->flags.reserve(sizeof(uint64_t) * n_all));
  uint32_t* d_order = ctx->val_a.as<uint32_t>();
  uint32_t* d_slots = d_order + n_all + 1;
  uint64_t* d_keys = ctx->flags.as<uint64_t>();
  k_select_updated<<<1, 1024, 0, s>>>(L->v, slots, static_cast<int>(n_all), d_order, d_order + n_all);
  uint32_t cnt_upd = 0;
  CG_CUDA(cudaMemcpyAsync(&cnt_upd, d_order + n_all, sizeof(uint32_t), cudaMemcpyDeviceToHost, s));
  CG_CUDA(cudaStreamSynchronize(s));
  const size_t n = cnt_upd;
  if (n_out) *n_out = n;
  if (n == 0 || (!idx && !voxels && !flags)) return CG_OK;
  if (capacity < n) {
    set_error("cg_layer_download_updated: capacity %zu < %zu blocks", capacity, n);
    return CG_ERR_INVALID_ARG;
  }
  k_compact_blocks<<<grid_for(n, 256), 256, 0, s>>>(keys, slots, d_order, static_cast<uint32_t>(n),
                                                    d_keys, d_slots);
  const size_t chunk = 2048;  // 96 MB staging
  CG_CUDA(ctx->stage_a.reserve(std::min(chunk, n) * CG_BLOCK_BYTES));
  CG_CUDA(ctx->stage_b.reserve(std::min(chunk, n) * 3 * sizeof(int32_t)));
  CG_CUDA(ctx->stage_c.reserve(std::min(chunk, n)));
  for (size_t first = 0; first < n; first += chunk) {
    const size_t cnt = std::min(chunk, n - first);
    k_gather_aos<<<static_cast<unsigned>(cnt), 256, 0, s>>>(
        L->v, d_slots, static_cast<int>(first), static_cast<int>(cnt), ctx->stage_a.as<uint32_t>(),
        ctx->stage_b.as<int32_t>(), ctx->stage_c.as<uint8_t>(), d_keys);
    if (voxels)
      CG_CUDA(cudaMemcpyAsync(voxels + first * kVoxelsPerBlock, ctx->stage_a.p,
                              cnt * CG_BLOCK_BYTES, cudaMemcpyDeviceToHost, s));
    if (idx)
      CG_CUDA(cudaMemcpyAsync(idx + first * 3, ctx->stage_b.p, cnt * 3 * sizeof(int32_t),
                              cudaMemcpyDeviceToHost, s));
    if (flags)
      CG_CUDA(cudaMemcpyAsync(flags + first, ctx->stage_c.p, cnt, cudaMemcpyDeviceToHost, s));
    CG_CUDA(cudaStreamSynchronize(s));
  }
  CG_CUDA(cudaGetLastError());
  return CG_OK;
}

int32_t cg_layer_download_blocks(const cg_layer* L, size_t n, const int32_t* idx,
                                 cg_tsdf_voxel* voxels, uint8_t* flags, uint8_t* found) {
  if (!L || (n && (!idx || !found))) {
    set_error("cg_layer_download_blocks: null argument");
    return CG_ERR_INVALID_ARG;
  }
  if (n == 0) return CG_OK;
  cg_context* ctx = L->ctx;
  cudaStream_t s = ctx->stream;
  const size_t chunk = 2048;
  CG_CUDA(ctx->stage_a.reserve(std::min(chunk, n) * CG_BLOCK_BYTES));
  CG_CUDA(ctx->stage_b.reserve(std::min(chunk, n) * 3 * sizeof(int32_t)));
  CG_CUDA(ctx->stage_c.reserve(std::min(chunk, n) * 2));
  CG_CUDA(ctx->key_b.reserve(std::min(chunk, n) * sizeof(uint64_t)));
  CG_CUDA(ctx->val_b.reserve(std::min(chunk, n) * sizeof(uint32_t)));
  for (size_t first = 0; first < n; first += chunk) {
    const size_t cnt = std::min(chunk, n - first);
    uint8_t* d_flags = ctx->stage_c.as<uint8_t>();
    uint8_t* d_found = d_flags + cnt;
    CG_CUDA(cudaMemcpyAsync(ctx->stage_b.p, idx + 3 * first, cnt * 3 * sizeof(int32_t),
                            cudaMemcpyHostToDevice, s));
    k_lookup_listed<<<grid_for(cnt, 256), 256, 0, s>>>(L->v, ctx->stage_b.as<int32_t>(),
                                                       static_cast<int>(cnt), ctx->val_b.as<uint32_t>(),
                                                       ctx->key_b.as<uint64_t>(), d_found);
    // blocks that are not allocated come back as whatever slot 0 holds; `found` tells
    k_gather_aos<<<static_cast<unsigned>(cnt), 256, 0, s>>>(
        L->v, ctx->val_b.as<uint32_t>(), 0, static_cast<int>(cnt), ctx->stage_a.as<uint32_t>(),
        nullptr, d_flags, ctx->key_b.as<uint64_t>());
    if (voxels)
      CG_CUDA(cudaMemcpyAsync(voxels + first * kVoxelsPerBlock, ctx->stage_a.p,
                              cnt * CG_BLOCK_BYTES, cudaMemcpyDeviceToHost, s));
    if (flags) CG_CUDA(cudaMemcpyAsync(flags + first, d_flags, cnt, cudaMemcpyDeviceToHost, s));
    CG_CUDA(cudaMemcpyAsync(found + first, d_found, cnt, cudaMemcpyDeviceToHost, s));
    CG_CUDA(cudaStreamSynchronize(s));
  }
  CG_CUDA(cudaGetLastError());
  return CG_OK;
}

int32_t cg_layer_hash_stats(const cg_layer* L, cg_hash_stats* out) {
  if (!L || !out) return CG_ERR_INVALID_ARG;
  cg_context* ctx = L->ctx;
  cudaStream_t s = ctx->stream;
  memset(out, 0, sizeof(*out));
  out->num_blocks = static_cast<uint64_t>(L->num_blocks);
  out->max_blocks = L->max_blocks;
  out->hash_capacity = L->hash_cap;
  out->load_factor = static_cast<double>(L->num_blocks) / static_cast<double>(L->hash_cap);
  if (L->num_blocks == 0) return CG_OK;
  CG_CUDA(ctx->stage_c.reserve(2 * sizeof(unsigned long long)));
  CG_CUDA(cudaMemsetAsync(ctx->stage_c.p, 0, 2 * sizeof(unsigned long long), s));
  k_probe_lengths<<<grid_for(static_cast<size_t>(L->num_blocks), 256), 256, 0, s>>>(
      L->v, static_cast<int>(L->num_blocks), ctx->stage_c.as<unsigned long long>());
  unsigned long long h[2] = {0, 0};
  CG_CUDA(cudaMemcpyAsync(h, ctx->stage_c.p, sizeof(h), cudaMemcpyDeviceToHost, s));
  CG_CUDA(cudaStreamSynchronize(s));
  out->mean_probe_length = static_cast<double>(h[0]) / static_cast<double>(L->num_blocks);
  out->max_probe_length = h[1];
  return CG_OK;
}

int32_t cg_layer_serialize(const cg_layer* L, int32_t only_updated, size_t capacity, int32_t* idx,
                           uint32_t* data, size_t* n_out) {
  if (!L) return CG_ERR_INVALID_ARG;
  cg_context* ctx = L->ctx;
  cudaStream_t s = ctx->stream;
  const size_t n_all = static_cast<size_t>(L->num_blocks);
  if (n_out) *n_out = 0;
  if (n_all == 0) return CG_OK;
  const uint64_t* keys;
  const uint32_t* slots;
  int32_t rc = sort_blocks(L, &keys, &slots);
  if (rc) return rc;
  size_t n = n_all;
  const uint32_t* order = nullptr;
  if (only_updated) {  // Layer::getAllUpdatedBlocks
    CG_CUDA(ctx->val_a.reserve(sizeof(uint32_t) * (n_all + 1)));  // val_a is free after the sort
    uint32_t* d_order = ctx->val_a.as<uint32_t>();
    k_select_updated<<<1, 1024, 0, s>>>(L->v, slots, static_cast<int>(n_all), d_order,
                                        d_order + n_all);
    uint32_t cnt = 0;
    CG_CUDA(cudaMemcpyAsync(&cnt, d_order + n_all, sizeof(uint32_t), cudaMemcpyDeviceToHost, s));
    CG_CUDA(cudaStreamSynchronize(s));
    n = cnt;
    order = d_order;
  }
  if (n_out) *n_out = n;
  if (n == 0 || (!idx && !data)) return CG_OK;
  if (capacity < n || !idx || !data) {
    set_error("cg_layer_serialize: capacity %zu < %zu blocks (or null output)", capacity, n);
    return CG_ERR_INVALID_ARG;
  }
  const size_t chunk = 2048;  // 96 MB staging
  CG_CUDA(ctx->stage_a.reserve(std::min(chunk, n) * CG_BLOCK_BYTES));
  CG_CUDA(ctx->stage_b.reserve(std::min(chunk, n) * 3 * sizeof(int32_t)));
  for (size_t first = 0; first < n; first += chunk) {
    const size_t cnt = std::min(chunk, n - first);
    k_serialize_blocks<<<static_cast<unsigned>(cnt), 256, 0, s>>>(
        L->v, order ? slots : slots + first, static_cast<int>(cnt), ctx->stage_a.as<uint32_t>(),
        ctx->stage_b.as<int32_t>(), order ? keys : keys + first, order ? order + first : nullptr);
    CG_CUDA(cudaMemcpyAsync(data + first * 3 * kVoxelsPerBlock, ctx->stage_a.p, cnt * CG_BLOCK_BYTES,
                            cudaMemcpyDeviceToHost, s));
    CG_CUDA(cudaMemcpyAsync(idx + first * 3, ctx->stage_b.p, cnt * 3 * sizeof(int32_t),
                            cudaMemcpyDeviceToHost, s));
    CG_CUDA(cudaStreamSynchronize(s));
  }
  CG_CUDA(cudaGetLastError());
  return CG_OK;
}

int32_t cg_layer_reset_updated(cg_layer* L) {
  if (!L) return CG_ERR_INVALID_ARG;
  if (L->num_blocks > 0)
    CG_CUDA(cudaMemsetAsync(L->v.updated, 0, static_cast<size_t>(L->num_blocks), L->ctx->stream));
  CG_CUDA(cudaStreamSynchronize(L->ctx->stream));
  return CG_OK;
}

int32_t cg_layer_deserialize(cg_layer* L, size_t n, const int32_t* idx, const uint32_t* data) {
  if (!L || (n && (!idx || !data))) return CG_ERR_INVALID_ARG;
  cg_context* ctx = L->ctx;
  cudaStream_t s = ctx->stream;
  const size_t chunk = 2048;
  CG_CUDA(ctx->stage_a.reserve(std::min(chunk, n) * CG_BLOCK_BYTES));
  CG_CUDA(ctx->stage_b.reserve(std::min(chunk, n) * 4 * sizeof(int32_t)));
  for (size_t first = 0; first < n; first += chunk) {
    const size_t cnt = std::min(chunk, n - first);
    int32_t* d_idx = ctx->stage_b.as<int32_t>();
    int32_t* d_entries = d_idx + 3 * cnt;
    CG_CUDA(cudaMemcpyAsync(d_idx, idx + 3 * first, cnt * 3 * sizeof(int32_t),
                            cudaMemcpyHostToDevice, s));
    CG_CUDA(cudaMemcpyAsync(ctx->stage_a.p, data + first * 3 * kVoxelsPerBlock, cnt * CG_BLOCK_BYTES,
                            cudaMemcpyHostToDevice, s));
    k_upload_insert<<<grid_for(cnt, 128), 128, 0, s>>>(L->v, d_idx, static_cast<int>(cnt),
                                                       d_entries);
    k_deserialize_write<<<static_cast<unsigned>(cnt), 256, 0, s>>>(
        L->v, d_entries, ctx->stage_a.as<uint32_t>(), static_cast<int>(cnt));
    CG_CUDA(cudaStreamSynchronize(s));
  }
  return finish_call(L, nullptr);
}

int32_t cg_layer_upload(cg_layer* L, size_t n, const int32_t* idx, const cg_tsdf_voxel* voxels,
                        const uint8_t* flags) {
  if (!L || (n && (!idx || !voxels))) return CG_ERR_INVALID_ARG;
  cg_context* ctx = L->ctx;
  cudaStream_t s = ctx->stream;
  const size_t chunk = 2048;
  CG_CUDA(ctx->stage_a.reserve(std::min(chunk, n) * CG_BLOCK_BYTES));
  CG_CUDA(ctx->stage_b.reserve(std::min(chunk, n) * 4 * sizeof(int32_t)));
  CG_CUDA(ctx->stage_c.reserve(std::min(chunk, n)));
  for (size_t first = 0; first < n; first += chunk) {
    const size_t cnt = std::min(chunk, n - first);
    int32_t* d_idx = ctx->stage_b.as<int32_t>();
    int32_t* d_entries = d_idx + 3 * cnt;
    CG_CUDA(cudaMemcpyAsync(d_idx, idx + 3 * first, cnt * 3 * sizeof(int32_t),
                            cudaMemcpyHostToDevice, s));
    CG_CUDA(cudaMemcpyAsync(ctx->stage_a.p, voxels + first * kVoxelsPerBlock, cnt * CG_BLOCK_BYTES,
                            cudaMemcpyHostToDevice, s));
    if (flags)
      CG_CUDA(cudaMemcpyAsync(ctx->stage_c.p, flags + first, cnt, cudaMemcpyHostToDevice, s));
    k_upload_insert<<<grid_for(cnt, 128), 128, 0, s>>>(L->v, d_idx, static_cast<int>(cnt),
                                                       d_entries);
    k_upload_write<<<static_cast<unsigned>(cnt), 256, 0, s>>>(
        L->v, d_entries, ctx->stage_a.as<uint32_t>(), flags ? ctx->stage_c.as<uint8_t>() : nullptr,
        static_cast<int>(cnt));
    CG_CUDA(cudaStreamSynchronize(s));
  }
  return finish_call(L, nullptr);
}

}  // extern "C"
