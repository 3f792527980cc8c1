// cg_internal.cuh — context / layer state and the GPU block hash shared by the .cu files.
//
// Layer<TsdfVoxel> replacement (SURVEY.md §2.2 E3, a4): an open-addressing hash
// (packed int3 block index -> pool slot) plus a block pool laid out for coalesced access:
// each 16^3 block is three 16 KB planes  [distance f32 x4096 | weight f32 x4096 | rgba u32 x4096]
// (49,152 B, the same size as voxblox's AoS block; converted to AoS only at the boundary).
// Unallocated pool slots are kept in the default-constructed state (d = 0, w = 0,
// colour (0,0,0,255)) so that a freshly claimed block needs no initialisation pass.
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>
#include <stdio.h>
#include <stdlib.h>

#include <chrono>

#include <string>
#include <vector>

#include "../../include/coxgraph_b200.h"
#include "cg_math.cuh"

namespace cg {

constexpr uint64_t kEmptyKey = ~0ull;
constexpr int kBlockIdxBits = 21;                    // per axis, offset 2^20
constexpr int kBlockIdxOffset = 1 << 20;
constexpr int kVoxIdxBits = 20;                      // per axis (bundle keys), offset 2^19
constexpr int kVoxIdxOffset = 1 << 19;
constexpr uint64_t kInvalidPointKey = ~0ull;         // sorts behind every valid key
constexpr int kClearingBit = 60;

enum ErrBits { kErrPoolFull = 1, kErrOutOfRange = 2, kErrTouchFull = 4, kErrSegmentFull = 8, kErrKeyRange = 16 };

// ------------------------------------------------------------------ key packing
__host__ __device__ __forceinline__ uint64_t pack_block_key(int x, int y, int z) {
  return (static_cast<uint64_t>(static_cast<uint32_t>(z + kBlockIdxOffset)) << 42) |
         (static_cast<uint64_t>(static_cast<uint32_t>(y + kBlockIdxOffset)) << 21) |
         static_cast<uint64_t>(static_cast<uint32_t>(x + kBlockIdxOffset));
}
__host__ __device__ __forceinline__ void unpack_block_key(uint64_t k, int& x, int& y, int& z) {
  x = static_cast<int>(k & 0x1FFFFF) - kBlockIdxOffset;
  y = static_cast<int>((k >> 21) & 0x1FFFFF) - kBlockIdxOffset;
  z = static_cast<int>((k >> 42) & 0x1FFFFF) - kBlockIdxOffset;
}
__device__ __forceinline__ uint64_t pack_voxel_key(int x, int y, int z) {
  return (static_cast<uint64_t>(static_cast<uint32_t>(z + kVoxIdxOffset)) << 40) |
         (static_cast<uint64_t>(static_cast<uint32_t>(y + kVoxIdxOffset)) << 20) |
         static_cast<uint64_t>(static_cast<uint32_t>(x + kVoxIdxOffset));
}
__device__ __forceinline__ bool voxel_index_in_range(int x, int y, int z) {
  return x >= -kVoxIdxOffset && x < kVoxIdxOffset && y >= -kVoxIdxOffset && y < kVoxIdxOffset &&
         z >= -kVoxIdxOffset && z < kVoxIdxOffset;
}
__host__ __device__ __forceinline__ uint32_t hash_key(uint64_t k) {
  k ^= k >> 33;
  k *= 0xff51afd7ed558ccdULL;
  k ^= k >> 33;
  k *= 0xc4ceb9fe1a85ec53ULL;
  k ^= k >> 33;
  return static_cast<uint32_t>(k);
}

// ------------------------------------------------------------------ device view of a layer
struct LayerView {
  uint64_t* hash_keys;   // [hash_cap] packed block key or kEmptyKey
  int32_t* hash_vals;    // [hash_cap] pool slot (-1: no slot, pool exhausted)
  uint64_t* block_keys;  // [max_blocks] slot -> packed block key
  uint8_t* has_data;     // [max_blocks]
  uint8_t* updated;      // [max_blocks]
  float* pool;           // [max_blocks * 3 * 4096] planes per block
  int32_t* num_blocks;   // device counter of claimed slots
  int32_t* err;          // device error bits
  uint32_t hash_mask;
  int32_t max_blocks;
  float voxel_size, voxel_size_inv, block_size, block_size_inv;

  __device__ __forceinline__ float* dist_plane(int slot) const {
    return pool + static_cast<size_t>(slot) * (3 * kVoxelsPerBlock);
  }
  __device__ __forceinline__ float* weight_plane(int slot) const {
    return dist_plane(slot) + kVoxelsPerBlock;
  }
  __device__ __forceinline__ uint32_t* color_plane(int slot) const {
    return reinterpret_cast<uint32_t*>(dist_plane(slot) + 2 * kVoxelsPerBlock);
  }

  // hash entry of `key`, or -1
  __device__ __forceinline__ int find_entry(uint64_t key) const {
    uint32_t h = hash_key(key) & hash_mask;
    for (;;) {
      const uint64_t k = hash_keys[h];
      if (k == key) return static_cast<int>(h);
      if (k == kEmptyKey) return -1;
      h = (h + 1) & hash_mask;
    }
  }
  __device__ __forceinline__ int find_slot(uint64_t key) const {
    const int e = find_entry(key);
    return e < 0 ? -1 : hash_vals[e];
  }
  // insert-or-find; returns the hash entry.  The inserting thread claims a pool slot and
  // publishes it in hash_vals[entry]; other kernels read it after this kernel completes.
  __device__ __forceinline__ int insert_entry(uint64_t key) const {
    uint32_t h = hash_key(key) & hash_mask;
    for (;;) {
      uint64_t k = hash_keys[h];
      if (k == key) return static_cast<int>(h);
      if (k == kEmptyKey) {
        const unsigned long long old =
            atomicCAS(reinterpret_cast<unsigned long long*>(&hash_keys[h]), kEmptyKey, key);
        if (old == kEmptyKey) {
          const int slot = atomicAdd(num_blocks, 1);
          if (slot < max_blocks) {
            hash_vals[h] = slot;
            block_keys[slot] = key;
          } else {
            hash_vals[h] = -1;
            atomicOr(err, kErrPoolFull);
          }
          return static_cast<int>(h);
        }
        if (old == key) return static_cast<int>(h);
      }
      h = (h + 1) & hash_mask;
    }
  }
};

// ------------------------------------------------------------------ host-side state
struct DevBuf {
  void* p = nullptr;
  size_t cap = 0;
  cudaError_t reserve(size_t bytes) {
    if (bytes <= cap) return cudaSuccess;
    const bool trace = getenv("CG_TRACE_ALLOC") != nullptr;
    const auto t0 = std::chrono::steady_clock::now();
    const size_t old_cap = cap;
    if (p) cudaFree(p);
    p = nullptr;
    cap = 0;
    size_t want = bytes + bytes / 2 + 256;  // geometric growth: every reallocation is a device-wide stall
    cudaError_t e = cudaMalloc(&p, want);
    if (e != cudaSuccess) {
      want = bytes;
      e = cudaMalloc(&p, want);
    }
    if (e == cudaSuccess) cap = want;
    if (trace) {
      const double ms = std::chrono::duration<double, std::milli>(std::chrono::steady_clock::now() - t0).count();
      fprintf(stderr, "[cg] scratch %zu -> %zu bytes in %.2f ms\n", old_cap, want, ms);
    }
    return e;
  }
  void release() {
    if (p) cudaFree(p);
    p = nullptr;
    cap = 0;
  }
  template <class T>
  T* as() const {
    return static_cast<T*>(p);
  }
};

// counters read back once per call (pinned host mirror)
struct CallCounters {
  unsigned long long rays;
  unsigned long long pairs;
  unsigned long long touched;
  unsigned long long general_pairs;
  unsigned long long segments;
  int key_lo[3], key_hi[3];  // extent of the job's points (voxel indices relative to the sensor voxel)
  unsigned long long candidates;
  unsigned long long blocks_out;
  unsigned long long far_points;   // points beyond the key reach, counted by the running front half
  unsigned long long far_dropped;  // ... of the front half the host has just synchronised on
  int err;
  int num_blocks;
};

// named stages (the reference wraps the same path in voxblox::timing::Timer scopes,
// coxgraph/include/coxgraph/map_comm/tsdf_recover.h:63,74-76)
enum Stage {
  kStagePointKeys = 0,
  kStageBundleSort,
  kStageBundleScan,
  kStageGather,
  kStageBundleOrder,
  kStageFoldWide,
  kStageFold,
  kStageBundleRays,
  kStageRayScan,
  kStageWalkSegments,
  kStageSegmentSort,
  kStageBlockAccumulate,
  kStagePairSort,
  kStageSegments,
  kStageVisits,
  kStageVoxelUpdate,
  kStageReplayWide,
  kStageFinalize,
  kStageMergeMark,
  kStageMergeResample,
  kStageTransfer,
  kNumStages
};
const char* stage_name(int s);
struct PendingEvent {
  int stage;
  cudaEvent_t start, stop;
};

// Everything a job's layer-independent front half (points -> one ray per bundle,
// integrate_front.cu) writes and its back half reads.  The context is set 0 (plain calls); cg_prepare_batch_* uses
// further sets on a second stream so that the front half of a later job overlaps the back half of
// the current one.
struct FrontBufs {
  void* h_tables = nullptr;                 // pinned + mapped: poses / frame offsets of the job
  size_t h_tables_cap = 0;
  const float* group_poses = nullptr;       // device poses of the group being fused
  int group_frames = 0;
  CallCounters* h_counters = nullptr;       // pinned
  CallCounters* d_counters = nullptr;
  DevBuf poses, frame_base;
  DevBuf key_a, key_b, scan, cub_tmp;
  DevBuf rays, ray_count, ray_offset, sorted_pts;
  DevBuf ray_id, frame_count;               // bundle -> ray id; (frame, chunk) bundle counts
  DevBuf scan_partials;
  DevBuf grazing_keys, grazing_ray_key;     // anti-grazing: the scan's bundle voxels
  uint32_t grazing_mask = 0;
  uint32_t* d_class_count = nullptr;        // bundle size-class histogram + scatter cursors
  int* d_key_bounds = nullptr;              // [6] running min / max of the bundle voxel fields
  uint32_t* d_select_count = nullptr;       // output count of the stream compactions
  int32_t* d_front_err = nullptr;           // error bits of a prepared front half (sets > 0)
  // independent stages of one job side by side (gather || bundle heads + order; short || long
  // update lists): a second stream forked from / joined to the job's stream by events
  cudaStream_t side = nullptr;
  cudaEvent_t ev_fork = nullptr, ev_join = nullptr;
};
// creates fb.side at the priority of `like` on first use; false: run everything on one stream
bool side_stream(FrontBufs& fb, cudaStream_t like);
cudaError_t init_front_words(FrontBufs& fb);  // the small device / pinned words of a set
void release_front(FrontBufs& fb);

}  // namespace cg

struct cg_comm;  // comm.cu: communicator + peer mappings of the multi-GPU merge
namespace cg {
struct HostStager;  // host_stage.cu: worker threads + pinned bounce buffer for pageable inputs
}

struct cg_context : cg::FrontBufs {
  int device = 0;
  cg_comm* comm = nullptr;
  cudaStream_t stream = nullptr;
  bool own_stream = false;
  cudaEvent_t wait_event = nullptr;         // cg_context_wait_stream
  cg::HostStager* stager = nullptr;         // pageable inputs (lazy, host_stage.cu)
  cudaStream_t copy_stream = nullptr;       // cg_stage_batch_async transfers (lazy)
  cg::DevBuf stage_pts[2], stage_cols[2];   // cg_stage_batch_async double buffer
  cudaEvent_t stage_ready[2] = {nullptr, nullptr};
  size_t stage_points[2] = {0, 0};
  int num_sms = 148;
  // integration scratch
  cg::DevBuf points, colors;
  cg::DevBuf val_a, val_b, flags;
  cg::DevBuf pkey_a, pkey_b, seg_start, long_list, long_partials, visits;
  cg::DevBuf seg_keys_a, seg_keys_b, seg_idx_a, seg_idx_b, seg_recs;  // (ray, block) segments
  cg::DevBuf seg_order;  // update lists in size-class order
  cg::DevBuf seg_bins;
  // per-call touch set (integrate_back.cu): kept all-clear between calls
  cg::DevBuf touch_ord, touch_entry, touch_acc, touch_bits;
  uint32_t* d_touch_count = nullptr;  // [0] blocks touched, [1] general (voxel, ray) keys emitted
  uint32_t* d_walk_counters = nullptr;  // [0],[1] dynamic work counters, [2] bundle key reach
  bool key_box_valid = false;           // bundle key layout (adaptive): union of the extents
  int key_lo[3] = {0, 0, 0}, key_hi[3] = {0, 0, 0};  // measured by the jobs of this context
  int key_win_lo[3] = {0, 0, 0}, key_win_hi[3] = {0, 0, 0}, key_win_jobs = 0;  // last <= 8 measured jobs
  unsigned key_jobs = 0;
  bool key_retry_measured = false;      // the pass that asked for a retry had measured the extent
  size_t touch_cap = 0;               // blocks the scratch holds
  bool touch_clean = false;
  unsigned long long* d_long_counter = nullptr;  // (#long segments << 32) | #sub-blocks
  uint32_t* d_work_counter = nullptr;  // dynamic work distribution of the persistent kernels
  // merge / transfer scratch
  cg::DevBuf cand_keys, cand_list, stage_a, stage_b, stage_c;
  cg::DevBuf batch_desc, merge_cands;  // batched projection (merge.cu)
  // mesh recovery (mesh_recover.cu)
  cg::DevBuf mesh_in, mesh_tri, mesh_pairs, mesh_pts_g, mesh_cols_g, mesh_pts_c, mesh_cols_c,
      mesh_frames;
  // marching cubes (mesh.cu)
  cg::DevBuf mc_counts, mc_index, mc_vertices, mc_normals, mc_colors;
  size_t mc_blocks = 0, mc_total = 0;  // size of the retained result (cg_mesh_fetch)
  cg::DevBuf weld_keys, weld_words, weld_out;  // vertex welding (mesh_connect.cu)
  // ESDF of a layer (esdf.cu): working / result planes in (z, y, x) block order, retained until
  // the next cg_layer_esdf_batch on this context
  cg::DevBuf esdf_keys, esdf_slots, esdf_dist, esdf_packed, esdf_fixed, esdf_slot_to_b,
      esdf_dirty, esdf_list, esdf_index, esdf_counters;
  size_t esdf_blocks = 0;
  float esdf_voxel_size = 0.0f, esdf_block_size = 0.0f;
  // instrumentation
  bool profiling = false;
  uint64_t own_launches = 0;  // kernels of this library launched (library sorts/scans excluded)
  // pipelined jobs (cg_prepare_batch_*): two further front-half sets on their own stream
  cg::FrontBufs prep[2];
  cudaStream_t prep_stream = nullptr;
  cudaEvent_t prep_done[2] = {nullptr, nullptr};
  struct PreparedJob {
    bool valid = false;
    cg_integrator_config cfg;
    std::vector<float> poses;
    std::vector<uint64_t> offs;  // relative to the job's first point
    const float* d_points = nullptr;
    const uint8_t* d_colors = nullptr;
    int freespace = 0;
    float voxel_size = 0.0f;
    bool front_queued = false;   // false: the job did not fit the one-group fast path
    // completes the staged copy of d_points / d_colors (cg_prepare_batch_staged); the job waits
    // on it only when it runs the plain way, on the context's stream
    cudaEvent_t inputs_ready = nullptr;
  } prepared[2];
  double stage_ms[cg::kNumStages] = {};
  uint64_t stage_launches[cg::kNumStages] = {};
  std::vector<cg::PendingEvent> pending;
  std::vector<cudaEvent_t> event_pool;
};

struct cg_layer {
  cg_context* ctx = nullptr;
  cg::LayerView v{};
  size_t hash_cap = 0;
  size_t max_blocks = 0;
  int64_t num_blocks = 0;  // host mirror, refreshed at the end of every mutating call
};

namespace cg {

void set_error(const char* fmt, ...);
int32_t cuda_fail(cudaError_t e, const char* what);
// pulls error bits + num_blocks back from the device; returns the status for the error bits
int32_t finish_call(cg_layer* layer, CallCounters* out);
// sorted (z,y,x) view of the allocated blocks: keys in ctx->key_b, slots in ctx->val_b
int32_t sort_blocks(const cg_layer* layer, const uint64_t** keys, const uint32_t** slots);
// Layer::removeBlock for every slot with d_remove[slot] != 0 (device flags, one per claimed slot):
// compacts the pool, rebuilds the hash; enqueued on the context's stream, host mirror updated
int32_t remove_flagged_blocks(cg_layer* layer, const uint8_t* d_remove, uint64_t* removed_out);

#define CG_CUDA(expr)                                         \
  do {                                                        \
    cudaError_t _e = (expr);                                  \
    if (_e != cudaSuccess) return cg::cuda_fail(_e, #expr);   \
  } while (0)

// RAII scope around one pipeline stage: counts the library's own kernel launches and, when
// profiling is on, brackets the stage with CUDA events on the context's stream.
struct StageScope {
  cg_context* ctx;
  int stage;
  cudaEvent_t start = nullptr, stop = nullptr;
  cudaStream_t stream;
  StageScope(cg_context* c, int st, int own_kernels, cudaStream_t on = nullptr)
      : ctx(c), stage(st), stream(on ? on : c->stream) {
    ctx->own_launches += own_kernels;
    ctx->stage_launches[st] += own_kernels;
    if (ctx->profiling) {
      start = take();
      stop = take();
      cudaEventRecord(start, stream);
    }
  }
  ~StageScope() {
    if (start) {
      cudaEventRecord(stop, stream);
      ctx->pending.push_back(PendingEvent{stage, start, stop});
    }
  }
  cudaEvent_t take() {
    if (!ctx->event_pool.empty()) {
      cudaEvent_t e = ctx->event_pool.back();
      ctx->event_pool.pop_back();
      return e;
    }
    cudaEvent_t e;
    cudaEventCreate(&e);
    return e;
  }
};

inline unsigned grid_for(size_t n, unsigned block) {
  return static_cast<unsigned>((n + block - 1) / block);
}

}  // namespace cg
