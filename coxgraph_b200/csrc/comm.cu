// comm.cu — the server's global merge across the GPUs of one box, behind the C ABI (SURVEY.md
// §8b cg_comm_init / cg_gather_global, §8e).
//
// Every rank projects its submaps into a *partial* global layer.  The exchange is an owner-pull
// over NVLink peer memory (peer pointers opened through CUDA IPC):
//   k_build_holders  every rank reads the block keys of every rank's partial layer (8 B per block)
//                    and builds the same map  block -> set of ranks that hold it
//   k_list_owned     the owner of a block is one of its HOLDERS, picked by a hash of the index: a
//                    block only one rank holds never crosses NVLink, contested blocks spread
//                    evenly over their holders
//   k_fold_owned     one CTA per owned block: the holders' copies are read straight out of their
//                    block pools, in ascending rank order, and folded in shared memory with
//                    voxblox::mergeLayerAintoLayerB's aligned form (Block::mergeBlock /
//                    mergeVoxelAIntoVoxelB, R10; reference call site of that overload:
//                    coxgraph/src/server/submap_collection.cpp:31-33); the block is written once
// — gather and fold are ONE kernel, there is no packing pass, no staging copy and no host
// synchronisation between listing, exchange and fold.  NCCL (loaded at run time from
// libnccl.so.2, the one torch has loaded if there is one) is the bootstrap and the barrier only:
// unique id -> communicator, one all-gather of the IPC handles when a partial layer is bound, and a
// one-word all-reduce on the stream before and after the kernels (all partial layers complete /
// all peers done reading).  The fold order is fixed, so the result is deterministic and equal to
// the packed exchange of exchange.cu (hash owner, NCCL all-to-all) block for block.
//
// cg_layer_mesh_sharded (mesh.cu) meshes the owned layers where they lie.  Its collective half is
// here: the owned layer is bound like the partial one (its own binding, so alternating gather and
// mesh calls map nothing again), and k_build_holders, run over every rank's owned keys, also
// records where each block's planes are.  The mesh kernel resolves the one-block halo (the +x/+y/+z
// neighbours and a vertex's colour block) through that map and reads the peer's planes over
// NVLink; a key two ranks hold is found while the map is built.
#include <dlfcn.h>
#include <string.h>

#include <vector>

#include "cg_internal.cuh"

namespace cg {

// ---- the few NCCL entry points, resolved with dlsym (the library stays loadable without NCCL)
typedef struct ncclComm* ncclComm_t;
typedef struct { char internal[128]; } ncclUniqueId;
enum { ncclSuccess = 0 };
enum { ncclInt8 = 0, ncclUint8 = 1, ncclInt32 = 2 };
enum { ncclSum = 0 };
struct Nccl {
  void* lib = nullptr;
  int (*GetUniqueId)(ncclUniqueId*) = nullptr;
  int (*CommInitRank)(ncclComm_t*, int, ncclUniqueId, int) = nullptr;
  int (*CommDestroy)(ncclComm_t) = nullptr;
  int (*AllReduce)(const void*, void*, size_t, int, int, ncclComm_t, cudaStream_t) = nullptr;
  int (*AllGather)(const void*, void*, size_t, int, ncclComm_t, cudaStream_t) = nullptr;
  const char* (*GetErrorString)(int) = nullptr;
};
static Nccl g_nccl;

static int32_t load_nccl() {
  if (g_nccl.lib) return CG_OK;
  void* h = dlopen("libnccl.so.2", RTLD_NOW | RTLD_GLOBAL);
  if (!h) h = dlopen("libnccl.so", RTLD_NOW | RTLD_GLOBAL);
  if (!h) {
    set_error("multi-GPU merge needs NCCL: %s", dlerror());
    return CG_ERR_UNSUPPORTED;
  }
  Nccl n;
  n.lib = h;
  n.GetUniqueId = reinterpret_cast<decltype(n.GetUniqueId)>(dlsym(h, "ncclGetUniqueId"));
  n.CommInitRank = reinterpret_cast<decltype(n.CommInitRank)>(dlsym(h, "ncclCommInitRank"));
  n.CommDestroy = reinterpret_cast<decltype(n.CommDestroy)>(dlsym(h, "ncclCommDestroy"));
  n.AllReduce = reinterpret_cast<decltype(n.AllReduce)>(dlsym(h, "ncclAllReduce"));
  n.AllGather = reinterpret_cast<decltype(n.AllGather)>(dlsym(h, "ncclAllGather"));
  n.GetErrorString = reinterpret_cast<decltype(n.GetErrorString)>(dlsym(h, "ncclGetErrorString"));
  if (!n.GetUniqueId || !n.CommInitRank || !n.CommDestroy || !n.AllReduce || !n.AllGather ||
      !n.GetErrorString) {
    set_error("libnccl.so.2 lacks an expected symbol");
    return CG_ERR_UNSUPPORTED;
  }
  g_nccl = n;
  return CG_OK;
}
#define CG_NCCL(expr)                                                        \
  do {                                                                       \
    const int _r = (expr);                                                   \
    if (_r != ncclSuccess) {                                                 \
      set_error("NCCL error %d (%s) at %s", _r, g_nccl.GetErrorString(_r), #expr); \
      return CG_ERR_CUDA;                                                    \
    }                                                                        \
  } while (0)

// What a peer needs of a rank's bound layer (device pointers valid in the READER's process).
struct PeerLayer {
  const float* pool;
  const uint64_t* block_keys;
  const uint8_t* has_data;
  const uint32_t* shared;  // [0] number of blocks of the layer (written per call)
};
constexpr int kMaxRanks = 64;

struct IpcRecord {  // one per rank, all-gathered
  cudaIpcMemHandle_t pool, keys, flags, shared;
  unsigned long long off_pool, off_keys, off_flags, off_shared;  // pointer - allocation base
  unsigned long long max_blocks;
  float voxel_size;
  int pad;
};

// One role a layer of this rank plays for its peers (the partial layer of cg_gather_global, the
// owned layer of cg_layer_mesh_sharded): its block count published in `shared`, and every rank's
// buffers as this process sees them.  Pools are allocated once in cg_layer_create, so a binding
// holds for the layer's lifetime; it is made again only when a layer of another serial takes the
// role.
struct Binding {
  uint64_t serial = 0;            // cg_layer::serial of the bound layer (0: none)
  uint32_t* shared = nullptr;     // peer-visible: [0] blocks of this rank's layer (written per call)
  PeerLayer* d_peers = nullptr;   // [nranks]
  std::vector<char*> held;        // peer mappings this binding uses (one reference each)
};
// A peer allocation mapped into this process.  Small buffers of different layers can share one
// allocation, and a handle can be opened once only, so the bindings share the mappings.
struct Mapping {
  int rank;
  cudaIpcMemHandle_t handle;
  char* p;
  int refs;
};
}  // namespace cg

struct cg_comm {
  cg::ncclComm_t comm = nullptr;
  int rank = 0, nranks = 1;
  int* d_token = nullptr;             // barrier word
  cg::Binding partial, owned;
  std::vector<cg::Mapping> maps;
  uint64_t maps_opened = 0;           // cudaIpcOpenMemHandle calls since cg_comm_init
  // the holder map (scratch, rebuilt every call): block key -> set of ranks holding the block
  unsigned long long* hkeys = nullptr;
  unsigned long long* hmask = nullptr;
  uint32_t* hbase = nullptr;          // owned entries: first element of the block's slot list
  uint32_t* mine = nullptr;           // entries this rank owns
  uint32_t* slots = nullptr;          // pool slots of the holders' copies, per owned block
  uint32_t* counters = nullptr;       // [0] owned entries, [1] slot list cursor, [2] overflow
  size_t hcap = 0, list_cap = 0;
  // the key map of cg_layer_mesh_sharded over every rank's owned layer (rebuilt every call)
  unsigned long long* mkeys = nullptr;
  unsigned long long* mmask = nullptr;
  const float** mplanes = nullptr;    // the block's distance plane in its holder's pool
  uint32_t* mcounters = nullptr;      // k_build_holders' words ([2] overflow: cannot happen)
  size_t mcap = 0;
};

namespace cg {

__device__ __forceinline__ uint32_t holder_find(const unsigned long long* __restrict__ hkeys,
                                                uint32_t hmask_cap, unsigned long long key) {
  uint32_t h = hash_key(key) & hmask_cap;
  while (hkeys[h] != key) h = (h + 1) & hmask_cap;
  return h;
}
// the owner of a block: one of its holders, picked by a hash of the block index
__device__ __forceinline__ int pick_owner(unsigned long long key, unsigned long long mask) {
  int n = static_cast<int>((hash_key(key ^ 0x9E3779B97F4A7C15ULL) >> 7) %
                           static_cast<uint32_t>(__popcll(mask)));
  unsigned long long m = mask;
  while (n-- > 0) m &= m - 1;
  return __ffsll(static_cast<long long>(m)) - 1;
}

// Every block key of every rank's layer (read through the peer mappings) enters the map with its
// rank's bit.  Grid y = rank.  With `planes` (the key map of cg_layer_mesh_sharded) the entry also
// records where the block's planes are, and a key that reaches an entry another rank has already
// marked is held twice: the smallest such key goes to *dup_key.
__global__ void k_build_holders(const PeerLayer* __restrict__ peers, unsigned long long* hkeys,
                                unsigned long long* hmask, uint32_t hcap_mask, uint32_t* counters,
                                const float** planes, unsigned long long* dup_key) {
  const int r = blockIdx.y;
  const PeerLayer P = peers[r];
  const uint32_t n = P.shared[0];
  for (uint32_t i = blockIdx.x * blockDim.x + threadIdx.x; i < n; i += gridDim.x * blockDim.x) {
    const unsigned long long key = P.block_keys[i];
    uint32_t h = hash_key(key) & hcap_mask;
    for (uint32_t tries = 0;; ++tries) {
      const unsigned long long k = hkeys[h];
      if (k == key) break;
      if (k == kEmptyKey) {
        const unsigned long long old = atomicCAS(&hkeys[h], kEmptyKey, key);
        if (old == kEmptyKey || old == key) break;
      }
      h = (h + 1) & hcap_mask;
      if (tries > hcap_mask) {  // cannot happen: the map holds every block of every rank
        atomicExch(&counters[2], 1u);
        return;
      }
    }
    const unsigned long long held = atomicOr(&hmask[h], 1ull << r);
    if (planes) {
      planes[h] = P.pool + static_cast<size_t>(i) * (3 * kVoxelsPerBlock);
      if (held) atomicMin(dup_key, key);
    }
  }
}
// entries this rank owns, each with room for its holders' slots
__global__ void k_list_owned(const unsigned long long* __restrict__ hkeys,
                             const unsigned long long* __restrict__ hmask, uint32_t hcap, int me,
                             uint32_t* __restrict__ hbase, uint32_t* __restrict__ mine,
                             uint32_t list_cap, uint32_t* counters) {
  for (uint32_t e = blockIdx.x * blockDim.x + threadIdx.x; e < hcap; e += gridDim.x * blockDim.x) {
    const unsigned long long mask = hmask[e];
    if (!mask || pick_owner(hkeys[e], mask) != me) continue;
    const uint32_t pos = atomicAdd(&counters[0], 1u);
    const uint32_t base = atomicAdd(&counters[1], static_cast<uint32_t>(__popcll(mask)));
    if (pos < list_cap) {
      mine[pos] = e;
      hbase[e] = base;
    } else {
      atomicExch(&counters[2], 1u);
    }
  }
}
// the pool slot of every holder's copy of the blocks this rank owns.  Grid y = rank.
__global__ void k_holder_slots(const PeerLayer* __restrict__ peers,
                               const unsigned long long* __restrict__ hkeys,
                               const unsigned long long* __restrict__ hmask,
                               const uint32_t* __restrict__ hbase, uint32_t hcap_mask, int me,
                               uint32_t* __restrict__ slots, uint32_t slots_cap) {
  const int r = blockIdx.y;
  const PeerLayer P = peers[r];
  const uint32_t n = P.shared[0];
  for (uint32_t i = blockIdx.x * blockDim.x + threadIdx.x; i < n; i += gridDim.x * blockDim.x) {
    const unsigned long long key = P.block_keys[i];
    const uint32_t e = holder_find(hkeys, hcap_mask, key);
    const unsigned long long mask = hmask[e];
    if (pick_owner(key, mask) != me) continue;
    const uint32_t at = hbase[e] + __popcll(mask & ((1ull << r) - 1ull));
    if (at < slots_cap) slots[at] = i;
  }
}

// One CTA per owned block: the destination block (fresh blocks are in the default state) is staged
// in shared memory, every holder's copy is read through its mapping — 16-byte loads, across
// NVLink for the peers — and folded in ascending rank order, and the result is written once.
constexpr int kFoldThreads = 256;
__global__ void __launch_bounds__(kFoldThreads)
k_fold_owned(LayerView B, const PeerLayer* __restrict__ peers,
             const unsigned long long* __restrict__ hkeys,
             const unsigned long long* __restrict__ hmask, const uint32_t* __restrict__ hbase,
             const uint32_t* __restrict__ mine, const uint32_t* __restrict__ slots,
             const uint32_t* __restrict__ counters, uint32_t list_cap, int blocks_before,
             unsigned long long* folded) {
  extern __shared__ __align__(16) unsigned char smem_raw[];
  uint4* t_d = reinterpret_cast<uint4*>(smem_raw);  // three planes of 4096 words
  uint4* t_w = t_d + kVoxelsPerBlock / 4;
  uint4* t_c = t_w + kVoxelsPerBlock / 4;
  __shared__ int s_slot, s_fresh;
  const uint32_t n = min(counters[0], list_cap);
  for (uint32_t i = blockIdx.x; i < n; i += gridDim.x) {
    const uint32_t e = mine[i];
    const unsigned long long key = hkeys[e];
    unsigned long long mask = hmask[e];
    const uint32_t base = hbase[e];
    // Block::mergeBlock skips a source block without data: is there one with data at all?
    bool any = false;
    {
      unsigned long long m = mask;
      for (int j = 0; m; ++j, m &= m - 1)
        any = any || peers[__ffsll(static_cast<long long>(m)) - 1].has_data[slots[base + j]] != 0;
    }
    __syncthreads();  // the previous block's tile has been written out
    if (!any) continue;
    if (threadIdx.x == 0) {
      const int he = B.insert_entry(key);
      s_slot = B.hash_vals[he];
      s_fresh = 0;
      if (s_slot >= 0) {
        // a slot claimed during this call holds a default-constructed block (the pool keeps
        // unclaimed slots in that state): nothing to read
        s_fresh = s_slot >= blocks_before;
        B.has_data[s_slot] = 1;
        B.updated[s_slot] = 1;
        atomicAdd(folded, static_cast<unsigned long long>(__popcll(mask)));
      }
    }
    __syncthreads();
    const int slot = s_slot;
    if (slot < 0) continue;  // pool exhausted: flagged by insert_entry
    uint4* dd = reinterpret_cast<uint4*>(B.dist_plane(slot));
    uint4* dw = reinterpret_cast<uint4*>(B.weight_plane(slot));
    uint4* dc = reinterpret_cast<uint4*>(B.color_plane(slot));
    if (s_fresh) {
      for (int q = threadIdx.x; q < kVoxelsPerBlock / 4; q += kFoldThreads) {
        t_d[q] = make_uint4(0u, 0u, 0u, 0u);
        t_w[q] = make_uint4(0u, 0u, 0u, 0u);
        t_c[q] = make_uint4(kDefaultColor, kDefaultColor, kDefaultColor, kDefaultColor);
      }
    } else {
      for (int q = threadIdx.x; q < kVoxelsPerBlock / 4; q += kFoldThreads) {
        t_d[q] = dd[q];
        t_w[q] = dw[q];
        t_c[q] = dc[q];
      }
    }
    for (int j = 0; mask; ++j, mask &= mask - 1) {  // ascending rank: the fold order is fixed
      const PeerLayer P = peers[__ffsll(static_cast<long long>(mask)) - 1];
      const uint32_t a = slots[base + j];
      if (!P.has_data[a]) continue;
      const uint4* sd =
          reinterpret_cast<const uint4*>(P.pool + static_cast<size_t>(a) * (3 * kVoxelsPerBlock));
      const uint4* sw = sd + kVoxelsPerBlock / 4;
      const uint4* sc = sw + kVoxelsPerBlock / 4;
      // each thread folds the same quads in every round: no synchronisation between sources
      for (int q = threadIdx.x; q < kVoxelsPerBlock / 4; q += kFoldThreads) {
        const uint4 ad = sd[q], aw = sw[q], ac = sc[q];
        const uint4 bd = t_d[q], bw = t_w[q], bc = t_c[q];
        VoxelState v0{__uint_as_float(bd.x), __uint_as_float(bw.x), bc.x};
        VoxelState v1{__uint_as_float(bd.y), __uint_as_float(bw.y), bc.y};
        VoxelState v2{__uint_as_float(bd.z), __uint_as_float(bw.z), bc.z};
        VoxelState v3{__uint_as_float(bd.w), __uint_as_float(bw.w), bc.w};
        merge_voxel(__uint_as_float(ad.x), __uint_as_float(aw.x), ac.x, v0);
        merge_voxel(__uint_as_float(ad.y), __uint_as_float(aw.y), ac.y, v1);
        merge_voxel(__uint_as_float(ad.z), __uint_as_float(aw.z), ac.z, v2);
        merge_voxel(__uint_as_float(ad.w), __uint_as_float(aw.w), ac.w, v3);
        t_d[q] = make_uint4(__float_as_uint(v0.d), __float_as_uint(v1.d), __float_as_uint(v2.d),
                            __float_as_uint(v3.d));
        t_w[q] = make_uint4(__float_as_uint(v0.w), __float_as_uint(v1.w), __float_as_uint(v2.w),
                            __float_as_uint(v3.w));
        t_c[q] = make_uint4(v0.c, v1.c, v2.c, v3.c);
      }
    }
    for (int q = threadIdx.x; q < kVoxelsPerBlock / 4; q += kFoldThreads) {
      dd[q] = t_d[q];
      dw[q] = t_w[q];
      dc[q] = t_c[q];
    }
  }
}

__global__ void k_publish_blocks(uint32_t* shared, int n) { shared[0] = static_cast<uint32_t>(n); }
__global__ void k_comm_overflow(const uint32_t* counters, int32_t* err) {
  if (counters[2]) atomicOr(err, kErrPoolFull);
}

// pointer -> (allocation base handle, offset): cudaMalloc may place small buffers inside a larger
// allocation, and an IPC handle always names the whole allocation
static int32_t ipc_of(const void* p, cudaIpcMemHandle_t* h, unsigned long long* off) {
  typedef int (*GetRange)(unsigned long long*, size_t*, unsigned long long);
  static GetRange get_range = nullptr;
  if (!get_range) {
    void* fn = nullptr;
    cudaDriverEntryPointQueryResult q;
    CG_CUDA(cudaGetDriverEntryPoint("cuMemGetAddressRange", &fn, cudaEnableDefault, &q));
    get_range = reinterpret_cast<GetRange>(fn);
    if (!get_range) {
      set_error("cuMemGetAddressRange is not available");
      return CG_ERR_CUDA;
    }
  }
  unsigned long long base = 0;
  size_t size = 0;
  if (get_range(&base, &size, reinterpret_cast<unsigned long long>(p)) != 0) {
    set_error("cuMemGetAddressRange failed");
    return CG_ERR_CUDA;
  }
  *off = reinterpret_cast<unsigned long long>(p) - base;
  CG_CUDA(cudaIpcGetMemHandle(h, reinterpret_cast<void*>(base)));
  return CG_OK;
}

static void release(cg_comm* c, Binding& b) {
  for (char* p : b.held) {
    for (size_t i = 0; i < c->maps.size(); ++i) {
      if (c->maps[i].p != p) continue;
      if (--c->maps[i].refs == 0) {
        cudaIpcCloseMemHandle(p);
        c->maps.erase(c->maps.begin() + static_cast<long>(i));
      }
      break;
    }
  }
  b.held.clear();
  b.serial = 0;
}

static void unbind(cg_comm* c) {
  for (Binding* b : {&c->partial, &c->owned}) {
    release(c, *b);
    if (b->shared) cudaFree(b->shared);
    if (b->d_peers) cudaFree(b->d_peers);
    b->shared = nullptr;
    b->d_peers = nullptr;
  }
  void* bufs[] = {c->hkeys, c->hmask, c->hbase, c->mine, c->slots, c->counters,
                  c->mkeys, c->mmask, c->mplanes, c->mcounters};
  for (void* p : bufs)
    if (p) cudaFree(p);
  c->hbase = c->mine = c->slots = c->counters = c->mcounters = nullptr;
  c->hkeys = c->hmask = c->mkeys = c->mmask = nullptr;
  c->mplanes = nullptr;
  c->hcap = c->list_cap = c->mcap = 0;
}

static int32_t barrier(cg_context* ctx) {
  cg_comm* c = ctx->comm;
  CG_NCCL(g_nccl.AllReduce(c->d_token, c->d_token, 1, ncclInt32, ncclSum, c->comm, ctx->stream));
  return CG_OK;
}

// the block key map of every layer of one role over all ranks: twice the blocks all ranks can hold
static size_t map_capacity(size_t max_blocks, int nranks) {
  size_t cap = 1024;
  while (cap < 2 * max_blocks * static_cast<size_t>(nranks)) cap <<= 1;
  return cap;
}

// All ranks call this with their own layer of one role (collective): IPC handles all-gathered, the
// layers checked against each other (same voxel size and max_blocks; every rank sees every record,
// so every rank rejects a mismatch), then the peers' buffers mapped.
static int32_t bind(cg_context* ctx, const cg_layer* layer, Binding& b, const char* who) {
  cg_comm* c = ctx->comm;
  release(c, b);
  cudaStream_t s = ctx->stream;
  const int R = c->nranks;
  if (!b.shared) CG_CUDA(cudaMalloc(&b.shared, 64));
  if (!b.d_peers) CG_CUDA(cudaMalloc(&b.d_peers, sizeof(PeerLayer) * R));
  CG_CUDA(cudaMemsetAsync(b.shared, 0, 64, s));
  IpcRecord mine;
  memset(&mine, 0, sizeof(mine));
  int32_t rc;
  if ((rc = ipc_of(layer->v.pool, &mine.pool, &mine.off_pool))) return rc;
  if ((rc = ipc_of(layer->v.block_keys, &mine.keys, &mine.off_keys))) return rc;
  if ((rc = ipc_of(layer->v.has_data, &mine.flags, &mine.off_flags))) return rc;
  if ((rc = ipc_of(b.shared, &mine.shared, &mine.off_shared))) return rc;
  mine.max_blocks = layer->max_blocks;
  mine.voxel_size = layer->v.voxel_size;
  void* d_all = nullptr;
  CG_CUDA(cudaMalloc(&d_all, sizeof(IpcRecord) * R));
  CG_CUDA(cudaMemcpyAsync(static_cast<char*>(d_all) + sizeof(IpcRecord) * c->rank, &mine,
                          sizeof(IpcRecord), cudaMemcpyHostToDevice, s));
  CG_NCCL(g_nccl.AllGather(static_cast<char*>(d_all) + sizeof(IpcRecord) * c->rank, d_all,
                           sizeof(IpcRecord), ncclInt8, c->comm, s));
  std::vector<IpcRecord> all(R);
  CG_CUDA(cudaMemcpyAsync(all.data(), d_all, sizeof(IpcRecord) * R, cudaMemcpyDeviceToHost, s));
  CG_CUDA(cudaStreamSynchronize(s));
  cudaFree(d_all);
  for (int r = 0; r < R; ++r) {
    if (all[r].max_blocks != layer->max_blocks || all[r].voxel_size != layer->v.voxel_size) {
      set_error("%s: rank %d's layer differs from rank %d's (max_blocks %llu / %zu, voxel size %g / %g)",
                who, r, c->rank, all[r].max_blocks, layer->max_blocks,
                static_cast<double>(all[r].voxel_size), static_cast<double>(layer->v.voxel_size));
      return CG_ERR_INVALID_ARG;
    }
  }
  std::vector<PeerLayer> peers(R);
  for (int r = 0; r < R; ++r) {
    if (r == c->rank) {
      peers[r] = PeerLayer{layer->v.pool, layer->v.block_keys, layer->v.has_data, b.shared};
      continue;
    }
    const cudaIpcMemHandle_t* hs[4] = {&all[r].pool, &all[r].keys, &all[r].flags, &all[r].shared};
    const unsigned long long offs[4] = {all[r].off_pool, all[r].off_keys, all[r].off_flags,
                                        all[r].off_shared};
    char* mapped[4] = {nullptr, nullptr, nullptr, nullptr};
    for (int k = 0; k < 4; ++k) {
      for (Mapping& m : c->maps) {
        if (m.rank == r && memcmp(&m.handle, hs[k], sizeof(cudaIpcMemHandle_t)) == 0) {
          ++m.refs;
          mapped[k] = m.p;
          break;
        }
      }
      if (!mapped[k]) {
        void* p = nullptr;
        const cudaError_t e = cudaIpcOpenMemHandle(&p, *hs[k], cudaIpcMemLazyEnablePeerAccess);
        if (e != cudaSuccess) {
          set_error("cudaIpcOpenMemHandle (rank %d's layer) failed: %s", r, cudaGetErrorString(e));
          return CG_ERR_CUDA;
        }
        ++c->maps_opened;
        mapped[k] = static_cast<char*>(p);
        c->maps.push_back(Mapping{r, *hs[k], mapped[k], 1});
      }
      b.held.push_back(mapped[k]);
    }
    peers[r] = PeerLayer{reinterpret_cast<const float*>(mapped[0] + offs[0]),
                         reinterpret_cast<const uint64_t*>(mapped[1] + offs[1]),
                         reinterpret_cast<const uint8_t*>(mapped[2] + offs[2]),
                         reinterpret_cast<const uint32_t*>(mapped[3] + offs[3])};
  }
  CG_CUDA(cudaMemcpyAsync(b.d_peers, peers.data(), sizeof(PeerLayer) * R, cudaMemcpyHostToDevice, s));
  CG_CUDA(cudaStreamSynchronize(s));
  b.serial = layer->serial;
  return CG_OK;
}

// the partial layer of cg_gather_global, with the holder map's scratch sized for it
static int32_t bind_partial(cg_context* ctx, const cg_layer* partial) {
  cg_comm* c = ctx->comm;
  const size_t list_cap = partial->max_blocks * static_cast<size_t>(c->nranks);
  const size_t hcap = map_capacity(partial->max_blocks, c->nranks);
  if (hcap != c->hcap || list_cap != c->list_cap) {
    void* bufs[] = {c->hkeys, c->hmask, c->hbase, c->mine, c->slots, c->counters};
    for (void* p : bufs)
      if (p) cudaFree(p);
    c->hkeys = c->hmask = nullptr;
    c->hbase = c->mine = c->slots = c->counters = nullptr;
    c->hcap = c->list_cap = 0;
    CG_CUDA(cudaMalloc(&c->hkeys, hcap * sizeof(unsigned long long)));
    CG_CUDA(cudaMalloc(&c->hmask, hcap * sizeof(unsigned long long)));
    CG_CUDA(cudaMalloc(&c->hbase, hcap * sizeof(uint32_t)));
    CG_CUDA(cudaMalloc(&c->mine, list_cap * sizeof(uint32_t)));
    CG_CUDA(cudaMalloc(&c->slots, list_cap * sizeof(uint32_t)));
    CG_CUDA(cudaMalloc(&c->counters, 4 * sizeof(uint32_t)));
    c->hcap = hcap;
    c->list_cap = list_cap;
  }
  return bind(ctx, partial, c->partial, "cg_gather_global");
}

// the owned layer of cg_layer_mesh_sharded, with the key map's scratch sized for it
static int32_t bind_owned(cg_context* ctx, const cg_layer* owned) {
  cg_comm* c = ctx->comm;
  const size_t mcap = map_capacity(owned->max_blocks, c->nranks);
  if (mcap != c->mcap) {
    void* bufs[] = {c->mkeys, c->mmask, c->mplanes, c->mcounters};
    for (void* p : bufs)
      if (p) cudaFree(p);
    c->mkeys = c->mmask = nullptr;
    c->mplanes = nullptr;
    c->mcounters = nullptr;
    c->mcap = 0;
    CG_CUDA(cudaMalloc(&c->mkeys, mcap * sizeof(unsigned long long)));
    CG_CUDA(cudaMalloc(&c->mmask, mcap * sizeof(unsigned long long)));
    CG_CUDA(cudaMalloc(&c->mplanes, mcap * sizeof(const float*)));
    CG_CUDA(cudaMalloc(&c->mcounters, 4 * sizeof(uint32_t)));
    c->mcap = mcap;
  }
  return bind(ctx, owned, c->owned, "cg_layer_mesh_sharded");
}

int32_t sharded_mesh_open(const cg_layer* owned, unsigned long long* dup_key, ShardedBlocks* out) {
  cg_context* ctx = owned->ctx;
  cg_comm* c = ctx->comm;
  cudaStream_t s = ctx->stream;
  int32_t rc;
  if (c->owned.serial != owned->serial && (rc = bind_owned(ctx, owned))) return rc;
  ctx->own_launches += 2;
  k_publish_blocks<<<1, 1, 0, s>>>(c->owned.shared, static_cast<int>(owned->num_blocks));
  CG_CUDA(cudaMemsetAsync(c->mkeys, 0xFF, c->mcap * sizeof(unsigned long long), s));
  CG_CUDA(cudaMemsetAsync(c->mmask, 0, c->mcap * sizeof(unsigned long long), s));
  CG_CUDA(cudaMemsetAsync(c->mcounters, 0, 4 * sizeof(uint32_t), s));
  CG_CUDA(cudaMemsetAsync(dup_key, 0xFF, sizeof(unsigned long long), s));
  // every rank's owned layer is complete and its block count published (stream-ordered)
  if ((rc = barrier(ctx))) return rc;
  const uint32_t cap_mask = static_cast<uint32_t>(c->mcap - 1);
  const dim3 per_rank(static_cast<unsigned>(ctx->num_sms), static_cast<unsigned>(c->nranks));
  k_build_holders<<<per_rank, 256, 0, s>>>(c->owned.d_peers, c->mkeys, c->mmask, cap_mask,
                                           c->mcounters, c->mplanes, dup_key);
  CG_CUDA(cudaGetLastError());
  *out = ShardedBlocks{c->mkeys, c->mplanes, cap_mask};
  return CG_OK;
}

int32_t sharded_mesh_close(cg_context* ctx) { return barrier(ctx); }

}  // namespace cg

using namespace cg;

extern "C" {

int32_t cg_comm_get_unique_id(uint8_t id[CG_COMM_ID_BYTES]) {
  if (!id) return CG_ERR_INVALID_ARG;
  int32_t rc = load_nccl();
  if (rc) return rc;
  ncclUniqueId u;
  CG_NCCL(g_nccl.GetUniqueId(&u));
  memcpy(id, u.internal, CG_COMM_ID_BYTES);
  return CG_OK;
}

int32_t cg_comm_init(cg_context* ctx, const uint8_t id[CG_COMM_ID_BYTES], int32_t rank,
                     int32_t nranks) {
  if (!ctx || !id || nranks < 1 || nranks > kMaxRanks || rank < 0 || rank >= nranks) {
    set_error("cg_comm_init: invalid argument");
    return CG_ERR_INVALID_ARG;
  }
  if (ctx->comm) {
    set_error("cg_comm_init: the context already has a communicator");
    return CG_ERR_INVALID_ARG;
  }
  int32_t rc = load_nccl();
  if (rc) return rc;
  CG_CUDA(cudaSetDevice(ctx->device));
  cg_comm* c = new cg_comm;
  c->rank = rank;
  c->nranks = nranks;
  ncclUniqueId u;
  memcpy(u.internal, id, CG_COMM_ID_BYTES);
  const int r = g_nccl.CommInitRank(&c->comm, nranks, u, rank);
  if (r != ncclSuccess) {
    set_error("ncclCommInitRank failed: %s", g_nccl.GetErrorString(r));
    delete c;
    return CG_ERR_CUDA;
  }
  if (cudaMalloc(&c->d_token, sizeof(int)) != cudaSuccess) {
    set_error("cg_comm_init: out of device memory");
    return CG_ERR_CUDA;
  }
  cudaMemset(c->d_token, 0, sizeof(int));
  ctx->comm = c;
  return CG_OK;
}

int32_t cg_comm_destroy(cg_context* ctx) {
  if (!ctx) return CG_ERR_INVALID_ARG;
  cg_comm* c = ctx->comm;
  if (!c) return CG_OK;
  cudaSetDevice(ctx->device);
  cudaStreamSynchronize(ctx->stream);
  unbind(c);
  if (c->d_token) cudaFree(c->d_token);
  if (c->comm) g_nccl.CommDestroy(c->comm);
  delete c;
  ctx->comm = nullptr;
  return CG_OK;
}

int32_t cg_comm_peer_mappings(const cg_context* ctx, uint64_t* opened_total, uint64_t* open_now) {
  if (!ctx || !ctx->comm) {
    set_error("cg_comm_peer_mappings: the context has no communicator");
    return CG_ERR_INVALID_ARG;
  }
  if (opened_total) *opened_total = ctx->comm->maps_opened;
  if (open_now) *open_now = ctx->comm->maps.size();
  return CG_OK;
}

int32_t cg_gather_global(const cg_layer* partial, cg_layer* owned, uint64_t* blocks_folded) {
  if (!partial || !owned || partial->ctx != owned->ctx || partial == owned) {
    set_error("cg_gather_global: partial and owned must be two layers of one context");
    return CG_ERR_INVALID_ARG;
  }
  cg_context* ctx = owned->ctx;
  cg_comm* c = ctx->comm;
  if (!c) {
    set_error("cg_gather_global: call cg_comm_init first");
    return CG_ERR_INVALID_ARG;
  }
  if (partial->v.voxel_size != owned->v.voxel_size) {
    set_error("cg_gather_global: the layers' voxel sizes differ");
    return CG_ERR_INVALID_ARG;
  }
  CG_CUDA(cudaSetDevice(ctx->device));
  cudaStream_t s = ctx->stream;
  int32_t rc;
  if (c->partial.serial != partial->serial && (rc = bind_partial(ctx, partial))) return rc;
  // CG_TRACE_COMM=1: per-phase device times of the exchange on stderr (diagnostics only)
  static const bool trace = getenv("CG_TRACE_COMM") != nullptr;
  cudaEvent_t tev[6] = {};
  int tn = 0;
  auto mark = [&]() {
    if (trace && tn < 6) {
      cudaEventCreate(&tev[tn]);
      cudaEventRecord(tev[tn++], s);
    }
  };
  mark();
  const int R = c->nranks;
  const uint32_t hmask_cap = static_cast<uint32_t>(c->hcap - 1);
  const uint32_t list_cap = static_cast<uint32_t>(std::min<size_t>(c->list_cap, 0xFFFFFFF0u));
  ctx->own_launches += 6;
  k_publish_blocks<<<1, 1, 0, s>>>(c->partial.shared, static_cast<int>(partial->num_blocks));
  CG_CUDA(cudaMemsetAsync(c->hkeys, 0xFF, c->hcap * sizeof(unsigned long long), s));
  CG_CUDA(cudaMemsetAsync(c->hmask, 0, c->hcap * sizeof(unsigned long long), s));
  CG_CUDA(cudaMemsetAsync(c->counters, 0, 4 * sizeof(uint32_t), s));
  CG_CUDA(cudaMemsetAsync(&ctx->d_counters->blocks_out, 0, sizeof(unsigned long long), s));
  // every rank's partial layer is complete and its block count published (stream-ordered)
  if ((rc = barrier(ctx))) return rc;
  mark();
  const dim3 per_rank(static_cast<unsigned>(ctx->num_sms), static_cast<unsigned>(R));
  k_build_holders<<<per_rank, 256, 0, s>>>(c->partial.d_peers, c->hkeys, c->hmask, hmask_cap,
                                           c->counters, nullptr, nullptr);
  k_list_owned<<<ctx->num_sms * 4, 256, 0, s>>>(c->hkeys, c->hmask, static_cast<uint32_t>(c->hcap),
                                                c->rank, c->hbase, c->mine, list_cap, c->counters);
  k_holder_slots<<<per_rank, 256, 0, s>>>(c->partial.d_peers, c->hkeys, c->hmask, c->hbase, hmask_cap,
                                          c->rank, c->slots, list_cap);
  mark();
  const size_t smem = 3 * kVoxelsPerBlock * sizeof(uint32_t);
  static bool attr_set[64] = {};
  if (ctx->device < 0 || ctx->device >= 64 || !attr_set[ctx->device]) {
    CG_CUDA(cudaFuncSetAttribute(k_fold_owned, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                 static_cast<int>(smem)));
    if (ctx->device >= 0 && ctx->device < 64) attr_set[ctx->device] = true;
  }
  k_fold_owned<<<ctx->num_sms * 4, kFoldThreads, smem, s>>>(
      owned->v, c->partial.d_peers, c->hkeys, c->hmask, c->hbase, c->mine, c->slots, c->counters, list_cap,
      static_cast<int>(owned->num_blocks), &ctx->d_counters->blocks_out);
  k_comm_overflow<<<1, 1, 0, s>>>(c->counters, owned->v.err);
  mark();
  // nobody clears or refills its partial layer while a peer still reads it
  if ((rc = barrier(ctx))) return rc;
  mark();
  CallCounters cc;
  rc = finish_call(owned, &cc);
  if (trace && tn == 5) {
    float t[4];
    for (int i = 0; i < 4; ++i) cudaEventElapsedTime(&t[i], tev[i], tev[i + 1]);
    fprintf(stderr, "[cg comm rank %d] reset+barrier %.3f  holders+list+slots %.3f  fold %.3f  barrier %.3f ms "
            "(partial %lld blocks, hash %zu)\n", c->rank, t[0], t[1], t[2], t[3],
            static_cast<long long>(partial->num_blocks), c->hcap);
  }
  for (int i = 0; i < tn; ++i) cudaEventDestroy(tev[i]);
  if (blocks_folded) *blocks_folded = cc.blocks_out;
  return rc;
}

int32_t cg_project_submaps_sharded(const cg_layer* const* submaps, const float* poses,
                                   size_t num_submaps, cg_layer* partial, cg_layer* owned,
                                   cg_merge_stats* stats) {
  if (!partial || !owned) return CG_ERR_INVALID_ARG;
  int32_t rc = cg_layer_clear(partial);
  if (rc) return rc;
  if (num_submaps) {
    rc = cg_project_submaps(submaps, poses, num_submaps, partial, stats);
    if (rc) return rc;
  } else if (stats) {
    memset(stats, 0, sizeof(*stats));
  }
  return cg_gather_global(partial, owned, nullptr);
}

}  // extern "C"
