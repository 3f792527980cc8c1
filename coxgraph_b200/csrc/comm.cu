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
// synchronisation between listing, exchange and fold.  For the gather and the sharded mesh, NCCL
// (loaded at run time from libnccl.so.2, the one torch has loaded if there is one) is the bootstrap
// and the barrier only: unique id -> communicator, one all-gather of the IPC handles when a layer
// is bound, and a one-word all-reduce on the stream before and after the kernels (all partial
// layers complete / all peers done reading).  The fold order is fixed, so the result is
// deterministic and equal to the packed exchange of exchange.cu (hash owner, NCCL all-to-all)
// block for block.
//
// cg_layer_mesh_sharded (mesh.cu) meshes the owned layers where they lie.  Its collective half is
// here: the owned layer is bound like the partial one (its own binding, so alternating gather and
// mesh calls map nothing again), and k_build_holders, run over every rank's owned keys, also
// records where each block's planes are.  The mesh kernel resolves the one-block halo (the +x/+y/+z
// neighbours and a vertex's colour block) through that map and reads the peer's planes over
// NVLink; a key two ranks hold is found while the map is built.
//
// cg_mesh_gather_sharded moves those block meshes to one root rank, where they become the mesh
// cg_layer_mesh leaves for the union of the owned layers.  The mesh buffers are per-call scratch
// that grows, so they are not mapped over IPC: one all-gather of a few words per rank (block and
// vertex counts, what the rank retains, the root) sizes the root's buffers, one all-reduce is the
// go/no-go, and NCCL point-to-point sends move each peer's block indices, vertex ranges, vertices,
// normals and colours into the root's staging buffer.  On the root, k_gather_keys + a radix sort
// put every rank's blocks in the packed-key order of sort_blocks, a scan of the per-block vertex
// counts gives vertex_begin, and k_place_blocks copies each block's range into fresh buffers that
// then replace the root's own share.
#include <cub/cub.cuh>
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
  int (*Send)(const void*, size_t, int, int, ncclComm_t, cudaStream_t) = nullptr;
  int (*Recv)(void*, size_t, int, int, ncclComm_t, cudaStream_t) = nullptr;
  int (*GroupStart)() = nullptr;
  int (*GroupEnd)() = nullptr;
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
  n.Send = reinterpret_cast<decltype(n.Send)>(dlsym(h, "ncclSend"));
  n.Recv = reinterpret_cast<decltype(n.Recv)>(dlsym(h, "ncclRecv"));
  n.GroupStart = reinterpret_cast<decltype(n.GroupStart)>(dlsym(h, "ncclGroupStart"));
  n.GroupEnd = reinterpret_cast<decltype(n.GroupEnd)>(dlsym(h, "ncclGroupEnd"));
  n.GetErrorString = reinterpret_cast<decltype(n.GetErrorString)>(dlsym(h, "ncclGetErrorString"));
  if (!n.GetUniqueId || !n.CommInitRank || !n.CommDestroy || !n.AllReduce || !n.AllGather ||
      !n.Send || !n.Recv || !n.GroupStart || !n.GroupEnd || !n.GetErrorString) {
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
  const uint32_t* shared;  // [0] number of blocks of the layer (written per call), see Binding
  const uint64_t* dirty_keys;  // partial role: the keys cg_reproject_submaps_sharded publishes
};
constexpr int kMaxRanks = 64;

struct IpcRecord {  // one per rank, all-gathered
  cudaIpcMemHandle_t pool, keys, flags, shared, dirty;
  unsigned long long off_pool, off_keys, off_flags, off_shared, off_dirty;  // pointer - allocation base
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
  // peer-visible words, written per call: [0] blocks of this rank's layer; the partial role's
  // cg_reproject_submaps_sharded also publishes [1] blocks of the owned layer, [2] dirty keys and
  // [3] the full-rebuild fraction (float bits; rank 0's is the one every rank uses)
  uint32_t* shared = nullptr;
  uint64_t* dirty = nullptr;      // partial role: peer-visible dirty keys (2 x max_blocks)
  uint32_t dirty_cap = 0;
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
  // cg_reproject_submaps_sharded: the union D of every rank's dirty keys (scratch, lazily sized)
  cg::DevBuf dset;
  size_t dcap = 0;
  uint32_t* dcounters = nullptr;      // [0] |D|, [1] owned blocks of all ranks, [2] overflow, [3] fraction
  // the holder map (scratch, rebuilt every call): block key -> set of ranks holding the block,
  // hcap entries of hkeys / hmask / hbase
  cg::DevBuf hkeys, hmask;
  cg::DevBuf hbase;                   // owned entries: first element of the block's slot list
  cg::DevBuf mine;                    // [list_cap] entries this rank owns
  cg::DevBuf slots;                   // [list_cap] pool slots of the holders' copies, per owned block
  cg::DevBuf counters;                // [0] owned entries, [1] slot list cursor, [2] overflow
  size_t hcap = 0, list_cap = 0;
  // the key map of cg_layer_mesh_sharded over every rank's owned layer (rebuilt every call), mcap
  // entries of mkeys / mmask / mplanes
  cg::DevBuf mkeys, mmask;
  cg::DevBuf mplanes;                 // the block's distance plane in its holder's pool
  cg::DevBuf mcounters;               // k_build_holders' words ([2] overflow: cannot happen)
  size_t mcap = 0;
  cg::DevBuf gwords;                  // cg_mesh_gather_sharded: every rank's GatherWords
};

namespace cg {

// the owner of a block: one of its holders, picked by a hash of the block index
__device__ __forceinline__ int pick_owner(unsigned long long key, unsigned long long mask) {
  int n = static_cast<int>(owner_pick(key, static_cast<uint32_t>(__popcll(mask))));
  unsigned long long m = mask;
  while (n-- > 0) m &= m - 1;
  return __ffsll(static_cast<long long>(m)) - 1;
}

// Every block key of every rank's layer (read through the peer mappings) enters the map with its
// rank's bit.  Grid y = rank.  With `planes` (the key map of cg_layer_mesh_sharded) the entry also
// records where the block's planes are, and a key that reaches an entry another rank has already
// marked is held twice: the smallest such key goes to *dup_key.  With `filter_keys` (a key set of
// filter_mask + 1 entries, cg_reproject_submaps_sharded) only the keys in it enter the map.
__global__ void k_build_holders(const PeerLayer* __restrict__ peers, KeySet map,
                                unsigned long long* hmask, uint32_t* counters,
                                const float** planes, unsigned long long* dup_key,
                                const unsigned long long* __restrict__ filter_keys,
                                uint32_t filter_mask) {
  const KeyLookup filter{filter_keys, filter_mask};
  const int r = blockIdx.y;
  const PeerLayer P = peers[r];
  const uint32_t n = P.shared[0];
  for (uint32_t i = blockIdx.x * blockDim.x + threadIdx.x; i < n; i += gridDim.x * blockDim.x) {
    const unsigned long long key = P.block_keys[i];
    if (filter.keys && !filter.contains(key)) continue;
    const int h = map.insert(key);
    if (h < 0) {  // cannot happen: the map holds every block of every rank
      atomicExch(&counters[2], 1u);
      return;
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
                               uint32_t* __restrict__ slots, uint32_t slots_cap,
                               const unsigned long long* __restrict__ filter_keys,
                               uint32_t filter_mask) {
  const KeyLookup map{hkeys, hcap_mask}, filter{filter_keys, filter_mask};
  const int r = blockIdx.y;
  const PeerLayer P = peers[r];
  const uint32_t n = P.shared[0];
  for (uint32_t i = blockIdx.x * blockDim.x + threadIdx.x; i < n; i += gridDim.x * blockDim.x) {
    const unsigned long long key = P.block_keys[i];
    if (filter.keys && !filter.contains(key)) continue;
    const int e = map.find(key);
    if (e < 0) continue;  // not in the map: k_build_holders raised its overflow word
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
// cg_reproject_submaps_sharded: every rank's published dirty keys (read through the peer mappings)
// enter the set D; counters [0] |D|, [1] owned blocks of all ranks, [2] a rank published more keys
// than its buffer holds, [3] rank 0's full-rebuild fraction.  Grid y = rank.
__global__ void k_union_dirty(const PeerLayer* __restrict__ peers, uint32_t dirty_cap, KeySet set,
                              uint32_t* counters) {
  const int r = blockIdx.y;
  const PeerLayer P = peers[r];
  const uint32_t published = P.shared[2];
  if (blockIdx.x == 0 && threadIdx.x == 0) {
    atomicAdd(&counters[1], P.shared[1]);
    if (published > dirty_cap) atomicExch(&counters[2], 1u);
    if (r == 0) counters[3] = P.shared[3];
  }
  const uint32_t n = min(published, dirty_cap);
  for (uint32_t i = blockIdx.x * blockDim.x + threadIdx.x; i < n; i += gridDim.x * blockDim.x) {
    bool inserted;
    set.insert(P.dirty_keys[i], &inserted);
    if (inserted) atomicAdd(&counters[0], 1u);
  }
}
__global__ void k_publish_words(uint32_t* shared, uint32_t partial_blocks, uint32_t owned_blocks,
                                uint32_t fraction_bits) {
  shared[0] = partial_blocks;
  shared[1] = owned_blocks;
  shared[3] = fraction_bits;
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
    if (b->dirty) cudaFree(b->dirty);
    if (b->d_peers) cudaFree(b->d_peers);
    b->shared = nullptr;
    b->dirty = nullptr;
    b->dirty_cap = 0;
    b->d_peers = nullptr;
  }
  c->dset.release();
  c->dcap = 0;
  if (c->dcounters) cudaFree(c->dcounters);
  c->dcounters = nullptr;
  for (DevBuf* d : {&c->hkeys, &c->hmask, &c->hbase, &c->mine, &c->slots, &c->counters, &c->mkeys,
                    &c->mmask, &c->mplanes, &c->mcounters, &c->gwords})
    d->release();
  c->hcap = c->list_cap = c->mcap = 0;
}

static int32_t barrier(cg_context* ctx) {
  cg_comm* c = ctx->comm;
  CG_NCCL(g_nccl.AllReduce(c->d_token, c->d_token, 1, ncclInt32, ncclSum, c->comm, ctx->stream));
  return CG_OK;
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
  if (b.dirty && (rc = ipc_of(b.dirty, &mine.dirty, &mine.off_dirty))) return rc;
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
      peers[r] = PeerLayer{layer->v.pool, layer->v.block_keys, layer->v.has_data, b.shared, b.dirty};
      continue;
    }
    const cudaIpcMemHandle_t* hs[5] = {&all[r].pool, &all[r].keys, &all[r].flags, &all[r].shared,
                                       &all[r].dirty};
    const unsigned long long offs[5] = {all[r].off_pool, all[r].off_keys, all[r].off_flags,
                                        all[r].off_shared, all[r].off_dirty};
    char* mapped[5] = {nullptr, nullptr, nullptr, nullptr, nullptr};
    for (int k = 0; k < (b.dirty ? 5 : 4); ++k) {
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
                         reinterpret_cast<const uint32_t*>(mapped[3] + offs[3]),
                         b.dirty ? reinterpret_cast<const uint64_t*>(mapped[4] + offs[4]) : nullptr};
  }
  CG_CUDA(cudaMemcpyAsync(b.d_peers, peers.data(), sizeof(PeerLayer) * R, cudaMemcpyHostToDevice, s));
  CG_CUDA(cudaStreamSynchronize(s));
  b.serial = layer->serial;
  return CG_OK;
}

// the partial layer of cg_gather_global, with the holder map's scratch sized for it (a key map
// over every rank's blocks)
static int32_t bind_partial(cg_context* ctx, const cg_layer* partial) {
  cg_comm* c = ctx->comm;
  release(c, c->partial);  // nothing uses the binding until bind() has made it again
  c->list_cap = partial->max_blocks * static_cast<size_t>(c->nranks);
  c->hcap = key_set_capacity(c->list_cap, 1024);
  CG_CUDA(c->hkeys.reserve(c->hcap * sizeof(unsigned long long)));
  CG_CUDA(c->hmask.reserve(c->hcap * sizeof(unsigned long long)));
  CG_CUDA(c->hbase.reserve(c->hcap * sizeof(uint32_t)));
  CG_CUDA(c->mine.reserve(c->list_cap * sizeof(uint32_t)));
  CG_CUDA(c->slots.reserve(c->list_cap * sizeof(uint32_t)));
  CG_CUDA(c->counters.reserve(4 * sizeof(uint32_t)));
  // the dirty keys of cg_reproject_submaps_sharded: the partial layer's blocks before and after a
  // call, so at most twice its pool
  const uint32_t dirty_cap = static_cast<uint32_t>(std::min<size_t>(2 * partial->max_blocks, 0xFFFFFFF0u));
  if (dirty_cap != c->partial.dirty_cap) {
    if (c->partial.dirty) cudaFree(c->partial.dirty);
    c->partial.dirty = nullptr;
    c->partial.dirty_cap = 0;
    CG_CUDA(cudaMalloc(&c->partial.dirty, dirty_cap * sizeof(uint64_t)));
    c->partial.dirty_cap = dirty_cap;
  }
  return bind(ctx, partial, c->partial, "cg_gather_global");
}

// the owned layer of cg_layer_mesh_sharded, with the key map's scratch sized for it
static int32_t bind_owned(cg_context* ctx, const cg_layer* owned) {
  cg_comm* c = ctx->comm;
  release(c, c->owned);  // nothing uses the binding until bind() has made it again
  c->mcap = key_set_capacity(owned->max_blocks * static_cast<size_t>(c->nranks), 1024);
  CG_CUDA(c->mkeys.reserve(c->mcap * sizeof(unsigned long long)));
  CG_CUDA(c->mmask.reserve(c->mcap * sizeof(unsigned long long)));
  CG_CUDA(c->mplanes.reserve(c->mcap * sizeof(const float*)));
  CG_CUDA(c->mcounters.reserve(4 * sizeof(uint32_t)));
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
  CG_CUDA(cudaMemsetAsync(c->mkeys.p, 0xFF, c->mcap * sizeof(unsigned long long), s));
  CG_CUDA(cudaMemsetAsync(c->mmask.p, 0, c->mcap * sizeof(unsigned long long), s));
  CG_CUDA(cudaMemsetAsync(c->mcounters.p, 0, 4 * sizeof(uint32_t), s));
  CG_CUDA(cudaMemsetAsync(dup_key, 0xFF, sizeof(unsigned long long), s));
  // every rank's owned layer is complete and its block count published (stream-ordered)
  if ((rc = barrier(ctx))) return rc;
  const KeySet map{c->mkeys.as<unsigned long long>(), static_cast<uint32_t>(c->mcap - 1)};
  const dim3 per_rank(static_cast<unsigned>(ctx->num_sms), static_cast<unsigned>(c->nranks));
  k_build_holders<<<per_rank, 256, 0, s>>>(c->owned.d_peers, map, c->mmask.as<unsigned long long>(),
                                           c->mcounters.as<uint32_t>(), c->mplanes.as<const float*>(),
                                           dup_key, nullptr, 0);
  CG_CUDA(cudaGetLastError());
  *out = ShardedBlocks{KeyLookup{map.keys, map.mask}, c->mplanes.as<const float*>()};
  return CG_OK;
}

int32_t sharded_mesh_close(cg_context* ctx) { return barrier(ctx); }

// The holder map of the fold, cleared (before the opening barrier) and built over every rank's
// partial layer; with `filter` (cg_reproject_submaps_sharded) over the blocks whose keys are in it.
static int32_t reset_holders(cg_context* ctx) {
  cg_comm* c = ctx->comm;
  cudaStream_t s = ctx->stream;
  CG_CUDA(cudaMemsetAsync(c->hkeys.p, 0xFF, c->hcap * sizeof(unsigned long long), s));
  CG_CUDA(cudaMemsetAsync(c->hmask.p, 0, c->hcap * sizeof(unsigned long long), s));
  CG_CUDA(cudaMemsetAsync(c->counters.p, 0, 4 * sizeof(uint32_t), s));
  CG_CUDA(cudaMemsetAsync(&ctx->d_counters->blocks_out, 0, sizeof(unsigned long long), s));
  return CG_OK;
}
static uint32_t fold_list_cap(const cg_comm* c) {
  return static_cast<uint32_t>(std::min<size_t>(c->list_cap, 0xFFFFFFF0u));
}
static void list_holders(cg_context* ctx, KeyLookup filter) {
  cg_comm* c = ctx->comm;
  cudaStream_t s = ctx->stream;
  const uint32_t list_cap = fold_list_cap(c);
  const KeySet map{c->hkeys.as<unsigned long long>(), static_cast<uint32_t>(c->hcap - 1)};
  unsigned long long* hmask = c->hmask.as<unsigned long long>();
  uint32_t* hbase = c->hbase.as<uint32_t>();
  uint32_t* counters = c->counters.as<uint32_t>();
  ctx->own_launches += 3;
  const dim3 per_rank(static_cast<unsigned>(ctx->num_sms), static_cast<unsigned>(c->nranks));
  k_build_holders<<<per_rank, 256, 0, s>>>(c->partial.d_peers, map, hmask, counters, nullptr,
                                           nullptr, filter.keys, filter.mask);
  k_list_owned<<<ctx->num_sms * 4, 256, 0, s>>>(map.keys, hmask, static_cast<uint32_t>(c->hcap),
                                                c->rank, hbase, c->mine.as<uint32_t>(), list_cap,
                                                counters);
  k_holder_slots<<<per_rank, 256, 0, s>>>(c->partial.d_peers, map.keys, hmask, hbase, map.mask,
                                          c->rank, c->slots.as<uint32_t>(), list_cap, filter.keys,
                                          filter.mask);
}
// every block the holder map gives this rank, folded into `owned` (blocks the layer holds are
// read as they are: fresh, or reset by cg_reproject_submaps_sharded)
static int32_t fold_owned(cg_context* ctx, cg_layer* owned) {
  cg_comm* c = ctx->comm;
  cudaStream_t s = ctx->stream;
  constexpr size_t smem = 3 * kVoxelsPerBlock * sizeof(uint32_t);
  CG_CUDA(allow_dynamic_smem<k_fold_owned>(ctx->device, smem));
  ctx->own_launches += 2;
  k_fold_owned<<<ctx->num_sms * 4, kFoldThreads, smem, s>>>(
      owned->v, c->partial.d_peers, c->hkeys.as<unsigned long long>(),
      c->hmask.as<unsigned long long>(), c->hbase.as<uint32_t>(), c->mine.as<uint32_t>(),
      c->slots.as<uint32_t>(), c->counters.as<uint32_t>(), fold_list_cap(c),
      static_cast<int>(owned->num_blocks), &ctx->d_counters->blocks_out);
  k_comm_overflow<<<1, 1, 0, s>>>(c->counters.as<uint32_t>(), owned->v.err);
  CG_CUDA(cudaGetLastError());
  return CG_OK;
}

// ---- cg_mesh_gather_sharded
// What every rank tells the others in the opening all-gather.
struct GatherWords {
  unsigned long long blocks, vertices;  // the retained mesh
  unsigned long long kind, calls;       // cg_context::mc_kind, mc_sharded_calls
  long long root;
};
// One rank's block meshes as the root reads them: its own retained buffers, or the regions of
// mg_in a peer's sends landed in.  Block b of the rank is block first + b of the concatenation.
struct MeshSource {
  const int32_t* idx;     // [3 blocks] block indices, (z, y, x) order
  const uint32_t* begin;  // [blocks + 1] vertex ranges
  const uint32_t* vertices;
  const uint32_t* normals;
  const uint32_t* colors;
  uint32_t blocks, first;
};
// every rank's block keys, with (rank << 32 | block) as payload.  Grid y = rank.
__global__ void k_gather_keys(const MeshSource* __restrict__ src, unsigned long long* __restrict__ keys,
                              unsigned long long* __restrict__ vals) {
  const int r = blockIdx.y;
  const MeshSource S = src[r];
  for (uint32_t b = blockIdx.x * blockDim.x + threadIdx.x; b < S.blocks; b += gridDim.x * blockDim.x) {
    keys[S.first + b] = pack_block_key(S.idx[3 * b], S.idx[3 * b + 1], S.idx[3 * b + 2]);
    vals[S.first + b] = (static_cast<unsigned long long>(r) << 32) | b;
  }
}
// vertex count of every block in sorted order, and a 0 behind the last (for the exclusive scan)
__global__ void k_gather_counts(const MeshSource* __restrict__ src,
                                const unsigned long long* __restrict__ vals, uint32_t n,
                                uint32_t* __restrict__ counts) {
  for (uint32_t i = blockIdx.x * blockDim.x + threadIdx.x; i <= n; i += gridDim.x * blockDim.x) {
    uint32_t k = 0;
    if (i < n) {
      const unsigned long long p = vals[i];
      const uint32_t* begin = src[p >> 32].begin;
      const uint32_t b = static_cast<uint32_t>(p);
      k = begin[b + 1] - begin[b];
    }
    counts[i] = k;
  }
}
// n words, one warp: 16-byte accesses when source and destination share their alignment
__device__ __forceinline__ void warp_copy(uint32_t* __restrict__ d, const uint32_t* __restrict__ s,
                                          uint32_t n, int lane) {
  if (((reinterpret_cast<uintptr_t>(d) ^ reinterpret_cast<uintptr_t>(s)) & 15u) == 0) {
    const uint32_t head = min(n, static_cast<uint32_t>(((16u - (reinterpret_cast<uintptr_t>(d) & 15u)) & 15u) >> 2));
    if (lane < static_cast<int>(head)) d[lane] = s[lane];
    d += head;
    s += head;
    n -= head;
    const uint32_t quads = n >> 2;
    for (uint32_t q = lane; q < quads; q += 32)
      reinterpret_cast<uint4*>(d)[q] = reinterpret_cast<const uint4*>(s)[q];
    const uint32_t tail = n & 3u;
    if (lane < static_cast<int>(tail)) d[4 * quads + lane] = s[4 * quads + lane];
  } else {
    for (uint32_t k = lane; k < n; k += 32) d[k] = s[k];
  }
}
// one warp per block in sorted order: its index and its vertex range (vertices, normals, colours)
// go to their place in the gathered mesh
constexpr int kPlaceThreads = 256;
__global__ void __launch_bounds__(kPlaceThreads)
k_place_blocks(const MeshSource* __restrict__ src, const unsigned long long* __restrict__ vals,
               const uint32_t* __restrict__ begin, uint32_t n, int32_t* __restrict__ idx,
               uint32_t* __restrict__ vertices, uint32_t* __restrict__ normals,
               uint32_t* __restrict__ colors) {
  const int lane = threadIdx.x & 31;
  const uint32_t warps = gridDim.x * (kPlaceThreads / 32);
  for (uint32_t i = blockIdx.x * (kPlaceThreads / 32) + (threadIdx.x >> 5); i < n; i += warps) {
    const unsigned long long p = vals[i];
    const MeshSource& S = src[p >> 32];
    const uint32_t b = static_cast<uint32_t>(p);
    const uint32_t lo = S.begin[b], k = S.begin[b + 1] - lo, at = begin[i];
    if (lane < 3) idx[3 * static_cast<size_t>(i) + lane] = S.idx[3 * static_cast<size_t>(b) + lane];
    warp_copy(vertices + 3 * static_cast<size_t>(at), S.vertices + 3 * static_cast<size_t>(lo), 3 * k, lane);
    warp_copy(normals + 3 * static_cast<size_t>(at), S.normals + 3 * static_cast<size_t>(lo), 3 * k, lane);
    warp_copy(colors + at, S.colors + lo, k, lane);
  }
}

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
  ctx->own_launches += 1;
  k_publish_blocks<<<1, 1, 0, s>>>(c->partial.shared, static_cast<int>(partial->num_blocks));
  if ((rc = reset_holders(ctx))) return rc;
  // every rank's partial layer is complete and its block count published (stream-ordered)
  if ((rc = barrier(ctx))) return rc;
  mark();
  list_holders(ctx, KeyLookup{});
  mark();
  if ((rc = fold_owned(ctx, owned))) return rc;
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

// ---- cg_reproject_submaps_sharded (DESIGN.md §5): the local re-projection of every rank's
// partial layer, then a fold of only the blocks whose holders or copies may have changed.
// The opening barrier carries a status word: one 8-bit count per failure kind, summed over the
// ranks, so that every rank knows whether (and how) some rank's local step failed.
static uint32_t status_bits(int32_t rc) {
  if (rc == CG_OK) return 0;
  const int field = rc == CG_ERR_INVALID_ARG ? 0 : rc == CG_ERR_OUT_OF_RANGE ? 1 : rc == CG_ERR_POOL_FULL ? 2 : 3;
  return 1u << (8 * field);
}
static int32_t status_of(uint32_t word) {  // the most severe failure a rank reported
  const int32_t kinds[4] = {CG_ERR_INVALID_ARG, CG_ERR_OUT_OF_RANGE, CG_ERR_POOL_FULL, CG_ERR_CUDA};
  for (int f = 3; f >= 0; --f)
    if ((word >> (8 * f)) & 0xFFu) return kinds[f];
  return CG_OK;
}
// A barrier that carries every rank's status_bits(local), summed into *word (one host
// synchronisation).
static int32_t status_barrier(cg_context* ctx, int32_t local, uint32_t* word) {
  cg_comm* c = ctx->comm;
  cudaStream_t s = ctx->stream;
  *word = status_bits(local);
  CG_CUDA(cudaMemcpyAsync(c->d_token, word, sizeof(*word), cudaMemcpyHostToDevice, s));
  int32_t rc;
  if ((rc = barrier(ctx))) return rc;
  CG_CUDA(cudaMemcpyAsync(word, c->d_token, sizeof(*word), cudaMemcpyDeviceToHost, s));
  CG_CUDA(cudaMemsetAsync(c->d_token, 0, sizeof(int), s));
  CG_CUDA(cudaStreamSynchronize(s));
  return CG_OK;
}

int32_t cg_reproject_submaps_sharded(const cg_layer* const* submaps, size_t n, size_t num_known,
                                     const float* poses_old, const float* poses_new,
                                     float eps_translation, float eps_rotation, cg_layer* partial,
                                     cg_layer* owned, uint8_t* changed_out,
                                     cg_reproject_sharded_stats* stats) {
  static const char* who = "cg_reproject_submaps_sharded";
  if (stats) memset(stats, 0, sizeof(*stats));
  if (!partial || !owned || partial->ctx != owned->ctx || partial == owned) {
    set_error("%s: partial and owned must be two layers of one context", who);
    return CG_ERR_INVALID_ARG;
  }
  cg_context* ctx = owned->ctx;
  cg_comm* c = ctx->comm;
  if (!c) {
    set_error("%s: call cg_comm_init first", who);
    return CG_ERR_INVALID_ARG;
  }
  CG_CUDA(cudaSetDevice(ctx->device));
  cudaStream_t s = ctx->stream;
  // This rank's arguments.  A rejected call still joins the opening barrier, so every rank returns
  // an error and no rank touches its owned layer.
  int32_t local = CG_ERR_INVALID_ARG;
  if (num_known > n) {
    set_error("%s: num_known (%zu) > num_submaps (%zu)", who, num_known, n);
  } else if (n && (!submaps || !poses_new || (num_known && !poses_old))) {
    set_error("%s: null submap or pose array", who);
  } else if (c->partial.serial == 0 || c->partial.serial != partial->serial) {
    set_error("%s: `partial` is not the partial layer of the last cg_gather_global on this context",
              who);
  } else if (partial->v.voxel_size != owned->v.voxel_size) {
    set_error("%s: the layers' voxel sizes differ", who);
  } else {
    local = CG_OK;
    for (size_t i = 0; i < n && local == CG_OK; ++i) {
      if (submaps[i] == owned) {
        set_error("%s: submap %zu is the owned layer", who, i);
        local = CG_ERR_INVALID_ARG;
      }
    }
  }
  cg_reproject_stats rs{};
  const int64_t owned_before = owned->num_blocks;
  if (local == CG_OK) {
    const DirtyKeysOut dk{c->partial.dirty, c->partial.shared + 2, c->partial.dirty_cap};
    local = cudaMemsetAsync(c->partial.shared + 2, 0, sizeof(uint32_t), s) == cudaSuccess
                ? CG_OK : cuda_fail(cudaGetLastError(), "cudaMemsetAsync");
    if (local == CG_OK)
      local = reproject_local(submaps, n, num_known, poses_old, poses_new, eps_translation,
                              eps_rotation, partial, changed_out, &rs, &dk, who);
  }
  if (local == CG_OK) {
    const float fraction = static_cast<float>(full_rebuild_fraction());
    uint32_t fbits;
    memcpy(&fbits, &fraction, sizeof(fbits));
    ctx->own_launches += 1;
    k_publish_words<<<1, 1, 0, s>>>(c->partial.shared, static_cast<uint32_t>(partial->num_blocks),
                                    static_cast<uint32_t>(owned->num_blocks), fbits);
  }
  uint32_t word = 0;
  int32_t rc;
  // every rank's partial layer, dirty keys and counts are complete (stream-ordered)
  if ((rc = status_barrier(ctx, local, &word))) return rc;
  if (local) return local;
  if (word) {
    set_error("%s: another rank's local step failed (status %d); no owned layer was changed", who,
              status_of(word));
    return status_of(word);
  }
  // D: the union of every rank's published keys, identical on every rank
  const int R = c->nranks;
  const size_t dcap = key_set_capacity(2 * partial->max_blocks * static_cast<size_t>(R), 1024);
  uint32_t h[4] = {0, 0, 0, 0};
  rc = [&]() -> int32_t {
    CG_CUDA(c->dset.reserve(dcap * sizeof(unsigned long long)));
    c->dcap = dcap;
    if (!c->dcounters) CG_CUDA(cudaMalloc(&c->dcounters, 4 * sizeof(uint32_t)));
    CG_CUDA(cudaMemsetAsync(c->dset.p, 0xFF, dcap * sizeof(unsigned long long), s));
    CG_CUDA(cudaMemsetAsync(c->dcounters, 0, 4 * sizeof(uint32_t), s));
    ctx->own_launches += 1;
    k_union_dirty<<<dim3(static_cast<unsigned>(ctx->num_sms), static_cast<unsigned>(R)), 256, 0, s>>>(
        c->partial.d_peers, c->partial.dirty_cap,
        KeySet{c->dset.as<unsigned long long>(), static_cast<uint32_t>(dcap - 1)}, c->dcounters);
    CG_CUDA(cudaMemcpyAsync(h, c->dcounters, sizeof(h), cudaMemcpyDeviceToHost, s));
    CG_CUDA(cudaStreamSynchronize(s));
    return CG_OK;
  }();
  if (rc) {
    barrier(ctx);
    return rc;
  }
  float fraction;
  memcpy(&fraction, &h[3], sizeof(fraction));
  const bool full = static_cast<double>(h[0]) > static_cast<double>(fraction) * static_cast<double>(h[1]);
  if (stats) {
    stats->submaps_moved = rs.submaps_moved;
    stats->submaps_added = n - num_known;
    stats->blocks_dirty_local = rs.blocks_dirty;
    stats->blocks_dirty = h[0];
    stats->full_rebuild = full ? 1 : 0;
  }
  if (h[2]) {  // cannot happen: a partial layer holds at most max_blocks blocks before and after
    barrier(ctx);
    set_error("%s: a rank published more dirty keys than its buffer holds", who);
    return CG_ERR_CUDA;
  }
  if (full) {
    // the whole gather, into the cleared owned layer (it opens and closes with its own barriers)
    rc = cg_layer_clear(owned);
    if (rc) {
      barrier(ctx);
      return rc;
    }
    rc = cg_gather_global(partial, owned, nullptr);
    if (stats) stats->blocks_folded = static_cast<uint64_t>(owned->num_blocks);
    return rc;
  }
  // The blocks of D this owned layer holds are reset, the blocks of D it owns now are folded (a
  // held block as it was reset, a new one fresh), and held blocks that were not folded again —
  // owned elsewhere now, or without data — are removed.
  CG_CUDA(ctx->stage_b.reserve((static_cast<size_t>(owned->num_blocks) + 2) * sizeof(uint32_t)));
  uint32_t* counts = ctx->stage_b.as<uint32_t>();  // [0] blocks of D the owned layer holds
  uint32_t* slots = counts + 2;
  rc = [&]() -> int32_t {
    if (h[0] == 0) return CG_OK;
    int32_t r = reset_dirty_blocks(owned, c->dset.as<uint64_t>(), static_cast<uint32_t>(dcap), slots,
                                   counts);
    if (r) return r;
    if ((r = reset_holders(ctx))) return r;
    list_holders(ctx, KeyLookup{c->dset.as<unsigned long long>(), static_cast<uint32_t>(dcap - 1)});
    return fold_owned(ctx, owned);
  }();
  // nobody clears or refills its partial layer while a peer still reads it
  const int32_t rb = barrier(ctx);
  if (rc) return rc;
  if (rb) return rb;
  uint64_t removed = 0;
  uint32_t listed = 0;
  if (h[0] > 0) {
    CG_CUDA(cudaMemcpyAsync(&listed, counts, sizeof(listed), cudaMemcpyDeviceToHost, s));
    if ((rc = finish_call(owned, nullptr))) return rc;
    if (listed > 0 && (rc = remove_dead_blocks(owned, slots, counts, listed, &removed))) return rc;
  }
  if (stats) {
    // blocks outside D are untouched: the owned blocks of D now are the ones folded
    stats->blocks_folded = static_cast<uint64_t>(owned->num_blocks - (owned_before - listed));
    stats->blocks_removed = removed;
  }
  return CG_OK;
}

// ---- cg_mesh_gather_sharded (DESIGN.md §5): every rank's block meshes -> the root, in the block
// order cg_layer_mesh gives the union of the owned layers.
static const char* kGatherWho = "cg_mesh_gather_sharded";

// The same verdict on every rank: it judges the all-gathered words only.
static int32_t gather_verdict(const std::vector<GatherWords>& all) {
  const char* who = kGatherWho;
  const int R = static_cast<int>(all.size());
  for (int r = 0; r < R; ++r) {
    if (all[r].root < 0 || all[r].root >= R) {
      set_error("%s: rank %d passed root %lld, outside [0, %d)", who, r, all[r].root, R);
      return CG_ERR_INVALID_ARG;
    }
  }
  for (int r = 1; r < R; ++r) {
    if (all[r].root != all[0].root) {
      set_error("%s: the ranks passed different roots (rank 0: %lld, rank %d: %lld)", who,
                all[0].root, r, all[r].root);
      return CG_ERR_INVALID_ARG;
    }
  }
  for (int r = 0; r < R; ++r) {
    const char* why = nullptr;
    switch (static_cast<int>(all[r].kind)) {
      case kMeshSharded: break;
      case kMeshLocal: why = "is from cg_layer_mesh, not cg_layer_mesh_sharded"; break;
      case kMeshGathered: why = "has been gathered already (call cg_layer_mesh_sharded again)"; break;
      case kMeshReused: why = "is gone: cg_esdf_free_points reused its buffers"; break;
      default: why = "does not exist (no mesh call yet, or the last one failed)"; break;
    }
    if (why) {
      set_error("%s: rank %d's retained mesh %s", who, r, why);
      return CG_ERR_INVALID_ARG;
    }
    if (all[r].calls != all[0].calls) {
      set_error("%s: rank %d's mesh is from its cg_layer_mesh_sharded call %llu, rank 0's from call %llu",
                who, r, all[r].calls, all[0].calls);
      return CG_ERR_INVALID_ARG;
    }
  }
  unsigned long long blocks = 0, vertices = 0;
  for (const GatherWords& w : all) {
    blocks += w.blocks;
    vertices += w.vertices;
  }
  if (vertices > 0xFFFFFFFFull || blocks > 0x7FFFFFF0ull) {
    set_error("%s: the gathered mesh would hold %llu blocks and %llu vertices; vertex_begin (uint32) "
              "indexes at most 4294967295 vertices", who, blocks, vertices);
    return CG_ERR_INVALID_ARG;
  }
  return CG_OK;
}

// Where a peer's sends land in the root's mg_in (byte offsets, 256-byte aligned).
struct PeerRegions {
  size_t idx, begin, vertices, normals, colors;
};

// Every buffer the root needs, reserved before the first byte moves.
static int32_t gather_reserve(cg_context* ctx, const std::vector<GatherWords>& all, int root,
                              std::vector<PeerRegions>* regions) {
  const size_t R = all.size();
  size_t N = 0, V = 0, in_bytes = 0;
  auto take = [&](size_t bytes) {
    const size_t at = in_bytes;
    in_bytes += (bytes + 255) & ~static_cast<size_t>(255);
    return at;
  };
  regions->assign(R, PeerRegions{0, 0, 0, 0, 0});
  for (size_t r = 0; r < R; ++r) {
    const size_t n = all[r].blocks, v = all[r].vertices;
    N += n;
    V += v;
    if (static_cast<int>(r) == root || n == 0) continue;
    PeerRegions& g = (*regions)[r];
    g.idx = take(3 * n * sizeof(int32_t));
    g.begin = take((n + 1) * sizeof(uint32_t));
    g.vertices = take(3 * v * sizeof(float));
    g.normals = take(3 * v * sizeof(float));
    g.colors = take(v * sizeof(uint32_t));
  }
  if (N == 0) return CG_OK;
  CG_CUDA(ctx->mg_in.reserve(in_bytes));
  CG_CUDA(ctx->mg_sort.reserve(4 * N * sizeof(unsigned long long)));
  CG_CUDA(ctx->mg_src.reserve(R * sizeof(MeshSource)));
  CG_CUDA(ctx->mg_counts.reserve((2 * (N + 1) + 2) * sizeof(uint32_t)));
  CG_CUDA(ctx->mg_index.reserve(3 * N * sizeof(int32_t)));
  CG_CUDA(ctx->mg_vertices.reserve(3 * V * sizeof(float)));
  CG_CUDA(ctx->mg_normals.reserve(3 * V * sizeof(float)));
  CG_CUDA(ctx->mg_colors.reserve(V * sizeof(uint32_t)));
  size_t sort_tmp = 0, scan_tmp = 0;
  CG_CUDA(cub::DeviceRadixSort::SortPairs(nullptr, sort_tmp, static_cast<const unsigned long long*>(nullptr),
                                          static_cast<unsigned long long*>(nullptr),
                                          static_cast<const unsigned long long*>(nullptr),
                                          static_cast<unsigned long long*>(nullptr),
                                          static_cast<int>(N), 0, 63, ctx->stream));
  CG_CUDA(cub::DeviceScan::ExclusiveSum(nullptr, scan_tmp, static_cast<const uint32_t*>(nullptr),
                                        static_cast<uint32_t*>(nullptr), static_cast<int>(N + 1),
                                        ctx->stream));
  CG_CUDA(ctx->cub_tmp.reserve(std::max(sort_tmp, scan_tmp)));
  return CG_OK;
}

// Each peer's block meshes to the root (NCCL point-to-point, one group); a rank without blocks
// sends nothing, and the root posts exactly the receives that match.
static int32_t gather_transfer(cg_context* ctx, const std::vector<GatherWords>& all, int root,
                               const std::vector<PeerRegions>& regions) {
  cg_comm* c = ctx->comm;
  cudaStream_t s = ctx->stream;
  int e = g_nccl.GroupStart();
  if (e != ncclSuccess) {
    set_error("%s: ncclGroupStart failed: %s", kGatherWho, g_nccl.GetErrorString(e));
    return CG_ERR_CUDA;
  }
  auto send = [&](const void* p, size_t bytes) {
    if (e == ncclSuccess && bytes) e = g_nccl.Send(p, bytes, ncclInt8, root, c->comm, s);
  };
  auto recv = [&](size_t at, size_t bytes, int peer) {
    if (e == ncclSuccess && bytes)
      e = g_nccl.Recv(ctx->mg_in.as<char>() + at, bytes, ncclInt8, peer, c->comm, s);
  };
  if (c->rank != root) {
    const size_t n = ctx->mc_blocks, v = ctx->mc_total;
    if (n > 0) {
      send(ctx->mc_index.p, 3 * n * sizeof(int32_t));
      send(ctx->mc_counts.as<uint32_t>() + (n + 1), (n + 1) * sizeof(uint32_t));
      send(ctx->mc_vertices.p, 3 * v * sizeof(float));
      send(ctx->mc_normals.p, 3 * v * sizeof(float));
      send(ctx->mc_colors.p, v * sizeof(uint32_t));
    }
  } else {
    for (int r = 0; r < c->nranks; ++r) {
      const size_t n = all[r].blocks, v = all[r].vertices;
      if (r == root || n == 0) continue;
      const PeerRegions& g = regions[r];
      recv(g.idx, 3 * n * sizeof(int32_t), r);
      recv(g.begin, (n + 1) * sizeof(uint32_t), r);
      recv(g.vertices, 3 * v * sizeof(float), r);
      recv(g.normals, 3 * v * sizeof(float), r);
      recv(g.colors, v * sizeof(uint32_t), r);
    }
  }
  const int end = g_nccl.GroupEnd();
  if (e == ncclSuccess) e = end;
  if (e != ncclSuccess) {
    set_error("%s: NCCL error %d (%s) in the transfer to rank %d", kGatherWho, e,
              g_nccl.GetErrorString(e), root);
    return CG_ERR_CUDA;
  }
  return CG_OK;
}

// On the root: every rank's blocks sorted by packed key, vertex_begin by a scan of their vertex
// counts, each block placed into the mg_* buffers, which then become the retained mesh.
static int32_t gather_place(cg_context* ctx, const std::vector<GatherWords>& all, int root,
                            const std::vector<PeerRegions>& regions) {
  cudaStream_t s = ctx->stream;
  const int R = static_cast<int>(all.size());
  size_t N = 0;
  for (const GatherWords& w : all) N += w.blocks;
  if (N == 0) return CG_OK;
  std::vector<MeshSource> src(R);
  uint32_t first = 0;
  uint32_t most = 0;
  for (int r = 0; r < R; ++r) {
    const uint32_t n = static_cast<uint32_t>(all[r].blocks);
    MeshSource& S = src[r];
    if (r == root) {
      S = MeshSource{ctx->mc_index.as<int32_t>(), ctx->mc_counts.as<uint32_t>() + (n + 1),
                     ctx->mc_vertices.as<uint32_t>(), ctx->mc_normals.as<uint32_t>(),
                     ctx->mc_colors.as<uint32_t>(), n, first};
    } else {
      const char* in = ctx->mg_in.as<char>();
      const PeerRegions& g = regions[r];
      S = MeshSource{reinterpret_cast<const int32_t*>(in + g.idx),
                     reinterpret_cast<const uint32_t*>(in + g.begin),
                     reinterpret_cast<const uint32_t*>(in + g.vertices),
                     reinterpret_cast<const uint32_t*>(in + g.normals),
                     reinterpret_cast<const uint32_t*>(in + g.colors), n, first};
    }
    first += n;
    most = std::max(most, n);
  }
  CG_CUDA(cudaMemcpyAsync(ctx->mg_src.p, src.data(), R * sizeof(MeshSource), cudaMemcpyHostToDevice, s));
  const MeshSource* d_src = ctx->mg_src.as<MeshSource>();
  unsigned long long* keys_in = ctx->mg_sort.as<unsigned long long>();
  unsigned long long *keys_out = keys_in + N, *vals_in = keys_out + N, *vals_out = vals_in + N;
  uint32_t* counts = ctx->mg_counts.as<uint32_t>();
  uint32_t* begin = counts + (N + 1);
  const uint32_t n = static_cast<uint32_t>(N);
  ctx->own_launches += 3;
  const unsigned per_rank = static_cast<unsigned>(std::min<size_t>(grid_for(most, 256), ctx->num_sms * 4));
  k_gather_keys<<<dim3(per_rank, static_cast<unsigned>(R)), 256, 0, s>>>(d_src, keys_in, vals_in);
  size_t tmp = ctx->cub_tmp.cap;
  CG_CUDA(cub::DeviceRadixSort::SortPairs(ctx->cub_tmp.p, tmp, keys_in, keys_out, vals_in, vals_out,
                                          static_cast<int>(n), 0, 63, s));
  k_gather_counts<<<std::min<unsigned>(grid_for(N + 1, 256), ctx->num_sms * 4), 256, 0, s>>>(
      d_src, vals_out, n, counts);
  tmp = ctx->cub_tmp.cap;
  CG_CUDA(cub::DeviceScan::ExclusiveSum(ctx->cub_tmp.p, tmp, counts, begin, static_cast<int>(n + 1), s));
  k_place_blocks<<<std::min<unsigned>(grid_for(N, kPlaceThreads / 32), ctx->num_sms * 16),
                   kPlaceThreads, 0, s>>>(d_src, vals_out, begin, n, ctx->mg_index.as<int32_t>(),
                                          ctx->mg_vertices.as<uint32_t>(), ctx->mg_normals.as<uint32_t>(),
                                          ctx->mg_colors.as<uint32_t>());
  CG_CUDA(cudaGetLastError());
  // the root's own share was a source: the placed buffers replace it, the old ones are the next
  // gather's scratch
  std::swap(ctx->mc_counts, ctx->mg_counts);
  std::swap(ctx->mc_index, ctx->mg_index);
  std::swap(ctx->mc_vertices, ctx->mg_vertices);
  std::swap(ctx->mc_normals, ctx->mg_normals);
  std::swap(ctx->mc_colors, ctx->mg_colors);
  return CG_OK;
}

int32_t cg_mesh_gather_sharded(cg_context* ctx, int32_t root, size_t* num_blocks_out,
                               size_t* num_vertices_out) {
  const char* who = kGatherWho;
  if (num_blocks_out) *num_blocks_out = 0;
  if (num_vertices_out) *num_vertices_out = 0;
  if (!ctx) {
    set_error("%s: null context", who);
    return CG_ERR_INVALID_ARG;
  }
  cg_comm* c = ctx->comm;
  if (!c) {
    set_error("%s: call cg_comm_init first", who);
    return CG_ERR_INVALID_ARG;
  }
  CG_CUDA(cudaSetDevice(ctx->device));
  cudaStream_t s = ctx->stream;
  const int R = c->nranks;
  // the opening: one all-gather of every rank's words (the retained mesh, its kind, the root)
  const GatherWords mine{ctx->mc_blocks, ctx->mc_total, static_cast<unsigned long long>(ctx->mc_kind),
                         ctx->mc_sharded_calls, root};
  CG_CUDA(c->gwords.reserve(R * sizeof(GatherWords)));
  char* d_all = c->gwords.as<char>();
  CG_CUDA(cudaMemcpyAsync(d_all + c->rank * sizeof(GatherWords), &mine, sizeof(GatherWords),
                          cudaMemcpyHostToDevice, s));
  CG_NCCL(g_nccl.AllGather(d_all + c->rank * sizeof(GatherWords), d_all, sizeof(GatherWords),
                           ncclInt8, c->comm, s));
  std::vector<GatherWords> all(R);
  CG_CUDA(cudaMemcpyAsync(all.data(), d_all, R * sizeof(GatherWords), cudaMemcpyDeviceToHost, s));
  CG_CUDA(cudaStreamSynchronize(s));
  // every check, and every reservation on the root, before the go/no-go
  int32_t local = gather_verdict(all);
  const int rt = static_cast<int>(all[0].root);
  std::vector<PeerRegions> regions;
  if (local == CG_OK && c->rank == rt) local = gather_reserve(ctx, all, rt, &regions);
  uint32_t word = 0;
  int32_t rc = status_barrier(ctx, local, &word);
  if (rc) return rc;
  if (word) {
    if (local == CG_OK)
      set_error("%s: rank %d (the root) could not reserve its buffers (status %d); nothing was moved",
                who, rt, status_of(word));
    const int32_t rb = barrier(ctx);
    return rb ? rb : status_of(word);
  }
  rc = gather_transfer(ctx, all, rt, regions);
  if (rc == CG_OK && c->rank == rt) rc = gather_place(ctx, all, rt, regions);
  // a rank re-meshes or clears its owned layer only after the root has everything
  const int32_t rb = barrier(ctx);
  if (rc) return rc;
  if (rb) return rb;
  size_t N = 0, V = 0;
  for (const GatherWords& w : all) {
    N += w.blocks;
    V += w.vertices;
  }
  if (c->rank == rt) {
    ctx->mc_blocks = N;
    ctx->mc_total = V;
  }
  ctx->mc_kind = kMeshGathered;
  if (num_blocks_out) *num_blocks_out = N;
  if (num_vertices_out) *num_vertices_out = V;
  return CG_OK;
}

}  // extern "C"
