// mesh_recover.cu — the recover node's front end on the device (SURVEY.md §8f N3).
//
// Replaces voxblox::MeshConverter::convertToPointCloud + getNextPointcloud
// (coxgraph/include/coxgraph/map_comm/mesh_converter.h:74-172, :186-209, interpolateTriangle
// :211-265) and the loop of TsdfRecover::processMesh around integratePointCloud
// (coxgraph/include/coxgraph/map_comm/tsdf_recover.h:59-99).  This code IS in the reference tree,
// so every step below follows its source, quirks included (edge p0-p2 blends colors[0] with
// colors[1], :235-236; the observation map is keyed by uint8_t, :274).
//
//   k_tri_count    per triangle: decode the uint16 vertices, count the edge samples, count the
//                  observation stamps of its history
//   scan           (triangle, stamp) pair offsets
//   k_tri_pairs    the pairs, in (triangle, stamp occurrence) order: bucket key = uint8(stamp)
//   radix sort     stable, by bucket: each bucket's triangles in mesh order — the order in which
//                  the reference appends to pointcloud_[stamp]
//   scan           point offsets of the pairs
//   k_tri_write    per pair: the triangle's 3 vertices, its edge samples and centroid, colours
//   k_frame_cloud  per trajectory pose: its bucket's cloud moved into the sensor frame
#include <cub/cub.cuh>
#include <math.h>
#include <string.h>

#include <algorithm>
#include <vector>

#include "cg_internal.cuh"

namespace cg {

struct MeshView {
  const int32_t* block_index;
  const uint8_t* block_has_history;
  const uint32_t* vertex_begin;
  const uint16_t *x, *y, *z;
  const uint8_t *r, *g, *b;
  const uint32_t* hist_begin;
  const uint32_t* hist;
  uint32_t num_blocks, num_triangles;
  float block_edge_length;
};

struct Tri {
  V3 p[3];
  uint32_t c[3];  // rgba packed r | g << 8 | b << 16 | a << 24
  bool live;      // its block has a history
};

__device__ __forceinline__ Tri load_triangle(const MeshView& M, uint32_t t) {
  // block of vertex 3 t: last b with vertex_begin[b] <= 3 t
  const uint32_t v0 = 3u * t;
  uint32_t lo = 0, hi = M.num_blocks;
  while (hi - lo > 1) {
    const uint32_t mid = (lo + hi) >> 1;
    if (M.vertex_begin[mid] <= v0) lo = mid; else hi = mid;
  }
  Tri T;
  T.live = M.block_has_history[lo] != 0;
  const float ix = static_cast<float>(M.block_index[3 * lo]);
  const float iy = static_cast<float>(M.block_index[3 * lo + 1]);
  const float iz = static_cast<float>(M.block_index[3 * lo + 2]);
  const float f = 2.0f / 65535.0f;  // point_conv_factor, mesh_converter.h:97-98
#pragma unroll
  for (int k = 0; k < 3; ++k) {
    const uint32_t i = v0 + k;
    T.p[k] = V3{(static_cast<float>(M.x[i]) * f + ix) * M.block_edge_length,
                (static_cast<float>(M.y[i]) * f + iy) * M.block_edge_length,
                (static_cast<float>(M.z[i]) * f + iz) * M.block_edge_length};
    T.c[k] = pack_rgba(M.r[i], M.g[i], M.b[i], 255u);
  }
  return T;
}

// number of samples of `for (float dist = vs; dist < len; dist += vs)`
__device__ __forceinline__ uint32_t edge_samples(float len, float vs) {
  uint32_t n = 0;
  for (float dist = vs; dist < len; dist += vs) ++n;
  return n;
}

__global__ void k_tri_count(MeshView M, float vs, uint32_t* __restrict__ tri_points,
                            uint32_t* __restrict__ tri_stamps) {
  const uint32_t t = blockIdx.x * blockDim.x + threadIdx.x;
  if (t >= M.num_triangles) return;
  const Tri T = load_triangle(M, t);
  uint32_t stamps = 0;
  if (T.live)
    for (uint32_t h = M.hist_begin[t]; h + 1 < M.hist_begin[t + 1]; h += 2)
      if (M.hist[h + 1] >= M.hist[h]) stamps += M.hist[h + 1] - M.hist[h] + 1;
  tri_stamps[t] = stamps;
  tri_points[t] = 3u + edge_samples(norm3(T.p[1] - T.p[0]), vs) + 1u +
                  edge_samples(norm3(T.p[2] - T.p[0]), vs) + edge_samples(norm3(T.p[2] - T.p[1]), vs);
}

__global__ void k_tri_pairs(MeshView M, const uint32_t* __restrict__ tri_stamps,
                            const uint32_t* __restrict__ pair_begin,
                            const uint32_t* __restrict__ tri_points, uint32_t* __restrict__ pair_key,
                            uint32_t* __restrict__ pair_tri, uint32_t* __restrict__ pair_points) {
  const uint32_t t = blockIdx.x * blockDim.x + threadIdx.x;
  if (t >= M.num_triangles || tri_stamps[t] == 0) return;
  uint32_t o = pair_begin[t];
  const uint32_t np = tri_points[t];
  for (uint32_t h = M.hist_begin[t]; h + 1 < M.hist_begin[t + 1]; h += 2)
    for (uint64_t j = M.hist[h]; j <= M.hist[h + 1]; ++j, ++o) {
      pair_key[o] = static_cast<uint32_t>(j) & 255u;  // std::map<uint8_t, ...>
      pair_tri[o] = t;
      pair_points[o] = np;
    }
}

// first point of every bucket (257 entries; [256] = total number of points)
__global__ void k_bucket_begin(const uint32_t* __restrict__ sorted_key,
                               const uint32_t* __restrict__ point_offset,
                               const uint32_t* __restrict__ sorted_points, uint32_t num_pairs,
                               uint32_t* __restrict__ bucket_first_point) {
  const uint32_t b = threadIdx.x + blockIdx.x * blockDim.x;
  if (b > 256) return;
  uint32_t lo = 0, hi = num_pairs;  // first pair with key >= b
  while (lo < hi) {
    const uint32_t mid = (lo + hi) >> 1;
    if (sorted_key[mid] < b) lo = mid + 1; else hi = mid;
  }
  bucket_first_point[b] = lo < num_pairs
                              ? point_offset[lo]
                              : point_offset[num_pairs - 1] + sorted_points[num_pairs - 1];
}

__global__ void k_tri_write(MeshView M, float vs, const uint32_t* __restrict__ sorted_tri,
                            const uint32_t* __restrict__ out_begin, uint32_t num_pairs,
                            float* __restrict__ pts, uint32_t* __restrict__ cols) {
  const uint32_t q = blockIdx.x * blockDim.x + threadIdx.x;
  if (q >= num_pairs) return;
  const Tri T = load_triangle(M, sorted_tri[q]);
  size_t o = out_begin[q];
  auto put = [&](V3 p, uint32_t c) {
    pts[3 * o] = p.x;
    pts[3 * o + 1] = p.y;
    pts[3 * o + 2] = p.z;
    cols[o] = c;
    ++o;
  };
  for (int k = 0; k < 3; ++k) put(T.p[k], T.c[k]);  // the triangle itself, :148-149
  // interpolateTriangle, :211-265: edge p0-p1, the centroid, edge p0-p2, edge p1-p2
  const V3 t01 = T.p[1] - T.p[0], t02 = T.p[2] - T.p[0], t12 = T.p[2] - T.p[1];
  const float n01 = norm3(t01), n02 = norm3(t02), n12 = norm3(t12);
  for (float dist = vs; dist < n01; dist += vs)
    put(T.p[0] + (t01 / n01) * dist, blend_colors(T.c[0], 1 - dist / n01, T.c[1], dist / n01));
  put(((T.p[0] + T.p[1]) + T.p[2]) / 3.0f,
      blend_colors(T.c[2], static_cast<float>(1 / 3.0), blend_colors(T.c[0], 0.5f, T.c[1], 0.5f),
                   static_cast<float>(2 / 3.0)));
  for (float dist = vs; dist < n02; dist += vs)  // colors[0] / colors[1]: as the reference, :235
    put(T.p[0] + (t02 / n02) * dist, blend_colors(T.c[0], 1 - dist / n02, T.c[1], dist / n02));
  for (float dist = vs; dist < n12; dist += vs)
    put(T.p[1] + (t12 / n12) * dist, blend_colors(T.c[1], 1 - dist / n12, T.c[2], dist / n12));
}

struct FrameMap {  // one per trajectory pose
  Xform T_C_G;     // inverse pose
  uint64_t src, dst;
  uint32_t n, pad;
};
__global__ void k_frame_cloud(const FrameMap* __restrict__ frames, const float* __restrict__ pts_g,
                              const uint32_t* __restrict__ cols_g, float* __restrict__ pts_c,
                              uint32_t* __restrict__ cols_c) {
  const FrameMap fm = frames[blockIdx.y];
  for (uint32_t i = blockIdx.x * blockDim.x + threadIdx.x; i < fm.n; i += gridDim.x * blockDim.x) {
    const size_t s = fm.src + i, d = fm.dst + i;
    const V3 pc = apply(fm.T_C_G, V3{pts_g[3 * s], pts_g[3 * s + 1], pts_g[3 * s + 2]});
    pts_c[3 * d] = pc.x;
    pts_c[3 * d + 1] = pc.y;
    pts_c[3 * d + 2] = pc.z;
    cols_c[d] = cols_g[s];
  }
}

// Builds the per-pose clouds on the device: ctx->mesh_pts_c / mesh_cols_c, offsets in *offs.
static int32_t mesh_frames_device(cg_context* ctx, const cg_mesh* m, float vs, size_t F,
                                  const float* poses, const double* stamps,
                                  std::vector<uint64_t>* offs) {
  cudaStream_t s = ctx->stream;
  offs->assign(F + 1, 0);
  if (!m || (m->num_blocks && (!m->block_index || !m->vertex_begin || !m->block_has_history)) ||
      !(vs > 0.0f) || (F && (!poses || !stamps))) {
    set_error("cg_mesh: invalid argument");
    return CG_ERR_INVALID_ARG;
  }
  const size_t B = m->num_blocks;
  const size_t V = B ? m->vertex_begin[B] : 0;
  if (V % 3 != 0 || V >= 0xFFFFFFF0ull) {
    set_error("cg_mesh: the vertex count must be a multiple of 3");
    return CG_ERR_INVALID_ARG;
  }
  const uint32_t Tn = static_cast<uint32_t>(V / 3);
  if (Tn == 0 || F == 0) return CG_OK;
  const size_t H = m->hist_begin[Tn];
  // mesh arrays -> one device buffer
  auto al = [](size_t x) { return (x + 255) & ~size_t(255); };
  const size_t o_idx = 0, o_has = al(o_idx + B * 12), o_vb = al(o_has + B), o_x = al(o_vb + (B + 1) * 4),
               o_y = al(o_x + V * 2), o_z = al(o_y + V * 2), o_r = al(o_z + V * 2), o_g = al(o_r + V),
               o_b = al(o_g + V), o_hb = al(o_b + V), o_h = al(o_hb + (size_t(Tn) + 1) * 4),
               total = al(o_h + H * 4);
  CG_CUDA(ctx->mesh_in.reserve(total));
  char* d = ctx->mesh_in.as<char>();
  auto up = [&](size_t off, const void* src, size_t bytes) {
    return bytes ? cudaMemcpyAsync(d + off, src, bytes, cudaMemcpyHostToDevice, s) : cudaSuccess;
  };
  CG_CUDA(up(o_idx, m->block_index, B * 12));
  CG_CUDA(up(o_has, m->block_has_history, B));
  CG_CUDA(up(o_vb, m->vertex_begin, (B + 1) * 4));
  CG_CUDA(up(o_x, m->x, V * 2));
  CG_CUDA(up(o_y, m->y, V * 2));
  CG_CUDA(up(o_z, m->z, V * 2));
  CG_CUDA(up(o_r, m->r, V));
  CG_CUDA(up(o_g, m->g, V));
  CG_CUDA(up(o_b, m->b, V));
  CG_CUDA(up(o_hb, m->hist_begin, (size_t(Tn) + 1) * 4));
  CG_CUDA(up(o_h, m->hist, H * 4));
  MeshView M;
  M.block_index = reinterpret_cast<const int32_t*>(d + o_idx);
  M.block_has_history = reinterpret_cast<const uint8_t*>(d + o_has);
  M.vertex_begin = reinterpret_cast<const uint32_t*>(d + o_vb);
  M.x = reinterpret_cast<const uint16_t*>(d + o_x);
  M.y = reinterpret_cast<const uint16_t*>(d + o_y);
  M.z = reinterpret_cast<const uint16_t*>(d + o_z);
  M.r = reinterpret_cast<const uint8_t*>(d + o_r);
  M.g = reinterpret_cast<const uint8_t*>(d + o_g);
  M.b = reinterpret_cast<const uint8_t*>(d + o_b);
  M.hist_begin = reinterpret_cast<const uint32_t*>(d + o_hb);
  M.hist = reinterpret_cast<const uint32_t*>(d + o_h);
  M.num_blocks = static_cast<uint32_t>(B);
  M.num_triangles = Tn;
  M.block_edge_length = m->block_edge_length;

  // per triangle counts, pair offsets
  CG_CUDA(ctx->mesh_tri.reserve(4 * (size_t(Tn) + 1) * sizeof(uint32_t)));
  uint32_t* tri_points = ctx->mesh_tri.as<uint32_t>();
  uint32_t* tri_stamps = tri_points + Tn + 1;
  uint32_t* pair_begin = tri_stamps + Tn + 1;
  CG_CUDA(cudaMemsetAsync(tri_stamps + Tn, 0, sizeof(uint32_t), s));
  ctx->own_launches += 1;
  k_tri_count<<<grid_for(Tn, 128), 128, 0, s>>>(M, vs, tri_points, tri_stamps);
  size_t tmp = 0;
  CG_CUDA(cub::DeviceScan::ExclusiveSum(nullptr, tmp, tri_stamps, pair_begin, static_cast<int>(Tn + 1), s));
  CG_CUDA(ctx->cub_tmp.reserve(tmp));
  CG_CUDA(cub::DeviceScan::ExclusiveSum(ctx->cub_tmp.p, tmp, tri_stamps, pair_begin,
                                        static_cast<int>(Tn + 1), s));
  uint32_t num_pairs = 0;
  CG_CUDA(cudaMemcpyAsync(&num_pairs, pair_begin + Tn, sizeof(uint32_t), cudaMemcpyDeviceToHost, s));
  CG_CUDA(cudaStreamSynchronize(s));
  CG_CUDA(cudaGetLastError());
  if (num_pairs == 0) return CG_OK;

  // pairs, sorted by bucket (stable: mesh order inside a bucket), point offsets
  const size_t P = num_pairs;
  CG_CUDA(ctx->mesh_pairs.reserve((6 * P + 2 * 260) * sizeof(uint32_t)));
  uint32_t* key_a = ctx->mesh_pairs.as<uint32_t>();
  uint32_t* key_b = key_a + P;
  uint32_t* tri_a = key_b + P;
  uint32_t* tri_b = tri_a + P;
  uint32_t* np_a = tri_b + P;      // points of the pair, then (sorted) exclusive offsets
  uint32_t* np_b = np_a + P;
  uint32_t* bucket_first = np_b + P;
  ctx->own_launches += 1;
  k_tri_pairs<<<grid_for(Tn, 128), 128, 0, s>>>(M, tri_stamps, pair_begin, tri_points, key_a, tri_a,
                                               np_a);
  // value = original pair position; the per-pair arrays are gathered after the sort
  CG_CUDA(ctx->val_a.reserve(P * sizeof(uint32_t)));
  CG_CUDA(ctx->val_b.reserve(P * sizeof(uint32_t)));
  {
    // sort (key, triangle) and (key, points) with the same stable key order
    size_t t1 = 0;
    CG_CUDA(cub::DeviceRadixSort::SortPairs(nullptr, t1, key_a, key_b, tri_a, tri_b,
                                            static_cast<int>(P), 0, 8, s));
    CG_CUDA(ctx->cub_tmp.reserve(t1));
    CG_CUDA(cub::DeviceRadixSort::SortPairs(ctx->cub_tmp.p, t1, key_a, key_b, tri_a, tri_b,
                                            static_cast<int>(P), 0, 8, s));
    uint32_t* key_c = ctx->val_a.as<uint32_t>();
    CG_CUDA(cub::DeviceRadixSort::SortPairs(ctx->cub_tmp.p, t1, key_a, key_c, np_a, np_b,
                                            static_cast<int>(P), 0, 8, s));
  }
  size_t t2 = 0;
  CG_CUDA(cub::DeviceScan::ExclusiveSum(nullptr, t2, np_b, np_a, static_cast<int>(P), s));
  CG_CUDA(ctx->cub_tmp.reserve(t2));
  CG_CUDA(cub::DeviceScan::ExclusiveSum(ctx->cub_tmp.p, t2, np_b, np_a, static_cast<int>(P), s));
  ctx->own_launches += 1;
  k_bucket_begin<<<2, 256, 0, s>>>(key_b, np_a, np_b, num_pairs, bucket_first);
  std::vector<uint32_t> h_first(257);
  CG_CUDA(cudaMemcpyAsync(h_first.data(), bucket_first, 257 * sizeof(uint32_t),
                          cudaMemcpyDeviceToHost, s));
  CG_CUDA(cudaStreamSynchronize(s));
  const size_t total_points = h_first[256];
  CG_CUDA(ctx->mesh_pts_g.reserve(total_points * 3 * sizeof(float)));
  CG_CUDA(ctx->mesh_cols_g.reserve(total_points * sizeof(uint32_t)));
  ctx->own_launches += 1;
  k_tri_write<<<grid_for(P, 128), 128, 0, s>>>(M, vs, tri_b, np_a, num_pairs,
                                              ctx->mesh_pts_g.as<float>(),
                                              ctx->mesh_cols_g.as<uint32_t>());
  // getNextPointcloud for every pose, mesh_converter.h:186-209
  std::vector<FrameMap> fm(F);
  uint64_t run = 0;
  for (size_t i = 0; i < F; ++i) {
    const double id = stamps[i] == stamps[0] ? 0 : round((stamps[i] - stamps[0]) / 0.05);
    const uint32_t bucket = static_cast<uint8_t>(static_cast<long long>(id));
    const uint64_t p0 = h_first[bucket], p1 = h_first[bucket + 1];
    fm[i].T_C_G = inverse_xform_host(make_xform(poses + 7 * i));
    fm[i].src = p0;
    fm[i].dst = run;
    fm[i].n = static_cast<uint32_t>(p1 - p0);
    fm[i].pad = 0;
    (*offs)[i] = run;
    run += p1 - p0;
  }
  (*offs)[F] = run;
  if (run == 0) return CG_OK;
  CG_CUDA(ctx->mesh_pts_c.reserve(run * 3 * sizeof(float)));
  CG_CUDA(ctx->mesh_cols_c.reserve(run * sizeof(uint32_t)));
  CG_CUDA(ctx->mesh_frames.reserve(F * sizeof(FrameMap)));
  CG_CUDA(cudaMemcpyAsync(ctx->mesh_frames.p, fm.data(), F * sizeof(FrameMap), cudaMemcpyHostToDevice, s));
  ctx->own_launches += 1;
  k_frame_cloud<<<dim3(64, static_cast<unsigned>(F)), 256, 0, s>>>(
      ctx->mesh_frames.as<FrameMap>(), ctx->mesh_pts_g.as<float>(), ctx->mesh_cols_g.as<uint32_t>(),
      ctx->mesh_pts_c.as<float>(), ctx->mesh_cols_c.as<uint32_t>());
  CG_CUDA(cudaStreamSynchronize(s));  // fm is a host temporary
  CG_CUDA(cudaGetLastError());
  return CG_OK;
}

}  // namespace cg

using namespace cg;

extern "C" {

int32_t cg_mesh_to_frames(cg_context* ctx, const cg_mesh* mesh, float vs, size_t F,
                          const float* poses, const double* stamps, uint64_t* frame_offsets,
                          float* pts, uint8_t* cols, size_t capacity_points) {
  if (!ctx || !frame_offsets) return CG_ERR_INVALID_ARG;
  CG_CUDA(cudaSetDevice(ctx->device));
  std::vector<uint64_t> offs;
  int32_t rc = mesh_frames_device(ctx, mesh, vs, F, poses, stamps, &offs);
  if (rc) return rc;
  memcpy(frame_offsets, offs.data(), (F + 1) * sizeof(uint64_t));
  const size_t n = offs[F];
  if (!pts || !cols || n == 0) return CG_OK;
  if (capacity_points < n) {
    set_error("cg_mesh_to_frames: capacity %zu < %zu points", capacity_points, n);
    return CG_ERR_INVALID_ARG;
  }
  CG_CUDA(cudaMemcpyAsync(pts, ctx->mesh_pts_c.p, n * 3 * sizeof(float), cudaMemcpyDeviceToHost,
                          ctx->stream));
  CG_CUDA(cudaMemcpyAsync(cols, ctx->mesh_cols_c.p, n * 4, cudaMemcpyDeviceToHost, ctx->stream));
  CG_CUDA(cudaStreamSynchronize(ctx->stream));
  return CG_OK;
}

int32_t cg_recover_mesh(cg_layer* L, const cg_integrator_config* cfg, const cg_mesh* mesh, float vs,
                        size_t F, const float* poses, const double* stamps,
                        cg_integrate_stats* stats) {
  if (!L || !cfg) return CG_ERR_INVALID_ARG;
  cg_context* ctx = L->ctx;
  CG_CUDA(cudaSetDevice(ctx->device));
  int32_t rc = cg_layer_clear(L);  // tsdf_recover.h:62
  if (rc) return rc;
  if (stats) memset(stats, 0, sizeof(*stats));
  std::vector<uint64_t> offs;
  rc = mesh_frames_device(ctx, mesh, vs, F, poses, stamps, &offs);
  if (rc) return rc;
  if (F == 0 || offs[F] == 0) return CG_OK;
  // one integratePointCloud per pose with a non-empty cloud (tsdf_recover.h:71-76), as one job
  return cg_integrate_batch_device(L, cfg, F, poses, ctx->mesh_pts_c.as<float>(),
                                   ctx->mesh_cols_c.as<uint8_t>(), offs.data(), 0, stats);
}

}  // extern "C"
