// host_api_check — drives the C++ host API (coxgraph_b200/host/coxgraph_b200.hpp) the way the
// reference's call sites do (tsdf_recover.h:59-99, map_server.cpp:59-73).  tests/test_host_cpp.py
// writes the input frames, runs this program on the GPU box and compares the layers it writes
// with the CPU oracle.
//   host_api_check nogpu                       -> exit 0 iff creating a context fails loudly
//   host_api_check run <in.bin> <out.bin>      -> integrate frames, merge, dump both layers (and
//                                                 the connected mesh as <out.bin>.ply)
//   host_api_check time <in.bin> <passes>      -> the live path as a C++ host drives it: one
//                                                 integratePointCloud call per frame with pageable
//                                                 std::vector inputs; prints the mean ms per call
// in.bin : u32 F, f32 voxel_size, f32 trunc, f32 T_M_S[7], then per frame: f32 T[7], u32 n,
//          n * 3 f32 points, n * 4 u8 colours
// out.bin: per layer (submap, global): u32 B, B * 3 i32, B * 4096 * 12 B voxels
#include <algorithm>
#include <chrono>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <string>

#include "../../coxgraph_b200/host/coxgraph_b200.hpp"

namespace cg = coxgraph_b200;

template <class T>
static bool rd(FILE* f, T* p, size_t n = 1) { return fread(p, sizeof(T), n, f) == n; }

static void dump(FILE* f, const cg::TsdfLayer& layer) {
  cg::BlockIndexList idx;
  std::vector<cg::TsdfVoxel> vox;
  layer.download(&idx, &vox);
  const uint32_t B = static_cast<uint32_t>(idx.size());
  fwrite(&B, 4, 1, f);
  if (B) {
    fwrite(idx.data(), sizeof(cg::BlockIndex), B, f);
    fwrite(vox.data(), sizeof(cg::TsdfVoxel), vox.size(), f);
  }
}

int main(int argc, char** argv) {
  cg::throw_on_error();
  if (argc >= 2 && std::string(argv[1]) == "nogpu") {
    try {
      cg::Context ctx(0);
    } catch (const cg::Error& e) {
      std::printf("no device: status %d (%s)\n", e.status, e.what());
      return e.status == CG_ERR_CUDA ? 0 : 2;
    }
    std::printf("a CUDA device is present\n");
    return 3;
  }
  if (argc >= 4 && std::string(argv[1]) == "time") {
    FILE* in = fopen(argv[2], "rb");
    if (!in) return 65;
    const int passes = std::atoi(argv[3]);
    uint32_t F = 0;
    float voxel_size = 0, trunc = 0;
    cg::Transformation T_M_S;
    if (!rd(in, &F) || !rd(in, &voxel_size) || !rd(in, &trunc) || !rd(in, &T_M_S.qw, 7)) return 66;
    std::vector<cg::Transformation> poses(F);
    std::vector<cg::Pointcloud> clouds(F);
    std::vector<cg::Colors> colours(F);
    size_t points = 0;
    for (uint32_t f = 0; f < F; ++f) {
      uint32_t n = 0;
      if (!rd(in, &poses[f].qw, 7) || !rd(in, &n)) return 67;
      clouds[f].resize(n);
      colours[f].resize(n);
      if (n && (!rd(in, clouds[f].data(), n) || !rd(in, colours[f].data(), n))) return 68;
      points += n;
    }
    fclose(in);
    cg::Context ctx(0);
    cg::TsdfLayer submap(ctx, voxel_size, 16, 4096);
    cg::TsdfIntegratorBase::Config config;
    config.default_truncation_distance = trunc;
    config.use_const_weight = 1;
    auto integrator = cg::TsdfIntegratorFactory::create("merged", config, &submap);
    double best = 1e30;
    for (int p = 0; p < passes + 1; ++p) {  // pass 0 warms up (scratch buffers, key box)
      submap.removeAllBlocks();
      const auto t0 = std::chrono::steady_clock::now();
      for (uint32_t f = 0; f < F; ++f)
        integrator->integratePointCloud(poses[f], clouds[f], colours[f], false);
      const double ms =
          std::chrono::duration<double, std::milli>(std::chrono::steady_clock::now() - t0).count();
      if (p > 0 && ms < best) best = ms;
    }
    std::printf("{\"ms_per_call\": %.6f, \"frames\": %u, \"points_per_call\": %.1f, "
                "\"blocks\": %lld}\n",
                best / F, F, double(points) / F, static_cast<long long>(submap.getNumberOfAllocatedBlocks()));
    return 0;
  }
  if (argc < 4 || std::string(argv[1]) != "run") return 64;
  FILE* in = fopen(argv[2], "rb");
  if (!in) return 65;
  uint32_t F = 0;
  float voxel_size = 0, trunc = 0;
  cg::Transformation T_M_S;
  if (!rd(in, &F) || !rd(in, &voxel_size) || !rd(in, &trunc) || !rd(in, &T_M_S.qw, 7)) return 66;
  cg::Context ctx(0);
  cg::TsdfLayer submap(ctx, voxel_size, 16, 2048), combined(ctx, voxel_size, 16, 4096);
  cg::TsdfIntegratorBase::Config config;
  config.default_truncation_distance = trunc;
  config.use_const_weight = 1;
  auto integrator = cg::TsdfIntegratorFactory::create("fast", config, &submap);
  submap.removeAllBlocks();  // tsdf_recover.h:62
  for (uint32_t f = 0; f < F; ++f) {
    cg::Transformation T_G_C;
    uint32_t n = 0;
    if (!rd(in, &T_G_C.qw, 7) || !rd(in, &n)) return 67;
    cg::Pointcloud points_C(n);
    cg::Colors colors(n);
    if (n && (!rd(in, points_C.data(), n) || !rd(in, colors.data(), n))) return 68;
    integrator->integratePointCloud(T_G_C, points_C, colors, false);  // tsdf_recover.h:75
  }
  fclose(in);
  combined.removeAllBlocks();                            // map_server.cpp:65
  cg::mergeLayerAintoLayerB(submap, T_M_S, &combined);   // map_server.cpp:67-69
  FILE* out = fopen(argv[3], "wb");
  if (!out) return 69;
  dump(out, submap);
  dump(out, combined);
  fclose(out);
  // what the server does next (server_visualizer.cpp:123-126): mesh the merged map; and a pose
  // update that moves nothing must leave it alone
  cg::LayerMesh mesh;
  cg::generateMesh(combined, &mesh);
  if (mesh.vertices.size() % 3 != 0 || mesh.vertex_begin.size() != mesh.block_indices.size() + 1 ||
      mesh.vertex_begin.back() != mesh.vertices.size())
    return 70;
  {  // the PLY step of saveAndPubCombinedMesh: shared vertices, three indices per triangle
    cg::ConnectedMesh connected;
    cg::getConnectedMesh(combined, &connected);
    if (connected.indices.size() != mesh.vertices.size() ||
        connected.vertices.size() >= mesh.vertices.size() || connected.vertices.empty())
      return 77;
    for (size_t i = 0; i < connected.indices.size(); ++i) {
      const cg::Point& a = connected.vertices[connected.indices[i]];
      const cg::Point& b = mesh.vertices[i];
      if (a.x != b.x || a.y != b.y || a.z != b.z) return 78;
    }
    if (!cg::outputMeshAsPly(std::string(argv[3]) + ".ply", connected)) return 79;
  }
  // ... and what the client's MapServer does with its combined map (map_server.h:141-145,
  // map_server.cpp:112-113): batch ESDF, then the traversable cloud
  {
    cg::EsdfIntegrator::Config ecfg;
    ecfg.min_distance_m = 0.1f;  // coxgraph_client.yaml:69
    cg::EsdfIntegrator esdf(ecfg, &combined);
    cg_esdf_stats est;
    esdf.updateFromTsdfLayerBatch(&est);
    cg::BlockIndexList eidx;
    std::vector<cg::EsdfVoxel> evox;
    esdf.getEsdfLayer(&eidx, &evox);
    if (eidx.size() != combined.getNumberOfAllocatedBlocks() || est.blocks != eidx.size()) return 72;
    size_t observed = 0, fixed = 0, free_voxels = 0;
    for (const cg::EsdfVoxel& v : evox) {
      observed += v.observed;
      fixed += v.fixed;
      free_voxels += (v.observed && v.distance >= 0.3f);
      if (v.in_queue || (v.fixed && !v.observed)) return 73;
    }
    if (observed != est.observed_voxels || fixed != est.fixed_voxels || fixed == 0) return 74;
    std::vector<cg::PointXYZI> cloud;
    esdf.createFreePointcloud(0.3f, &cloud);
    if (cloud.size() != free_voxels) return 75;
    for (const cg::PointXYZI& p : cloud)
      if (!(p.intensity >= 0.3f)) return 76;
  }
  const size_t before = combined.getNumberOfAllocatedBlocks();
  const std::vector<uint8_t> moved =
      cg::reprojectSubmaps({&submap}, {T_M_S}, {T_M_S}, &combined);
  if (moved[0] != 0 || combined.getNumberOfAllocatedBlocks() != before) return 71;
  // listed-block download and the hash statistics: every allocated block found, an absent one not
  {
    cg::BlockIndexList all, ask;
    std::vector<cg::TsdfVoxel> vox, got;
    std::vector<uint8_t> found;
    combined.download(&all, &vox);
    ask.assign(all.begin(), all.begin() + std::min<size_t>(all.size(), 5));
    cg::BlockIndex absent;
    absent.x = 30000, absent.y = -30000, absent.z = 7;
    ask.push_back(absent);
    combined.downloadBlocks(ask, &got, &found);
    for (size_t i = 0; i + 1 < ask.size(); ++i)
      if (!found[i] || std::memcmp(&got[i * CG_VOXELS_PER_BLOCK], &vox[i * CG_VOXELS_PER_BLOCK],
                                   CG_VOXELS_PER_BLOCK * sizeof(cg::TsdfVoxel)) != 0)
        return 72;
    if (found.back()) return 73;
    const cg_hash_stats hs = combined.hashStats();
    if (hs.num_blocks != all.size()) return 74;
  }
  // the same frames as ONE pipelined job (staged copy, prepared first half) into a second
  // submap: same block count as the per-frame calls
  {
    FILE* again = fopen(argv[2], "rb");
    if (!again) return 75;
    uint32_t F2 = 0;
    float skip[9];
    if (!rd(again, &F2) || !rd(again, skip, 9)) return 76;
    std::vector<cg::Transformation> poses(F2);
    std::vector<uint64_t> offs(F2 + 1, 0);
    cg::Pointcloud pts;
    cg::Colors cols;
    for (uint32_t f = 0; f < F2; ++f) {
      uint32_t n = 0;
      if (!rd(again, &poses[f].qw, 7) || !rd(again, &n)) return 77;
      pts.resize(offs[f] + n);
      cols.resize(offs[f] + n);
      if (n && (!rd(again, pts.data() + offs[f], n) || !rd(again, cols.data() + offs[f], n))) return 78;
      offs[f + 1] = offs[f] + n;
    }
    fclose(again);
    cg::TsdfLayer submap2(ctx, voxel_size, 16, 2048);
    auto integ2 = cg::TsdfIntegratorFactory::create("fast", config, &submap2);
    ctx.stageBatchAsync(0, pts, cols);
    integ2->prepareStaged(0, poses, 0, offs);
    integ2->integratePrepared(0);
    if (submap2.getNumberOfAllocatedBlocks() != submap.getNumberOfAllocatedBlocks()) return 79;
  }
  std::printf("mesh: %zu triangles over %zu blocks\n", mesh.vertices.size() / 3,
              mesh.block_indices.size());
  std::printf("ok: submap %zu blocks, combined %zu blocks, %llu kernel launches\n",
              submap.getNumberOfAllocatedBlocks(), combined.getNumberOfAllocatedBlocks(),
              static_cast<unsigned long long>(ctx.kernelLaunches()));
  return 0;
}
