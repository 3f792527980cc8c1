// mesh_gather_check — saveAndPubCombinedMesh's PLY through the C++ mirror, on a one-rank
// communicator: generateMeshSharded -> gatherMeshSharded -> getConnectedMesh -> outputMeshAsPly
// must write the same file as generateMesh -> getConnectedMesh -> outputMeshAsPly of the same
// layer.  tests/test_host_mesh_gather.py runs it (libnccl.so.2 on the library path).
//   mesh_gather_check nogpu     -> exit 0 iff creating a context fails loudly
//   mesh_gather_check run DIR   -> exit 0 iff both PLY files (written to DIR) are identical and
//                                  the gathered mesh equals generateMesh's; one line per check
#include <cmath>
#include <cstdio>
#include <cstring>
#include <fstream>
#include <sstream>
#include <string>
#include <vector>

#include "../../coxgraph_b200/host/coxgraph_b200.hpp"

namespace cg = coxgraph_b200;

static std::string slurp(const std::string& path) {
  std::ifstream f(path, std::ios::binary);
  std::stringstream ss;
  ss << f.rdbuf();
  return ss.str();
}

template <class T>
static bool same_bytes(const std::vector<T>& a, const std::vector<T>& b) {
  return a.size() == b.size() && (a.empty() || std::memcmp(a.data(), b.data(), a.size() * sizeof(T)) == 0);
}

static bool same_mesh(const cg::LayerMesh& a, const cg::LayerMesh& b) {
  return same_bytes(a.block_indices, b.block_indices) && same_bytes(a.vertex_begin, b.vertex_begin) &&
         same_bytes(a.vertices, b.vertices) && same_bytes(a.normals, b.normals) &&
         same_bytes(a.colors, b.colors);
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
  if (argc < 3 || std::string(argv[1]) != "run") return 64;
  const std::string dir = argv[2];
  const float vs = 0.05f;
  cg::Context ctx(0);
  cg::commInit(ctx, cg::commUniqueId(), 0, 1);
  cg::TsdfLayer layer(ctx, vs, 16, 256);
  // a sphere of radius 0.6 m in a 6 x 4 x 2 block box, truncated at 0.16 m, coloured by position
  cg::BlockIndexList idx;
  std::vector<cg::TsdfVoxel> vox;
  for (int bz = 0; bz < 2; ++bz)
    for (int by = 0; by < 4; ++by)
      for (int bx = 0; bx < 6; ++bx) {
        idx.push_back({bx, by, bz});
        for (int i = 0; i < 4096; ++i) {
          const float x = (bx * 16 + (i & 15) + 0.5f) * vs - 2.4f, y = (by * 16 + ((i >> 4) & 15) + 0.5f) * vs - 1.6f,
                      z = (bz * 16 + (i >> 8) + 0.5f) * vs - 0.8f;
          cg::TsdfVoxel v{};
          v.distance = std::fmax(-0.16f, std::fmin(0.16f, std::sqrt(x * x + y * y + z * z) - 0.6f));
          v.weight = (i % 17 == 0) ? 0.0f : 1.0f;
          v.r = static_cast<uint8_t>(40 * bx + (i & 15));
          v.g = static_cast<uint8_t>(60 * by + ((i >> 4) & 15));
          v.b = static_cast<uint8_t>(100 * bz + (i >> 8));
          v.a = 255;
          vox.push_back(v);
        }
      }
  layer.upload(idx, vox);
  int failures = 0;
  auto report = [&](bool ok, const char* what) {
    std::printf("%s %s\n", ok ? "ok" : "MISMATCH", what);
    failures += ok ? 0 : 1;
  };

  cg::LayerMesh own, gathered;
  cg::generateMeshSharded(layer, &own);
  const auto totals = cg::gatherMeshSharded(ctx, 0, &gathered);
  cg::ConnectedMesh sharded_connected;
  cg::getConnectedMesh(layer, &sharded_connected);
  const std::string sharded_ply = dir + "/sharded.ply", single_ply = dir + "/single.ply";
  const bool wrote_sharded = cg::outputMeshAsPly(sharded_ply, sharded_connected);

  cg::LayerMesh single;
  cg::generateMesh(layer, &single);
  cg::ConnectedMesh single_connected;
  cg::getConnectedMesh(layer, &single_connected);
  const bool wrote_single = cg::outputMeshAsPly(single_ply, single_connected);

  report(totals.first == single.block_indices.size() && totals.second == single.vertices.size() &&
             !single.vertices.empty(),
         "global totals");
  report(same_mesh(gathered, single), "gathered mesh == generateMesh");
  const std::string a = slurp(sharded_ply), b = slurp(single_ply);
  report(wrote_sharded && wrote_single && !a.empty() && a == b, "PLY files identical");

  // a mesh is gathered once per generateMeshSharded
  cg::generateMeshSharded(layer, &own);
  cg::gatherMeshSharded(ctx, 0, nullptr);
  bool rejected = false;
  try {
    cg::gatherMeshSharded(ctx, 0, nullptr);
  } catch (const cg::Error& e) {
    rejected = e.status == CG_ERR_INVALID_ARG;
  }
  report(rejected, "second gather rejected");
  std::printf("%zu blocks, %zu vertices, %zu connected vertices, %zu PLY bytes\n", totals.first,
              totals.second, single_connected.vertices.size(), a.size());
  return failures ? 1 : 0;
}
