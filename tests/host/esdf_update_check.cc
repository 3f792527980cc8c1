// esdf_update_check — drives EsdfIntegrator::updateFromTsdfLayer (coxgraph_b200.hpp) through a
// chain of layer edits and compares every result with updateFromTsdfLayerBatch on a copy of the
// layer in a second context, bit for bit.  tests/test_host_esdf_update.py runs it.
//   esdf_update_check nogpu -> exit 0 iff creating a context fails loudly
//   esdf_update_check run   -> exit 0 iff every step matched; one line per step on stdout
#include <cmath>
#include <cstdio>
#include <cstring>
#include <string>
#include <vector>

#include "../../coxgraph_b200/host/coxgraph_b200.hpp"

namespace cg = coxgraph_b200;

static bool same_esdf(const cg::BlockIndexList& ia, const std::vector<cg::EsdfVoxel>& va,
                      const cg::BlockIndexList& ib, const std::vector<cg::EsdfVoxel>& vb) {
  if (ia.size() != ib.size() || va.size() != vb.size()) return false;
  for (size_t i = 0; i < ia.size(); ++i)
    if (ia[i].x != ib[i].x || ia[i].y != ib[i].y || ia[i].z != ib[i].z) return false;
  for (size_t i = 0; i < va.size(); ++i) {
    const cg::EsdfVoxel &a = va[i], &b = vb[i];
    if (std::memcmp(&a.distance, &b.distance, sizeof(float)) != 0 || a.observed != b.observed ||
        a.hallucinated != b.hallucinated || a.fixed != b.fixed || a.parent[0] != b.parent[0] ||
        a.parent[1] != b.parent[1] || a.parent[2] != b.parent[2])
      return false;
  }
  return true;
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
  if (argc < 2 || std::string(argv[1]) != "run") return 64;
  const float vs = 0.05f;
  cg::Context ctx(0), ref_ctx(0);
  cg::TsdfLayer layer(ctx, vs, 16, 256);
  // a sphere of radius 0.6 m in a 6 x 4 x 2 block box, truncated at 0.16 m
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
          vox.push_back(v);
        }
      }
  layer.upload(idx, vox);
  cg::EsdfIntegrator::Config config;
  config.min_distance_m = 0.1f;
  cg::EsdfIntegrator esdf(config, &layer);
  int failures = 0;
  auto step = [&](const char* what, int want_full) {
    cg_esdf_stats st{};
    cg_esdf_update_stats ust{};
    esdf.updateFromTsdfLayer(true, &st, &ust);  // the flag is accepted and ignored
    cg::BlockIndexList got_idx, cur_idx, want_idx;
    std::vector<cg::EsdfVoxel> got, want;
    esdf.getEsdfLayer(&got_idx, &got);
    std::vector<cg::TsdfVoxel> cur;
    std::vector<uint8_t> flags;
    layer.download(&cur_idx, &cur, &flags);
    cg::TsdfLayer copy(ref_ctx, vs, 16, 256);
    copy.upload(cur_idx, cur, &flags);
    cg::EsdfIntegrator ref(config, &copy);
    cg_esdf_stats rst{};
    ref.updateFromTsdfLayerBatch(&rst);
    ref.getEsdfLayer(&want_idx, &want);
    const bool ok = same_esdf(got_idx, got, want_idx, want) && st.blocks == rst.blocks &&
                    st.observed_voxels == rst.observed_voxels && st.fixed_voxels == rst.fixed_voxels &&
                    ust.full_rebuild == want_full;
    std::printf("%s %s: blocks %llu changed %llu removed %llu region %llu full %d\n", ok ? "ok" : "MISMATCH",
                what, static_cast<unsigned long long>(st.blocks),
                static_cast<unsigned long long>(ust.blocks_changed),
                static_cast<unsigned long long>(ust.blocks_removed),
                static_cast<unsigned long long>(ust.blocks_region), ust.full_rebuild);
    failures += ok ? 0 : 1;
  };
  step("first", 1);
  vox[3 * 4096 + 1234].distance = 0.01f;  // a new fixed voxel in block 3
  layer.upload(idx, vox);
  step("fixed voxel", 0);
  layer.removeBlock(idx[7]);
  step("removed block", 0);
  layer.upload({cg::BlockIndex{6, 0, 0}}, std::vector<cg::TsdfVoxel>(vox.begin(), vox.begin() + 4096));
  step("new block", 0);
  step("unchanged", 0);
  return failures ? 1 : 0;
}
