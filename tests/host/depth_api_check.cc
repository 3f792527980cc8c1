// depth_api_check — integrates registered depth + colour images through the C++ host API
// (TsdfIntegratorBase::integrateDepthImage / integrateDepthImages, coxgraph_b200.hpp) the way a
// node that receives sensor_msgs/Image pairs would.  tests/test_host_depth.py writes the frames,
// runs this program on the GPU box and compares the layer with the Python path, bit for bit.
//   depth_api_check nogpu                  -> exit 0 iff creating a context fails loudly
//   depth_api_check run <in.bin> <out.bin> -> frame 0 alone, then the others as one job
// in.bin : u32 F, i32 W, H, depth encoding, colour encoding, f64 fx, fy, cx, cy, f32 voxel_size,
//          f32 trunc, then per frame: f32 T[7], W*H depth pixels, W*H colour pixels
// out.bin: u32 B, B * 3 i32, B * 4096 * 12 B voxels, B flag bytes
#include <cstdio>
#include <string>
#include <vector>

#include "../../coxgraph_b200/host/coxgraph_b200.hpp"

namespace cg = coxgraph_b200;

template <class T>
static bool rd(FILE* f, T* p, size_t n = 1) { return fread(p, sizeof(T), n, f) == n; }

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
  if (argc < 4 || std::string(argv[1]) != "run") return 64;
  FILE* in = fopen(argv[2], "rb");
  if (!in) return 65;
  uint32_t F = 0;
  cg_depth_camera cam{};
  float voxel_size = 0, trunc = 0;
  if (!rd(in, &F) || !rd(in, &cam.width) || !rd(in, &cam.height) || !rd(in, &cam.depth_encoding) ||
      !rd(in, &cam.color_encoding) || !rd(in, &cam.fx) || !rd(in, &cam.fy) || !rd(in, &cam.cx) ||
      !rd(in, &cam.cy) || !rd(in, &voxel_size) || !rd(in, &trunc) || F == 0)
    return 66;
  const size_t px = static_cast<size_t>(cam.width) * cam.height;
  const size_t dsize = cam.depth_encoding == CG_DEPTH_16UC1 ? 2 : 4;
  const size_t csize = cam.color_encoding == CG_COLOR_MONO8 ? 1
                       : (cam.color_encoding == CG_COLOR_RGBA8 ||
                          cam.color_encoding == CG_COLOR_BGRA8) ? 4 : 3;
  std::vector<cg::Transformation> poses(F);
  std::vector<std::vector<uint8_t>> depth(F, std::vector<uint8_t>(px * dsize)),
      color(F, std::vector<uint8_t>(px * csize));
  for (uint32_t f = 0; f < F; ++f)
    if (!rd(in, &poses[f].qw, 7) || !rd(in, depth[f].data(), depth[f].size()) ||
        !rd(in, color[f].data(), color[f].size()))
      return 67;
  fclose(in);
  cg::Context ctx(0);
  cg::TsdfLayer layer(ctx, voxel_size, 16, 4096);
  cg::TsdfIntegratorBase::Config config;
  config.default_truncation_distance = trunc;
  cg::TsdfIntegratorBase integrator(config, &layer);
  integrator.integrateDepthImage(poses[0], {depth[0].data()}, {color[0].data()}, cam);
  std::vector<cg::Transformation> rest(poses.begin() + 1, poses.end());
  std::vector<cg::TsdfIntegratorBase::DepthImage> d;
  std::vector<cg::TsdfIntegratorBase::ColorImage> c;
  for (uint32_t f = 1; f < F; ++f) {
    d.push_back({depth[f].data()});
    c.push_back({color[f].data()});
  }
  if (!rest.empty()) integrator.integrateDepthImages(rest, d, c, cam);
  cg::BlockIndexList idx;
  std::vector<cg::TsdfVoxel> vox;
  std::vector<uint8_t> flags;
  layer.download(&idx, &vox, &flags);
  FILE* out = fopen(argv[3], "wb");
  if (!out) return 69;
  const uint32_t B = static_cast<uint32_t>(idx.size());
  fwrite(&B, 4, 1, out);
  if (B) {
    fwrite(idx.data(), sizeof(cg::BlockIndex), B, out);
    fwrite(vox.data(), sizeof(cg::TsdfVoxel), vox.size(), out);
    fwrite(flags.data(), 1, B, out);
  }
  fclose(out);
  return 0;
}
