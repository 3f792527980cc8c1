"""The depth-image contract restated in numpy float32: the cloud depth_image_proc's
point_cloud_xyzrgb publishes (depth_conversions.h convert<T>, depth_traits.h) for registered depth
and colour images, after voxblox_ros TsdfServer's convertPointcloud has dropped the points with a
non-finite coordinate.  numpy float32 arithmetic rounds every operation (no FMA), as the library
does.  `CONVERT_CC` is a verbatim C++ transcription of the same two steps; the CPU tests compile it
with -ffp-contract=off and check the two against each other."""
import numpy as np

# encoding -> ((r, g, b) byte offsets, bytes per pixel), as point_cloud_xyzrgb sets them
COLOR_LAYOUT = {"rgb8": ((0, 1, 2), 3), "rgba8": ((0, 1, 2), 4), "bgr8": ((2, 1, 0), 3),
                "bgra8": ((2, 1, 0), 4), "mono8": ((0, 0, 0), 1)}
DEPTH_ENCODINGS = ("16UC1", "32FC1")


def constants(cam):
    """(center_x, center_y, constant_x, constant_y) of convert<T> as float32."""
    unit = float(np.float32(0.001)) if cam["depth_encoding"] == "16UC1" else 1.0
    return (np.float32(cam["cx"]), np.float32(cam["cy"]), np.float32(unit / float(cam["fx"])),
            np.float32(unit / float(cam["fy"])))


def depth_cloud(depth, color, cam, form="contract"):
    """One frame: depth [H,W] (uint16 for 16UC1, float32 for 32FC1), color [H,W,pixel bytes] ->
    (points float32 [N,3], colors uint8 [N,4]) in row-major pixel order.

    form="contract" is the contract.  Two wrong forms exist so that the tests can show they tell
    them apart: "nan" keeps the invalid pixels as NaN points (N = H*W), "fma" rounds x and y once
    instead of after each operation (the fused evaluation)."""
    H, W = depth.shape
    cx, cy, kx, ky = constants(cam)
    d = depth.astype(np.float32)
    u = np.arange(W, dtype=np.float32)[None, :]
    v = np.arange(H, dtype=np.float32)[:, None]
    with np.errstate(all="ignore"):
        if form == "fma":
            x = ((u.astype(np.float64) - cx) * d * np.float64(kx)).astype(np.float32)
            y = ((v.astype(np.float64) - cy) * d * np.float64(ky)).astype(np.float32)
        else:
            x = ((u - cx) * d) * kx
            y = ((v - cy) * d) * ky
        z = d * np.float32(0.001) if cam["depth_encoding"] == "16UC1" else d.copy()
    x, y, z = np.broadcast_to(x, (H, W)), np.broadcast_to(y, (H, W)), z
    valid = depth != 0 if cam["depth_encoding"] == "16UC1" else np.isfinite(depth)
    pts = np.stack([x, y, z], axis=-1).reshape(-1, 3).astype(np.float32)
    pts[~valid.reshape(-1)] = np.nan
    (ro, go, bo), pix = COLOR_LAYOUT[cam["color_encoding"]]
    c = np.ascontiguousarray(color, np.uint8).reshape(H * W, pix)
    cols = np.stack([c[:, ro], c[:, go], c[:, bo], np.full(H * W, 255, np.uint8)], axis=1)
    if form != "nan":
        keep = np.isfinite(pts).all(axis=1)
        pts, cols = pts[keep], cols[keep]
    return np.ascontiguousarray(pts), np.ascontiguousarray(cols)


def depth_batch_cloud(depth, color, cam, form="contract"):
    """F frames -> (points, colors, frame_offsets uint64 [F+1]) for cg_integrate_batch_device."""
    parts = [depth_cloud(depth[f], color[f], cam, form) for f in range(len(depth))]
    offs = np.cumsum([0] + [len(p) for p, _ in parts]).astype(np.uint64)
    pts = np.concatenate([p for p, _ in parts]) if parts else np.zeros((0, 3), np.float32)
    cols = np.concatenate([c for _, c in parts]) if parts else np.zeros((0, 4), np.uint8)
    return pts, cols, offs


# depth_image_proc convert<T> (depth_conversions.h) over a PointCloud2 iterator, then voxblox's
# convertPointcloud filter (std::isfinite on x, y, z), kept verbatim apart from the containers.
# argv: depth encoding (0 = 16UC1, 1 = 32FC1), W, H, fx, fy, cx, cy (%a hex floats), colour pixel
# size, r/g/b offsets, depth file, colour file, output file.  Output: N, then N x (x, y, z float,
# r, g, b, a uint8).
CONVERT_CC = r"""
#include <cmath>
#include <cstdint>
#include <cstdio>
#include <cstdlib>
#include <limits>
#include <vector>

template <typename T> struct DepthTraits {};
template <> struct DepthTraits<uint16_t> {
  static inline bool valid(uint16_t depth) { return depth != 0; }
  static inline float toMeters(uint16_t depth) { return depth * 0.001f; }  // originally mm
};
template <> struct DepthTraits<float> {
  static inline bool valid(float depth) { return std::isfinite(depth); }
  static inline float toMeters(float depth) { return depth; }
};

struct PinholeCameraModel {  // image_geometry: the intrinsics are doubles
  double fx_, fy_, cx_, cy_;
  double fx() const { return fx_; }
  double fy() const { return fy_; }
  double cx() const { return cx_; }
  double cy() const { return cy_; }
};

struct Point { float x, y, z; uint8_t r, g, b, a; };

template <typename T>
void convert(const std::vector<uint8_t>& depth_data, int width, int height,
             const std::vector<uint8_t>& rgb_data, std::vector<Point>& cloud,
             const PinholeCameraModel& model, int red_offset, int green_offset, int blue_offset,
             int color_step) {
  // Use correct principal point from calibration
  float center_x = model.cx();
  float center_y = model.cy();

  // Combine unit conversion (if necessary) with scaling by focal length for computing (X,Y)
  double unit_scaling = DepthTraits<T>::toMeters(T(1));
  float constant_x = unit_scaling / model.fx();
  float constant_y = unit_scaling / model.fy();
  float bad_point = std::numeric_limits<float>::quiet_NaN();

  const T* depth_row = reinterpret_cast<const T*>(&depth_data[0]);
  int row_step = width;  // depth_msg->step / sizeof(T), tightly packed
  const uint8_t* rgb = &rgb_data[0];
  int rgb_skip = 0;  // rgb_msg->step - rgb_msg->width * color_step, tightly packed

  cloud.resize(static_cast<size_t>(width) * height);
  Point* iter = cloud.data();
  for (int v = 0; v < height; ++v, depth_row += row_step, rgb += rgb_skip) {
    for (int u = 0; u < width; ++u, rgb += color_step, ++iter) {
      T depth = depth_row[u];

      // Check for invalid measurements
      if (!DepthTraits<T>::valid(depth)) {
        iter->x = iter->y = iter->z = bad_point;
      } else {
        // Fill in XYZ
        iter->x = (u - center_x) * depth * constant_x;
        iter->y = (v - center_y) * depth * constant_y;
        iter->z = DepthTraits<T>::toMeters(depth);
      }

      // Fill in color
      iter->a = 255;
      iter->r = rgb[red_offset];
      iter->g = rgb[green_offset];
      iter->b = rgb[blue_offset];
    }
  }
}

static std::vector<uint8_t> slurp(const char* path) {
  std::vector<uint8_t> out;
  FILE* f = fopen(path, "rb");
  if (!f) exit(2);
  uint8_t buf[65536];
  size_t n;
  while ((n = fread(buf, 1, sizeof(buf), f)) > 0) out.insert(out.end(), buf, buf + n);
  fclose(f);
  return out;
}

int main(int argc, char** argv) {
  if (argc != 15) return 2;
  const int enc = atoi(argv[1]), width = atoi(argv[2]), height = atoi(argv[3]);
  PinholeCameraModel model{strtod(argv[4], nullptr), strtod(argv[5], nullptr),
                           strtod(argv[6], nullptr), strtod(argv[7], nullptr)};
  const int step = atoi(argv[8]), ro = atoi(argv[9]), go = atoi(argv[10]), bo = atoi(argv[11]);
  const std::vector<uint8_t> depth = slurp(argv[12]), rgb = slurp(argv[13]);
  std::vector<Point> cloud;
  if (enc == 0)
    convert<uint16_t>(depth, width, height, rgb, cloud, model, ro, go, bo, step);
  else
    convert<float>(depth, width, height, rgb, cloud, model, ro, go, bo, step);
  // voxblox convertPointcloud: skip the points with a non-finite coordinate
  std::vector<Point> kept;
  for (const Point& p : cloud)
    if (std::isfinite(p.x) && std::isfinite(p.y) && std::isfinite(p.z)) kept.push_back(p);
  FILE* f = fopen(argv[14], "wb");
  const uint64_t n = kept.size();
  fwrite(&n, sizeof(n), 1, f);
  for (const Point& p : kept) {
    fwrite(&p.x, 4, 3, f);
    const uint8_t c[4] = {p.r, p.g, p.b, p.a};
    fwrite(c, 1, 4, f);
  }
  fclose(f);
  return 0;
}
"""
