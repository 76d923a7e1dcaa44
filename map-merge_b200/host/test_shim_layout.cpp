// estimateMapsTransforms and composeMaps of the C++ API on raw maps, for tests/test_layout_gpu.py.
//   test_shim_layout <out_dir> <descriptor_type> <resolution> <map.bin>...
// Each map file holds float32[n][4] = x, y, z, rgba bits (an empty file is an empty map).  Writes <out_dir>/transforms.bin
// (float32[k][16], column-major) and <out_dir>/composed.bin (the composed cloud's PointT records exactly as they lie in memory).
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <vector>

#include <map_merge_3d/map_merging.h>

using namespace map_merge_3d;

static std::vector<float> read_file(const char* path)
{
  std::vector<float> v;
  FILE* f = std::fopen(path, "rb");
  if (!f) return v;
  std::fseek(f, 0, SEEK_END);
  const long bytes = std::ftell(f);
  std::fseek(f, 0, SEEK_SET);
  v.resize(bytes / sizeof(float));
  if (std::fread(v.data(), sizeof(float), v.size(), f) != v.size()) v.clear();
  std::fclose(f);
  return v;
}

static void write_file(const std::string& path, const void* data, size_t bytes)
{
  FILE* f = std::fopen(path.c_str(), "wb");
  if (!f || std::fwrite(data, 1, bytes, f) != bytes) {
    std::fprintf(stderr, "cannot write %s\n", path.c_str());
    std::exit(2);
  }
  std::fclose(f);
}

int main(int argc, char** argv)
{
  if (argc < 5) {
    std::fprintf(stderr, "usage: %s <out_dir> <descriptor_type> <resolution> <map.bin>...\n", argv[0]);
    return 2;
  }
  const std::string out_dir = argv[1];
  MapMergingParams params;
  params.descriptor_type = enums::from_string<Descriptor>(argv[2]);
  const double resolution = std::atof(argv[3]);
  std::vector<PointCloudConstPtr> clouds;
  for (int a = 4; a < argc; ++a) {
    const std::vector<float> raw = read_file(argv[a]);
    PointCloudPtr c(new PointCloud);
    c->points.resize(raw.size() / 4);
    for (size_t i = 0; i < c->points.size(); ++i) {
      PointT& p = c->points[i];
      p.x = raw[4 * i];
      p.y = raw[4 * i + 1];
      p.z = raw[4 * i + 2];
      std::memcpy(&p.rgba, &raw[4 * i + 3], 4);
    }
    c->width = (uint32_t)c->points.size();
    clouds.push_back(c);
  }
  const std::vector<Eigen::Matrix4f> T = estimateMapsTransforms(clouds, params);
  std::vector<float> t(T.size() * 16);
  for (size_t i = 0; i < T.size(); ++i) std::memcpy(&t[16 * i], T[i].data(), 64);
  write_file(out_dir + "/transforms.bin", t.data(), t.size() * sizeof(float));
  const PointCloudPtr out = composeMaps(clouds, T, resolution);
  write_file(out_dir + "/composed.bin", out->points.data(), out->points.size() * sizeof(PointT));
  std::printf("%zu transforms, %zu composed points\n", T.size(), out->points.size());
  return 0;
}
