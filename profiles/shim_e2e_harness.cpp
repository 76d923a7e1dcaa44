// shim_e2e_harness.cpp — end-to-end time of the C++ API's two hot calls against the paths around them (profiles/shim_e2e.py
// builds and drives it).
//   shim_e2e_harness estimate|compose <timed calls> <map.bin>...   (map files: float32[n][4] = x, y, z, rgba bits)
// Variants, run alternately after one warm-up call each:
//   a  the previous C++ path: single-thread pack() of every pcl::PointXYZRGB into a pageable std::vector<float>, the packed
//      C ABI call, and for composeMaps the per-point unpack() into a new cloud
//   b  map_merge_3d::estimateMapsTransforms / composeMaps (host/shim.cpp: the points go to the library as they lie)
//   c  the C ABI on pinned, pre-packed 16-byte points (bench.py's e2e path); the composed points stay in the output pool
// Prints one JSON object: per-variant call times (ms) and whether the three results are bit-identical.
//   shim_e2e_harness upload <timed calls> <map.bin>...
// The staged upload inside b on its own (mm3d_maps_upload_layout with the PointT layout): call times, the per-kernel profile
// of one call, and the time of the same bytes' host-to-device copies from one pinned 8 MiB slot.  Run with MM3D_HOST_TRACE=1
// the library adds its host copy time per call on stderr.
#include <cuda_runtime.h>

#include <algorithm>
#include <chrono>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <string>
#include <vector>

#include <map_merge_3d/map_merging.h>

#include "../include/mm3d.h"

using namespace map_merge_3d;

static double now_ms() { return std::chrono::duration<double, std::milli>(std::chrono::steady_clock::now().time_since_epoch()).count(); }

static void die(const char* what)
{
  std::fprintf(stderr, "shim_e2e_harness: %s\n", what);
  std::exit(2);
}

static std::vector<float> pack(const PointCloud* cloud)  // the shim's former pack()
{
  std::vector<float> out;
  if (!cloud) return out;
  out.resize(cloud->points.size() * 4);
  for (size_t i = 0; i < cloud->points.size(); ++i) {
    const PointT& p = cloud->points[i];
    out[4 * i] = p.x;
    out[4 * i + 1] = p.y;
    out[4 * i + 2] = p.z;
    std::memcpy(&out[4 * i + 3], &p.rgba, 4);
  }
  return out;
}

static PointCloudPtr unpack(const float* pts, uint64_t n)  // the shim's unpack(), still used by its low-level functions
{
  PointCloudPtr out(new PointCloud);
  out->points.resize(n);
  for (uint64_t i = 0; i < n; ++i) {
    PointT& p = out->points[i];
    p.x = pts[4 * i];
    p.y = pts[4 * i + 1];
    p.z = pts[4 * i + 2];
    std::memcpy(&p.rgba, &pts[4 * i + 3], 4);
  }
  out->width = (uint32_t)n;
  out->height = 1;
  out->is_dense = true;
  return out;
}

int main(int argc, char** argv)
{
  if (argc < 5) die("usage: shim_e2e_harness estimate|compose <timed calls> <map.bin>...");
  const bool compose = std::strcmp(argv[1], "compose") == 0;
  const int reps = std::atoi(argv[2]);
  std::vector<PointCloudConstPtr> clouds;
  std::vector<float*> pinned;
  std::vector<uint64_t> sizes;
  for (int a = 3; a < argc; ++a) {
    FILE* f = std::fopen(argv[a], "rb");
    if (!f) die("cannot open a map file");
    std::fseek(f, 0, SEEK_END);
    const size_t n = (size_t)std::ftell(f) / 16;
    std::fseek(f, 0, SEEK_SET);
    float* p = nullptr;
    if (cudaHostAlloc((void**)&p, std::max<size_t>(n, 1) * 16, cudaHostAllocDefault) != cudaSuccess) die("cudaHostAlloc failed");
    if (std::fread(p, 16, n, f) != n) die("short read");
    std::fclose(f);
    PointCloudPtr c(new PointCloud);
    c->points.resize(n);
    for (size_t i = 0; i < n; ++i) {
      c->points[i].x = p[4 * i];
      c->points[i].y = p[4 * i + 1];
      c->points[i].z = p[4 * i + 2];
      std::memcpy(&c->points[i].rgba, &p[4 * i + 3], 4);
    }
    c->width = (uint32_t)n;
    clouds.push_back(c);
    pinned.push_back(p);
    sizes.push_back(n);
  }
  const int M = (int)clouds.size();
  mm3d_ctx* ctx = nullptr;
  if (mm3d_create(&ctx, 0, nullptr) != MM3D_OK) die("mm3d_create failed");
  MapMergingParams params;
  params.descriptor_type = Descriptor::FPFH;  // bench.py's c3
  mm3d_params cp;
  mm3d_params_default(&cp);
  cp.descriptor_type = MM3D_DESC_FPFH;
  const double res = 0.05;                    // bench.py's c5
  std::vector<float> T(16 * M, 0.f);
  for (int m = 0; m < M; ++m) T[16 * m] = T[16 * m + 5] = T[16 * m + 10] = T[16 * m + 15] = 1.f;
  std::vector<Eigen::Matrix4f> Te(M, Eigen::Matrix4f::Identity());

  std::vector<float> out_a(16 * M), out_b(16 * M), out_c(16 * M);  // estimate
  std::vector<unsigned char> rec_a, rec_b;                          // compose: PointT records
  std::vector<float> pts_c;                                         // compose: packed points
  auto run = [&](char v) {
    const double t0 = now_ms();
    double t1 = 0.0;  // the copies of the composed results into rec_* / pts_c are not part of a call: timed out
    if (!compose) {
      int n_out = 0;
      if (v == 'a') {
        std::vector<std::vector<float>> packed(M);
        std::vector<const float*> ptrs(M);
        for (int m = 0; m < M; ++m) {
          packed[m] = pack(clouds[m].get());
          ptrs[m] = packed[m].empty() ? nullptr : packed[m].data();
        }
        if (mm3d_estimate_maps_transforms(ctx, M, ptrs.data(), sizes.data(), &cp, out_a.data(), &n_out) != MM3D_OK) die(mm3d_last_error(ctx));
      } else if (v == 'b') {
        const std::vector<Eigen::Matrix4f> r = estimateMapsTransforms(clouds, params);
        for (size_t i = 0; i < r.size(); ++i) std::memcpy(&out_b[16 * i], r[i].data(), 64);
      } else {
        if (mm3d_estimate_maps_transforms(ctx, M, (const float* const*)pinned.data(), sizes.data(), &cp, out_c.data(), &n_out) != MM3D_OK)
          die(mm3d_last_error(ctx));
      }
    } else {
      float* out = nullptr;
      uint64_t n = 0;
      if (v == 'a') {
        std::vector<std::vector<float>> packed(M);
        std::vector<const float*> ptrs(M);
        for (int m = 0; m < M; ++m) {
          packed[m] = pack(clouds[m].get());
          ptrs[m] = packed[m].empty() ? nullptr : packed[m].data();
        }
        if (mm3d_compose_maps(ctx, M, ptrs.data(), sizes.data(), M, T.data(), res, &out, &n) != MM3D_OK) die(mm3d_last_error(ctx));
        PointCloudPtr r = unpack(out, n);
        mm3d_free(out);
        t1 = now_ms();
        rec_a.assign((const unsigned char*)r->points.data(), (const unsigned char*)(r->points.data() + r->points.size()));
      } else if (v == 'b') {
        PointCloudPtr r = composeMaps(clouds, Te, res);
        t1 = now_ms();
        rec_b.assign((const unsigned char*)r->points.data(), (const unsigned char*)(r->points.data() + r->points.size()));
      } else {
        if (mm3d_compose_maps(ctx, M, (const float* const*)pinned.data(), sizes.data(), M, T.data(), res, &out, &n) != MM3D_OK)
          die(mm3d_last_error(ctx));
        t1 = now_ms();
        pts_c.assign(out, out + 4 * n);
        mm3d_free(out);
      }
    }
    return (t1 > 0.0 ? t1 : now_ms()) - t0;
  };
  auto list = [](const std::vector<double>& v) {
    std::string s = "[";
    for (size_t i = 0; i < v.size(); ++i) s += (i ? ", " : "") + std::to_string(v[i]);
    return s + "]";
  };
  if (std::strcmp(argv[1], "upload") == 0) {
    static const PointT proto;
    const mm3d_layout l = {(uint32_t)sizeof(PointT), (int32_t)((const char*)&proto.x - (const char*)&proto),
                           (int32_t)((const char*)&proto.y - (const char*)&proto), (int32_t)((const char*)&proto.z - (const char*)&proto),
                           (int32_t)((const char*)&proto.rgba - (const char*)&proto), &proto};
    std::vector<const void*> ptrs(M);
    size_t bytes = 0;
    for (int m = 0; m < M; ++m) {
      ptrs[m] = clouds[m]->points.data();
      bytes += sizes[m] * sizeof(PointT);
    }
    auto upload = [&] {
      mm3d_maps* maps = nullptr;
      const double t0 = now_ms();
      if (mm3d_maps_upload_layout(ctx, M, ptrs.data(), sizes.data(), &l, &maps) != MM3D_OK) die(mm3d_last_error(ctx));
      const double ms = now_ms() - t0;
      mm3d_maps_free(maps);
      return ms;
    };
    upload();
    std::vector<double> tu;
    for (int r = 0; r < reps; ++r) tu.push_back(upload());
    char* prof = nullptr;
    mm3d_profile_begin(ctx);
    upload();
    mm3d_profile_end(ctx, &prof);
    const size_t slot = (size_t)8 << 20;
    void *h = nullptr, *d = nullptr;
    if (cudaHostAlloc(&h, slot, cudaHostAllocDefault) != cudaSuccess || cudaMalloc(&d, slot) != cudaSuccess) die("staging buffers");
    std::memset(h, 0, slot);
    cudaEvent_t e0, e1;
    cudaEventCreate(&e0);
    cudaEventCreate(&e1);
    std::vector<double> tcp;
    for (int r = 0; r < reps + 1; ++r) {
      cudaEventRecord(e0, 0);
      for (size_t o = 0; o < bytes; o += slot) cudaMemcpyAsync(d, h, std::min(slot, bytes - o), cudaMemcpyHostToDevice, 0);
      cudaEventRecord(e1, 0);
      cudaEventSynchronize(e1);
      float ms = 0.f;
      cudaEventElapsedTime(&ms, e0, e1);
      if (r) tcp.push_back(ms);
    }
    std::printf("{\"workload\": \"upload\", \"maps\": %d, \"record_bytes\": %zu, \"upload_ms\": %s, \"h2d_copy_ms\": %s, \"profile\": %s}\n", M, bytes,
                list(tu).c_str(), list(tcp).c_str(), prof ? prof : "null");
    mm3d_free(prof);
    cudaFreeHost(h);
    cudaFree(d);
    mm3d_destroy(ctx);
    return 0;
  }
  std::vector<double> ta, tb, tc;
  for (char v : {'a', 'b', 'c'}) run(v);  // warm-up
  for (int r = 0; r < reps; ++r) {
    for (char v : {'a', 'b', 'c'}) {
      const double ms = run(v);
      (v == 'a' ? ta : v == 'b' ? tb : tc).push_back(ms);
    }
  }
  bool same = true;
  if (!compose) {
    same = std::memcmp(out_a.data(), out_b.data(), out_a.size() * 4) == 0 && std::memcmp(out_b.data(), out_c.data(), out_b.size() * 4) == 0;
  } else {
    same = rec_a.size() == rec_b.size() && std::memcmp(rec_a.data(), rec_b.data(), rec_a.size()) == 0 && pts_c.size() / 4 * sizeof(PointT) == rec_b.size();
    for (size_t i = 0; same && i < pts_c.size() / 4; ++i) {
      const PointT& p = ((const PointT*)rec_b.data())[i];
      same = std::memcmp(&p.x, &pts_c[4 * i], 12) == 0 && std::memcmp(&p.rgba, &pts_c[4 * i + 3], 4) == 0;
    }
  }
  std::printf("{\"workload\": \"%s\", \"maps\": %d, \"points\": %llu, \"output_points\": %zu, \"a_ms\": %s, \"b_ms\": %s, \"c_ms\": %s, "
              "\"bit_identical\": %s}\n",
              compose ? "compose" : "estimate", M, (unsigned long long)[&] { uint64_t s = 0; for (uint64_t n : sizes) s += n; return s; }(),
              compose ? rec_b.size() / sizeof(PointT) : (size_t)0, list(ta).c_str(), list(tb).c_str(), list(tc).c_str(), same ? "true" : "false");
  mm3d_destroy(ctx);
  for (float* p : pinned) cudaFreeHost(p);
  return same ? 0 : 1;
}
