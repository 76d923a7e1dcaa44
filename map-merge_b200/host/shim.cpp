// shim.cpp — map_merge_3d's C++ API (include/map_merge_3d/*.h) implemented on the C ABI of libmm3d.
//
// Function-for-function stand-in for the reference's static library `map_merging`
// (map_merge_3d/CMakeLists.txt:67-74: features.cpp, matching.cpp, map_merging.cpp, graph.cpp).
// Only data marshalling happens here: estimateMapsTransforms and composeMaps hand PCL's 32-byte points to the library as
// they are (mm3d_layout; the GPU converts them), the low-level functions pack them to the 16-byte device layout, and errors
// become the exceptions / in-band sentinels the reference uses.  There is no CPU fallback.
#include <map_merge_3d/map_merging.h>

#include <cstdlib>
#include <cstring>
#include <mutex>
#include <stdexcept>
#include <string>

#include "../../include/mm3d.h"

namespace map_merge_3d
{
namespace
{
// One context per thread: the ROS node calls estimateMapsTransforms and composeMaps from different
// spinner threads at the same time (map_merge_node.cpp:32-40, 264-265); contexts share nothing.
mm3d_ctx* context()
{
  struct Holder {
    mm3d_ctx* c = nullptr;
    ~Holder() { mm3d_destroy(c); }
  };
  static thread_local Holder h;
  if (!h.c) {
    // MM3D_DEVICE=n: that device only.  MM3D_DEVICES=0,2,3: those devices.  Neither: every visible device —
    // estimateMapsTransforms and composeMaps shard their maps and pairs over all of them (include/mm3d.h, multi-GPU interface).
    int rc;
    if (const char* e = std::getenv("MM3D_DEVICE")) {
      rc = mm3d_create(&h.c, std::atoi(e), nullptr);
    } else {
      std::vector<int> devs;
      if (const char* l = std::getenv("MM3D_DEVICES")) {
        const char* p = l;
        while (*p) {
          char* end = nullptr;
          const long v = std::strtol(p, &end, 10);
          if (end == p) break;
          devs.push_back((int)v);
          p = (*end == ',') ? end + 1 : end;
        }
      }
      rc = mm3d_create_multi(&h.c, devs.empty() ? nullptr : devs.data(), (int)devs.size());
      if (rc == MM3D_ERR_UNSUPPORTED) rc = mm3d_create(&h.c, devs.empty() ? 0 : devs[0], nullptr);  // no NCCL on this machine: one GPU
    }
    if (rc != MM3D_OK) throw std::runtime_error("libmm3d: no usable CUDA device (the registration path has no CPU fallback)");
  }
  return h.c;
}

void check(int rc)
{
  if (rc < 0) throw std::runtime_error(std::string("libmm3d: ") + mm3d_last_error(context()));
}

std::vector<float> pack(const PointCloud* cloud)
{
  std::vector<float> out;
  if (!cloud) return out;  // a robot that has not published yet: treated as an empty map
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

PointCloudPtr unpack(const float* pts, uint64_t n)
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

// Where x, y, z and rgba sit in a PointT, taken from a default-constructed point (PCL's PointXYZRGB is not standard-layout,
// so offsetof does not apply); output records start as that point's bytes.
const mm3d_layout& point_layout()
{
  static const PointT proto;
  auto at = [](const void* field) { return (int32_t)((const char*)field - (const char*)&proto); };
  static const mm3d_layout l = {(uint32_t)sizeof(PointT), at(&proto.x), at(&proto.y), at(&proto.z), at(&proto.rgba), &proto};
  return l;
}

// the points of each cloud as they lie in memory; a null or empty cloud is an empty map
void point_arrays(const std::vector<PointCloudConstPtr>& clouds, std::vector<const void*>& ptrs, std::vector<uint64_t>& sizes)
{
  ptrs.assign(clouds.size(), nullptr);
  sizes.assign(clouds.size(), 0);
  for (size_t i = 0; i < clouds.size(); ++i)
    if (clouds[i] && !clouds[i]->points.empty()) {
      ptrs[i] = clouds[i]->points.data();
      sizes[i] = clouds[i]->points.size();
    }
}

std::vector<float> pack_normals(const SurfaceNormals& nm)
{
  std::vector<float> out(nm.points.size() * 4);
  for (size_t i = 0; i < nm.points.size(); ++i) {
    out[4 * i] = nm.points[i].normal_x;
    out[4 * i + 1] = nm.points[i].normal_y;
    out[4 * i + 2] = nm.points[i].normal_z;
    out[4 * i + 3] = nm.points[i].curvature;
  }
  return out;
}

struct DescInfo {
  const char* field;  // PCLPointCloud2 field name (dispatch_descriptors.h:38-48)
  int dim;
  int id;
};
const DescInfo kDesc[] = {{"pfh", 125, MM3D_DESC_PFH},  {"pfhrgb", 250, MM3D_DESC_PFHRGB}, {"fpfh", 33, MM3D_DESC_FPFH},
                          {"r_min", 2, MM3D_DESC_RSD},  {"shot", 1344, MM3D_DESC_SHOT},    {"shape_context", 1980, MM3D_DESC_SC3D}};

const DescInfo& desc_by_name(const std::string& name)
{
  for (const DescInfo& d : kDesc)
    if (name == d.field) return d;
  throw std::runtime_error("unknown descriptor type");
}

// descriptors travel as a PCLPointCloud2 whose first field names the type (features.cpp:146-147, matching.cpp:102)
LocalDescriptorsPtr make_descriptors(const DescInfo& d, const float* data, uint64_t n)
{
  LocalDescriptorsPtr out(new LocalDescriptors);
  pcl::PCLPointField f;
  f.name = d.field;
  f.offset = 0;
  f.datatype = 7;
  f.count = (uint32_t)d.dim;
  out->fields.push_back(f);
  out->point_step = (uint32_t)d.dim * 4;
  out->width = (uint32_t)n;
  out->height = 1;
  out->row_step = out->point_step * out->width;
  out->data.resize((size_t)n * d.dim * 4);
  if (n) std::memcpy(out->data.data(), data, out->data.size());
  return out;
}

void assertDescriptorsPair(const LocalDescriptorsPtr& a, const LocalDescriptorsPtr& b)
{
  if (a->fields.empty() || b->fields.empty())
    throw std::runtime_error("descriptors must contain at least one field with descriptors.");
}

Eigen::Matrix4f to_matrix(const float* colmajor)
{
  Eigen::Matrix4f m;
  std::memcpy(m.data(), colmajor, 64);
  return m;
}

mm3d_params to_c(const MapMergingParams& p)
{
  mm3d_params c;
  c.resolution = p.resolution;
  c.descriptor_radius = p.descriptor_radius;
  c.outliers_min_neighbours = p.outliers_min_neighbours;
  c.normal_radius = p.normal_radius;
  c.keypoint_type = (int32_t)p.keypoint_type;
  c.keypoint_threshold = p.keypoint_threshold;
  c.descriptor_type = (int32_t)p.descriptor_type;
  c.estimation_method = (int32_t)p.estimation_method;
  c.refine_transform = p.refine_transform ? 1 : 0;
  c.inlier_threshold = p.inlier_threshold;
  c.max_correspondence_distance = p.max_correspondence_distance;
  c.max_iterations = p.max_iterations;
  c.matching_k = p.matching_k;
  c.transform_epsilon = p.transform_epsilon;
  c.confidence_threshold = p.confidence_threshold;
  c.output_resolution = p.output_resolution;
  return c;
}

// pcl::console::parse_argument: value = the argument following the LAST occurrence of the flag
template <typename F>
void parse_argument(int argc, char** argv, const char* flag, F assign)
{
  for (int i = argc - 2; i >= 1; --i)
    if (std::strcmp(argv[i], flag) == 0) {
      assign(argv[i + 1]);
      return;
    }
}
}  // namespace

// ---------------------------------------------------------------- features.h
PointCloudPtr downSample(const PointCloudConstPtr& input, double resolution)
{
  std::vector<float> in = pack(input.get());
  if (in.empty()) return PointCloudPtr(new PointCloud);  // no device needed (test_map_merging.cpp:34-40)
  float* out = nullptr;
  uint64_t n = 0;
  check(mm3d_downsample(context(), in.data(), in.size() / 4, resolution, &out, &n));
  PointCloudPtr r = unpack(out, n);
  mm3d_free(out);
  return r;
}

PointCloudPtr removeOutliers(const PointCloudConstPtr& input, double radius, int min_neighbours)
{
  std::vector<float> in = pack(input.get());
  if (in.empty()) return PointCloudPtr(new PointCloud);
  float* out = nullptr;
  uint64_t n = 0;
  check(mm3d_remove_outliers(context(), in.data(), in.size() / 4, radius, min_neighbours, 0.0, &out, &n, nullptr));
  PointCloudPtr r = unpack(out, n);
  mm3d_free(out);
  return r;
}

SurfaceNormalsPtr computeSurfaceNormals(const PointCloudConstPtr& input, double radius)
{
  SurfaceNormalsPtr r(new SurfaceNormals);
  std::vector<float> in = pack(input.get());
  if (in.empty()) return r;
  float* out = nullptr;
  check(mm3d_normals(context(), in.data(), in.size() / 4, radius, 0.0, &out));
  r->points.resize(in.size() / 4);
  for (size_t i = 0; i < r->points.size(); ++i) {
    r->points[i].normal_x = out[4 * i];
    r->points[i].normal_y = out[4 * i + 1];
    r->points[i].normal_z = out[4 * i + 2];
    r->points[i].curvature = out[4 * i + 3];
    if (out[4 * i] != out[4 * i]) r->is_dense = false;
  }
  r->width = (uint32_t)r->points.size();
  mm3d_free(out);
  return r;
}

PointCloudPtr detectKeypoints(const PointCloudConstPtr& points, const SurfaceNormalsPtr& normals, Keypoint type, double threshold, double radius,
                              double resolution)
{
  std::vector<float> in = pack(points.get());
  if (in.empty()) return PointCloudPtr(new PointCloud);
  std::vector<float> nm = normals ? pack_normals(*normals) : std::vector<float>();
  float* out = nullptr;
  uint64_t n = 0;
  check(mm3d_keypoints(context(), in.data(), in.size() / 4, nm.empty() ? nullptr : nm.data(), (int)type, threshold, radius, resolution, &out, &n,
                       nullptr, nullptr));
  PointCloudPtr r = unpack(out, n);
  mm3d_free(out);
  return r;
}

LocalDescriptorsPtr computeLocalDescriptors(const PointCloudConstPtr& points, const SurfaceNormalsPtr& normals, const PointCloudPtr& keypoints,
                                            Descriptor descriptor, double feature_radius)
{
  const DescInfo& d = kDesc[(int)descriptor];
  std::vector<float> in = pack(points.get()), kp = pack(keypoints.get());
  std::vector<float> nm = pack_normals(*normals);
  float *kout = nullptr, *desc = nullptr;
  uint64_t n = 0;
  int dim = 0;
  check(mm3d_descriptors(context(), in.data(), in.size() / 4, nm.data(), kp.data(), kp.size() / 4, d.id, feature_radius, 0.0, &kout, &n, &desc,
                         &dim, nullptr));
  PointCloudPtr kept = unpack(kout, n);
  *keypoints = *kept;  // keypoints and descriptors stay synchronised (features.cpp:137-141)
  LocalDescriptorsPtr r = make_descriptors(d, desc, n);
  mm3d_free(kout);
  mm3d_free(desc);
  return r;
}

// ---------------------------------------------------------------- matching.h
CorrespondencesPtr findFeatureCorrespondences(const LocalDescriptorsPtr& source_descriptors, const LocalDescriptorsPtr& target_descriptors, size_t k)
{
  assertDescriptorsPair(source_descriptors, target_descriptors);
  const DescInfo& d = desc_by_name(source_descriptors->fields[0].name);
  int32_t* pairs = nullptr;
  float* dist = nullptr;
  uint64_t nc = 0;
  check(mm3d_match(context(), (const float*)source_descriptors->data.data(), source_descriptors->width, (const float*)target_descriptors->data.data(),
                   target_descriptors->width, d.dim, k, &pairs, &dist, &nc));
  CorrespondencesPtr r(new Correspondences);
  r->reserve(nc);
  for (uint64_t i = 0; i < nc; ++i) r->emplace_back(pairs[2 * i], pairs[2 * i + 1], dist[i]);
  mm3d_free(pairs);
  mm3d_free(dist);
  return r;
}

Eigen::Matrix4f estimateTransformFromCorrespondences(const PointCloudPtr& source_keypoints, const PointCloudPtr& target_keypoints,
                                                     const CorrespondencesPtr& correspondences, CorrespondencesPtr& inliers, double inlier_threshold)
{
  inliers.reset(new Correspondences);
  std::vector<float> s = pack(source_keypoints.get()), t = pack(target_keypoints.get());
  std::vector<int32_t> pairs(correspondences->size() * 2);
  for (size_t i = 0; i < correspondences->size(); ++i) {
    pairs[2 * i] = (*correspondences)[i].index_query;
    pairs[2 * i + 1] = (*correspondences)[i].index_match;
  }
  float T[16];
  int32_t* inl = nullptr;
  uint64_t ni = 0;
  check(mm3d_ransac(context(), s.data(), s.size() / 4, t.data(), t.size() / 4, pairs.data(), correspondences->size(), inlier_threshold, T, &inl, &ni,
                    nullptr, nullptr, nullptr));
  for (uint64_t i = 0; i < ni; ++i) inliers->push_back((*correspondences)[inl[i]]);
  mm3d_free(inl);
  return to_matrix(T);
}

Eigen::Matrix4f estimateTransformFromDescriptorsSets(const PointCloudPtr& source_keypoints, const LocalDescriptorsPtr& source_descriptors,
                                                     const PointCloudPtr& target_keypoints, const LocalDescriptorsPtr& target_descriptors,
                                                     double min_sample_distance, double max_correspondence_distance, int max_iterations)
{
  assertDescriptorsPair(source_descriptors, target_descriptors);
  const DescInfo& d = desc_by_name(source_descriptors->fields[0].name);
  std::vector<float> s = pack(source_keypoints.get()), t = pack(target_keypoints.get());
  // the reference draws from the process-global C rand() stream; the shim keeps the running call count per thread
  static thread_local uint64_t rand_calls = 0;
  float T[16];
  check(mm3d_sac_ia(context(), s.data(), s.size() / 4, (const float*)source_descriptors->data.data(), t.data(), t.size() / 4,
                    (const float*)target_descriptors->data.data(), d.dim, min_sample_distance, max_correspondence_distance, max_iterations,
                    &rand_calls, T, nullptr, nullptr));
  return to_matrix(T);
}

Eigen::Matrix4f estimateTransformICP(const PointCloudPtr& source_points, const PointCloudPtr& target_points, const Eigen::Matrix4f& initial_guess,
                                     double max_correspondence_distance, double outlier_rejection_threshold, int max_iterations,
                                     double transformation_epsilon)
{
  std::vector<float> s = pack(source_points.get()), t = pack(target_points.get());
  float T[16];
  check(mm3d_icp(context(), s.data(), s.size() / 4, t.data(), t.size() / 4, initial_guess.data(), max_correspondence_distance,
                 outlier_rejection_threshold, max_iterations, transformation_epsilon, 0.0, T, nullptr, nullptr, nullptr));
  return to_matrix(T);
}

Eigen::Matrix4f estimateTransform(const PointCloudPtr& source_points, const PointCloudPtr& source_keypoints,
                                  const LocalDescriptorsPtr& source_descriptors, const PointCloudPtr& target_points,
                                  const PointCloudPtr& target_keypoints, const LocalDescriptorsPtr& target_descriptors, EstimationMethod method,
                                  bool refine, double inlier_threshold, double max_correspondence_distance, int max_iterations, size_t matching_k,
                                  double transform_epsilon)
{
  Eigen::Matrix4f transform = Eigen::Matrix4f::Zero();
  switch (method) {
    case EstimationMethod::MATCHING: {
      CorrespondencesPtr inliers;
      CorrespondencesPtr correspondences = findFeatureCorrespondences(source_descriptors, target_descriptors, matching_k);
      transform = estimateTransformFromCorrespondences(source_keypoints, target_keypoints, correspondences, inliers, inlier_threshold);
    } break;
    case EstimationMethod::SAC_IA: {
      transform = estimateTransformFromDescriptorsSets(source_keypoints, source_descriptors, target_keypoints, target_descriptors, inlier_threshold,
                                                       max_correspondence_distance, max_iterations);
    } break;
  }
  if (refine)
    transform = estimateTransformICP(source_points, target_points, transform, max_correspondence_distance, inlier_threshold, max_iterations,
                                     transform_epsilon);
  return transform;
}

double transformScore(const PointCloudPtr& source_points, const PointCloudPtr& target_points, const Eigen::Matrix4f& transform, double max_distance)
{
  std::vector<float> s = pack(source_points.get()), t = pack(target_points.get());
  double score = 0.0;
  check(mm3d_score(context(), s.data(), s.size() / 4, t.data(), t.size() / 4, transform.data(), max_distance, 0.0, &score));
  return score;
}

// ---------------------------------------------------------------- map_merging.h
MapMergingParams MapMergingParams::fromCommandLine(int argc, char** argv)
{
  MapMergingParams params;
  auto dbl = [&](const char* flag, double& v) { parse_argument(argc, argv, flag, [&](const char* s) { v = std::atof(s); }); };
  auto integer = [&](const char* flag, int& v) { parse_argument(argc, argv, flag, [&](const char* s) { v = std::atoi(s); }); };
  auto str = [&](const char* flag, std::string& v) { parse_argument(argc, argv, flag, [&](const char* s) { v = s; }); };
  dbl("--resolution", params.resolution);
  dbl("--descriptor_radius", params.descriptor_radius);
  integer("--outliers_min_neighbours", params.outliers_min_neighbours);
  dbl("--normal_radius", params.normal_radius);
  std::string keypoint_type;
  str("--keypoint_type", keypoint_type);
  if (!keypoint_type.empty()) params.keypoint_type = enums::from_string<Keypoint>(keypoint_type);
  dbl("--keypoint_threshold", params.keypoint_threshold);
  std::string descriptor_type;
  str("--descriptor_type", descriptor_type);
  if (!descriptor_type.empty()) params.descriptor_type = enums::from_string<Descriptor>(descriptor_type);
  std::string estimation_method;
  str("--estimation_method", estimation_method);
  if (!estimation_method.empty()) params.estimation_method = enums::from_string<EstimationMethod>(estimation_method);
  int refine = params.refine_transform ? 1 : 0;
  integer("--refine_transform", refine);  // pcl::console::parse_argument(bool&): val = atoi(arg) == 1
  params.refine_transform = refine == 1;
  dbl("--inlier_threshold", params.inlier_threshold);
  dbl("--max_correspondence_distance", params.max_correspondence_distance);
  integer("--max_iterations", params.max_iterations);
  int matching_k = -1;
  integer("--matching_k", matching_k);
  if (matching_k > 0) params.matching_k = size_t(matching_k);
  dbl("--transform_epsilon", params.transform_epsilon);
  dbl("--confidence_threshold", params.confidence_threshold);
  dbl("--output_resolution", params.output_resolution);
  return params;
}

#ifdef MM3D_HAVE_ROS
MapMergingParams MapMergingParams::fromROSNode(const ros::NodeHandle& n)
{
  MapMergingParams params;
  n.getParam("resolution", params.resolution);
  n.getParam("descriptor_radius", params.descriptor_radius);
  n.getParam("outliers_min_neighbours", params.outliers_min_neighbours);
  n.getParam("normal_radius", params.normal_radius);
  std::string s;
  if (n.getParam("keypoint_type", s) && !s.empty()) params.keypoint_type = enums::from_string<Keypoint>(s);
  n.getParam("keypoint_threshold", params.keypoint_threshold);
  if (n.getParam("descriptor_type", s) && !s.empty()) params.descriptor_type = enums::from_string<Descriptor>(s);
  if (n.getParam("estimation_method", s) && !s.empty()) params.estimation_method = enums::from_string<EstimationMethod>(s);
  n.getParam("refine_transform", params.refine_transform);
  n.getParam("inlier_threshold", params.inlier_threshold);
  n.getParam("max_correspondence_distance", params.max_correspondence_distance);
  n.getParam("max_iterations", params.max_iterations);
  int matching_k = -1;
  n.getParam("matching_k", matching_k);
  if (matching_k > 0) params.matching_k = size_t(matching_k);
  n.getParam("transform_epsilon", params.transform_epsilon);
  n.getParam("confidence_threshold", params.confidence_threshold);
  n.getParam("output_resolution", params.output_resolution);
  return params;
}
#endif

std::ostream& operator<<(std::ostream& stream, const MapMergingParams& params)
{
  stream << "resolution: " << params.resolution << std::endl;
  stream << "descriptor_radius: " << params.descriptor_radius << std::endl;
  stream << "outliers_min_neighbours: " << params.outliers_min_neighbours << std::endl;
  stream << "normal_radius: " << params.normal_radius << std::endl;
  stream << "keypoint_type: " << params.keypoint_type << std::endl;
  stream << "keypoint_threshold: " << params.keypoint_threshold << std::endl;
  stream << "descriptor_type: " << params.descriptor_type << std::endl;
  stream << "estimation_method: " << params.estimation_method << std::endl;
  stream << "refine_transform: " << params.refine_transform << std::endl;
  stream << "inlier_threshold: " << params.inlier_threshold << std::endl;
  stream << "max_correspondence_distance: " << params.max_correspondence_distance << std::endl;
  stream << "max_iterations: " << params.max_iterations << std::endl;
  stream << "matching_k: " << params.matching_k << std::endl;
  stream << "transform_epsilon: " << params.transform_epsilon << std::endl;
  stream << "confidence_threshold: " << params.confidence_threshold << std::endl;
  stream << "output_resolution: " << params.output_resolution << std::endl;
  return stream;
}

std::vector<Eigen::Matrix4f> estimateMapsTransforms(const std::vector<PointCloudConstPtr>& clouds, const MapMergingParams& params)
{
  if (clouds.empty()) return {};
  if (clouds.size() == 1) return {Eigen::Matrix4f::Identity()};
  std::vector<const void*> ptrs;
  std::vector<uint64_t> sizes;
  point_arrays(clouds, ptrs, sizes);
  const mm3d_params cp = to_c(params);
  std::vector<float> out(clouds.size() * 16);
  int n_out = 0;
  check(mm3d_estimate_maps_transforms_layout(context(), (int)clouds.size(), ptrs.data(), sizes.data(), &point_layout(), &cp, out.data(), &n_out));
  std::vector<Eigen::Matrix4f> r;
  for (int i = 0; i < n_out; ++i) r.push_back(to_matrix(out.data() + 16 * i));
  return r;
}

PointCloudPtr composeMaps(const std::vector<PointCloudConstPtr>& clouds, const std::vector<Eigen::Matrix4f>& transforms, double resolution)
{
  if (clouds.empty()) return nullptr;
  if (clouds.size() != transforms.size()) throw std::runtime_error("composeMaps: clouds and transforms size must be the same.");
  std::vector<const void*> ptrs;
  std::vector<uint64_t> sizes;
  point_arrays(clouds, ptrs, sizes);
  bool any = false;
  for (uint64_t n : sizes) any = any || n > 0;
  if (!any) return PointCloudPtr(new PointCloud);
  std::vector<float> T(transforms.size() * 16);
  for (size_t i = 0; i < transforms.size(); ++i) std::memcpy(&T[16 * i], transforms[i].data(), 64);
  void* out = nullptr;
  uint64_t n = 0;
  const mm3d_layout& l = point_layout();
  const int rc = mm3d_compose_maps_layout(context(), (int)clouds.size(), ptrs.data(), sizes.data(), &l, (int)transforms.size(), T.data(), resolution,
                                          &l, &out, &n);
  if (rc == 1) return nullptr;
  check(rc);
  // the records are default-constructed points with x, y, z and rgba filled in, which is what unpack() builds
  PointCloudPtr r(new PointCloud);
  r->points.resize(n);
  if (n) std::memcpy((void*)r->points.data(), out, n * sizeof(PointT));
  r->width = (uint32_t)n;
  r->height = 1;
  r->is_dense = true;
  mm3d_free(out);
  return r;
}

}  // namespace map_merge_3d
