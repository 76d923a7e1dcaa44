// pipeline.cuh — the two halves of estimateMapsTransforms (map_merge_3d/src/map_merging.cpp:188-275) as host functions
// over device data, shared by the single-GPU C ABI (api.cu) and the multi-GPU driver (dist.cu).
#pragma once
#include <memory>
#include <vector>

#include "../../include/mm3d.h"
#include "mm3d_internal.cuh"

struct mm3d_team;

struct mm3d_ctx {
  mm3d::Ctx c;
  std::unique_ptr<mm3d_team> team;  // set by mm3d_create_multi: one sub-context + NCCL communicator per device
  mm3d_ctx();
  ~mm3d_ctx();
};

struct mm3d_maps {
  std::vector<mm3d::DCloud> clouds;
};

struct mm3d_shard {
  mm3d::DCloud cloud;  // this rank's transformed points in (map, point) order
};

namespace mm3d {

struct MapFeat {
  DCloud cloud;  // downsampled + outlier-filtered cloud (clouds_resized[i])
  DCloud keypoints;
  DBuf<float> desc;
};

// non-owning view of one map's registration inputs (a MapFeat, or a slice of the buffer the feature exchange filled)
struct FeatView {
  CloudView cloud;
  CloudView keypoints;
  const float* desc;
};

struct PairOut {
  float T[16];  // row-major
  double confidence;
  int n_corr, n_inliers, icp_iterations, icp_converged;
};

// src/map_merging.cpp:212-242, stage-major over all maps; stage_ms (optional, 10 floats) accumulates device time per stage
void compute_features(Ctx& c, const std::vector<CloudView>& raw, const mm3d_params& p, std::vector<MapFeat>& out, float* stage_ms);
// src/map_merging.cpp:256-269 + src/matching.cpp:223-257 for a list of pairs
void register_pairs(Ctx& c, const std::vector<FeatView>& f, int dim, const std::vector<PairJob>& jobs, const mm3d_params& p,
                    std::vector<PairOut>& out, float* stage_ms);
int desc_dim(const mm3d_params& p);
// throws UnsupportedError for an enum value the library does not know
void check_supported(const mm3d_params& p);
std::vector<FeatView> feat_views(const std::vector<MapFeat>& f);
void to_colmajor(const float* rm, float* cm);
void from_colmajor(const float* cm, float* rm);

// layout.cu: records in a caller's layout (include/mm3d.h, mm3d_layout)
extern const mm3d_layout kPackedLayout;  // {16, 0, 4, 8, 12, NULL}
bool layout_valid(const mm3d_layout* l);
bool layout_packed(const mm3d_layout& l);
// host records in layout l -> device clouds (a NULL pointer is an empty cloud); the copies are enqueued on c.stream and
// the caller's buffers are no longer read when the call returns
std::vector<DCloud> upload_clouds(Ctx& c, const std::vector<const void*>& src, const std::vector<uint64_t>& n, const mm3d_layout& l);
DCloud upload_cloud(Ctx& c, const float* pts, uint64_t n);  // one cloud in the packed layout
// n device points -> n records in layout l in a host_out_alloc block; the copy is enqueued on c.stream (the caller synchronises)
void* download_records(Ctx& c, const float4* pts, size_t n, const mm3d_layout& l);
void staging_release(Ctx& c);

// dist.cu: one rank's part of composeMaps on device clouds (cm = NULL: a single rank); *out = records in out_layout
// (host_out_alloc)
void dist_compose(Ctx& c, mm3d_comm* cm, const std::vector<CloudView>& local, const std::vector<const float*>& transforms_rowmajor,
                  double resolution, const mm3d_layout& out_layout, void** out, uint64_t* n_out);
// composeMaps' skip rule (map_merging.cpp:293-295): true for a zero transform or an empty cloud; rowmajor = the transform
bool skip_map(const float* colmajor, const void* cloud, uint64_t n, float* rowmajor);
// dist.cu: the high-level calls over the devices of a mm3d_create_multi context (one host thread per device)
int team_size(const mm3d_ctx* ctx);
int team_estimate(mm3d_ctx* master, int n_maps, const void* const* clouds, const uint64_t* n_points, const mm3d_layout& layout,
                  const mm3d_params& p, float* out_transforms);
void team_compose(mm3d_ctx* master, int n_maps, const void* const* clouds, const uint64_t* n_points, const mm3d_layout& in_layout,
                  const float* transforms, double resolution, const mm3d_layout& out_layout, void** out, uint64_t* n_out);

}  // namespace mm3d

// Body of a C ABI entry point: errors thrown by the pipeline become status codes and the context's last error.
#define MM_TRY(ctx) \
  if (!(ctx)) return MM3D_ERR_ARG; \
  Ctx& c = (ctx)->c; \
  try { \
    MM_CUDA(cudaSetDevice(c.device));
#define MM_CATCH \
  } catch (const UnsupportedError& e) { \
    c.err = e.what(); \
    return MM3D_ERR_UNSUPPORTED; \
  } catch (const CudaError& e) { \
    c.err = e.what(); \
    cudaGetLastError(); \
    return MM3D_ERR_CUDA; \
  } catch (const std::exception& e) { \
    c.err = e.what(); \
    cudaGetLastError(); \
    return MM3D_ERR; \
  } \
  return MM3D_OK;

struct mm3d_features {
  std::vector<mm3d::MapFeat> maps;
  int dim = 33;
};
