// api.cu — the C ABI (include/mm3d.h) and the orchestration of the hot path:
// stage-major per-map loops and the all-pairs loop of
// map_merge_3d/src/map_merging.cpp:188-275, each stage one batched launch set.
#include <chrono>
#include <cmath>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <memory>

#include <nvtx3/nvToolsExt.h>

#include "../../include/mm3d.h"
#include "mm3d_internal.cuh"
#include "pipeline.cuh"

using namespace mm3d;

namespace {

const char* kStageNames[10] = {"downsampling", "removing outliers", "normals computation", "keypoints detection", "descriptors computation",
                               "finding correspondences", "initial alignment", "ICP alignment", "scoring", "graph"};

struct StageTimer {
  Ctx& c;
  float* ms;
  cudaEvent_t ev[2];
  bool host_trace;  // MM3D_HOST_TRACE=1: host wall-clock per stage on stderr, no extra synchronisation (where does the host wait?)
  bool nvtx;        // MM3D_NVTX=1: one NVTX range per stage (registration_visualisation.cpp:51-158 uses pcl::ScopeTime for the same blocks)
  std::chrono::steady_clock::time_point h0;
  explicit StageTimer(Ctx& ctx, float* out) : c(ctx), ms(out)
  {
    const char* e = std::getenv("MM3D_HOST_TRACE");
    host_trace = e && e[0] == '1';
    const char* n = std::getenv("MM3D_NVTX");
    nvtx = n && n[0] == '1';
    if (ms) {
      cudaEventCreate(&ev[0]);
      cudaEventCreate(&ev[1]);
    }
  }
  ~StageTimer()
  {
    if (ms) {
      cudaEventDestroy(ev[0]);
      cudaEventDestroy(ev[1]);
    }
  }
  void begin(int stage)
  {
    if (nvtx) nvtxRangePushA(kStageNames[stage]);  // the reference's eight pcl::ScopeTime labels (+ scoring, graph) as NVTX ranges
    if (host_trace) h0 = std::chrono::steady_clock::now();
    if (ms) cudaEventRecord(ev[0], c.stream);
  }
  void end(int stage)
  {
    if (nvtx) nvtxRangePop();
    if (host_trace)
      fprintf(stderr, "[mm3d host] %-26s %8.2f ms\n", kStageNames[stage],
              std::chrono::duration<double, std::milli>(std::chrono::steady_clock::now() - h0).count());
    if (!ms) return;
    cudaEventRecord(ev[1], c.stream);
    cudaEventSynchronize(ev[1]);
    float t = 0.f;
    cudaEventElapsedTime(&t, ev[0], ev[1]);
    ms[stage] += t;
  }
};

template <typename T>
T* host_copy(Ctx& c, const T* dev, size_t count)
{
  T* h = (T*)host_out_alloc(std::max<size_t>(count, 1) * sizeof(T));
  if (count) MM_CUDA(cudaMemcpyAsync(h, dev, count * sizeof(T), cudaMemcpyDeviceToHost, c.stream));
  return h;
}

double auto_leaf(double index_leaf, double radius, double ratio)
{
  if (index_leaf > 0.0) return index_leaf;
  return radius / ratio;
}

void check_supported(const mm3d_params& p)
{
  if (p.keypoint_type != MM3D_KP_SIFT && p.keypoint_type != MM3D_KP_HARRIS) throw UnsupportedError("unsupported: unknown keypoint_type");
  if (p.descriptor_type < MM3D_DESC_PFH || p.descriptor_type > MM3D_DESC_SC3D) throw UnsupportedError("unsupported: unknown descriptor_type");
  if (p.estimation_method != MM3D_EST_MATCHING && p.estimation_method != MM3D_EST_SAC_IA) throw UnsupportedError("unsupported: unknown estimation_method");
}

}  // namespace

namespace mm3d {

namespace {
struct PinnedPool {
  std::mutex mu;
  std::unordered_map<void*, size_t> live;                     // pinned blocks handed out: pointer -> size class
  std::unordered_map<size_t, std::vector<void*>> free_blocks;  // size class -> cached blocks
  size_t cached = 0;
};
PinnedPool& pinned_pool()
{
  static PinnedPool* p = new PinnedPool();  // never destroyed: blocks may be released after the CUDA runtime has shut down
  return *p;
}
constexpr size_t PINNED_MIN = (size_t)1 << 20, PINNED_CACHE_MAX = (size_t)2 << 30;
}  // namespace

void* host_out_alloc(size_t bytes)
{
  if (bytes < PINNED_MIN) return malloc(std::max<size_t>(bytes, 1));
  const size_t cls = BlockCache::size_class(bytes);
  PinnedPool& pp = pinned_pool();
  {
    std::lock_guard<std::mutex> lk(pp.mu);
    auto it = pp.free_blocks.find(cls);
    if (it != pp.free_blocks.end() && !it->second.empty()) {
      void* p = it->second.back();
      it->second.pop_back();
      pp.cached -= cls;
      pp.live[p] = cls;
      return p;
    }
  }
  void* p = nullptr;
  if (cudaHostAlloc(&p, cls, cudaHostAllocPortable) != cudaSuccess) {
    cudaGetLastError();
    return malloc(bytes);
  }
  std::lock_guard<std::mutex> lk(pp.mu);
  pp.live[p] = cls;
  return p;
}

void host_out_free(void* p)
{
  if (!p) return;
  PinnedPool& pp = pinned_pool();
  size_t cls = 0;
  bool keep = false;
  {
    std::lock_guard<std::mutex> lk(pp.mu);
    auto it = pp.live.find(p);
    if (it != pp.live.end()) {
      cls = it->second;
      pp.live.erase(it);
      if (pp.cached + cls <= PINNED_CACHE_MAX) {
        pp.free_blocks[cls].push_back(p);
        pp.cached += cls;
        keep = true;
      }
    }
  }
  if (cls == 0) free(p);
  else if (!keep) cudaFreeHost(p);
}

HostProf& host_prof()
{
  static HostProf hp;
  static bool init = false;
  if (!init) {
    const char* e = std::getenv("MM3D_HOST_TRACE");
    hp.on = e && e[0] == '1';
    init = true;
  }
  return hp;
}
double host_now_ms() { return std::chrono::duration<double, std::milli>(std::chrono::steady_clock::now().time_since_epoch()).count(); }

void to_colmajor(const float* rm, float* cm)
{
  for (int r = 0; r < 4; ++r)
    for (int c = 0; c < 4; ++c) cm[c * 4 + r] = rm[r * 4 + c];
}
void from_colmajor(const float* cm, float* rm)
{
  for (int r = 0; r < 4; ++r)
    for (int c = 0; c < 4; ++c) rm[r * 4 + c] = cm[c * 4 + r];
}

// src/map_merging.cpp:212-242, stage-major over all maps
void compute_features(Ctx& c, const std::vector<CloudView>& raw, const mm3d_params& p, std::vector<MapFeat>& out, float* stage_ms)
{
  check_supported(p);
  const int M = (int)raw.size();
  out.clear();
  out.resize(M);
  StageTimer tm(c, stage_ms);
  const float leaf = (float)p.resolution;

  tm.begin(0);
  std::vector<DCloud> resized;
  std::vector<VoxGeom> vgeom;
  voxel_downsample_batch(c, raw, leaf, resized, &vgeom);
  tm.end(0);

  tm.begin(1);
  std::vector<CloudView> rv(M);
  for (int m = 0; m < M; ++m) rv[m] = resized[m].view();
  std::vector<DCloud> filtered;
  {
    std::vector<DIndex> idx;
    build_index_batch(c, rv, leaf, 2, 0, 0, idx, nullptr, &vgeom);
    remove_outliers_batch(c, rv, idx, p.descriptor_radius, p.outliers_min_neighbours, filtered, nullptr);
  }
  tm.end(1);

  tm.begin(2);
  std::vector<CloudView> fv(M);
  for (int m = 0; m < M; ++m) fv[m] = filtered[m].view();
  std::vector<DIndex> idx;
  build_index_batch(c, fv, leaf, 2, 0, 0, idx, nullptr, &vgeom);
  std::vector<DBuf<float4>> normals;
  normals_batch(c, fv, idx, p.normal_radius, normals);
  tm.end(2);

  tm.begin(3);
  std::vector<DCloud> kps;
  std::vector<const float4*> np(M);
  for (int m = 0; m < M; ++m) np[m] = normals[m].p;
  if (p.keypoint_type == MM3D_KP_HARRIS)  // detectKeypoints(..., threshold, normal_radius, resolution)  (map_merging.cpp:230-235)
    harris_batch(c, fv, idx, np, (float)p.keypoint_threshold, (float)p.normal_radius, kps, nullptr, nullptr);
  else
    sift_batch(c, fv, (float)p.resolution, 3, 3, (float)p.keypoint_threshold, kps, nullptr);
  tm.end(3);

  tm.begin(4);
  std::vector<DBuf<float>> desc;
  if (p.descriptor_type == MM3D_DESC_SHOT) shot_batch(c, fv, idx, np, kps, p.descriptor_radius, desc, nullptr);
  else if (p.descriptor_type == MM3D_DESC_PFH) pfh_batch(c, fv, idx, np, kps, p.descriptor_radius, desc, false);
  else if (p.descriptor_type == MM3D_DESC_PFHRGB) pfh_batch(c, fv, idx, np, kps, p.descriptor_radius, desc, true);
  else if (p.descriptor_type == MM3D_DESC_RSD) rsd_batch(c, fv, idx, np, kps, p.descriptor_radius, desc);
  else if (p.descriptor_type == MM3D_DESC_SC3D) sc3d_batch(c, fv, idx, np, kps, p.descriptor_radius, desc);
  else fpfh_batch(c, fv, idx, np, kps, p.descriptor_radius, desc, nullptr);
  tm.end(4);

  for (int m = 0; m < M; ++m) {
    out[m].cloud = std::move(filtered[m]);
    out[m].keypoints = std::move(kps[m]);
    out[m].desc = std::move(desc[m]);
  }
  c.sync();
}

// src/map_merging.cpp:256-269 + src/matching.cpp:223-257 for a list of pairs
void register_pairs(Ctx& c, const std::vector<FeatView>& f, int dim, const std::vector<PairJob>& jobs, const mm3d_params& p,
                    std::vector<PairOut>& out, float* stage_ms)
{
  check_supported(p);
  const int P = (int)jobs.size();
  out.assign(P, PairOut());
  if (P == 0) return;
  const int M = (int)f.size();
  StageTimer tm(c, stage_ms);
  std::vector<CloudView> clouds(M), kps(M);
  std::vector<const float*> desc(M);
  std::vector<int> nk(M);
  for (int m = 0; m < M; ++m) {
    clouds[m] = f[m].cloud;
    kps[m] = f[m].keypoints;
    desc[m] = f[m].desc;
    nk[m] = f[m].keypoints.n;
  }
  std::vector<DCorr> corr(P);
  std::vector<RansacOut> rs(P);
  if (p.estimation_method == MM3D_EST_SAC_IA) {
    // estimateTransformFromDescriptorsSets(min_sample_distance = inlier_threshold, max_correspondence_distance, max_iterations)
    // (matching.cpp:242-247).  The C rand() stream runs through the complete row-major pair list of the feature set.
    tm.begin(6);
    std::vector<PairJob> all_pairs;
    for (int i = 0; i < M - 1; ++i)
      for (int j2 = i + 1; j2 < M; ++j2)
        if (nk[i] > 0 && nk[j2] > 0) all_pairs.push_back(PairJob{i, j2});
    std::vector<int> wanted(P, -1);
    for (int k = 0; k < P; ++k)
      for (size_t a = 0; a < all_pairs.size(); ++a)
        if (all_pairs[a].a == jobs[k].a && all_pairs[a].b == jobs[k].b) wanted[k] = (int)a;
    for (int k = 0; k < P; ++k)
      if (wanted[k] < 0) throw std::runtime_error("register_pairs(SAC_IA): pair is not in the row-major pair list (i < j, both with keypoints)");
    std::vector<SacOut> so;
    sac_ia_batch(c, kps, desc, dim, all_pairs, wanted, p.inlier_threshold, p.max_correspondence_distance, p.max_iterations, 0, so);
    for (int k = 0; k < P; ++k) {
      memset(&rs[k], 0, sizeof(RansacOut));
      memcpy(rs[k].T, so[k].T, sizeof(float) * 16);
    }
    tm.end(6);
  } else {
    tm.begin(5);
    match_batch(c, desc, nk, dim, jobs, (size_t)p.matching_k, corr);
    tm.end(5);

    tm.begin(6);
    ransac_batch(c, kps, jobs, corr, p.inlier_threshold, rs, nullptr);
    tm.end(6);
  }

  // neighbour index over every map that is a target of some pair
  std::vector<CloudView> tv(M, CloudView{nullptr, 0});
  for (const PairJob& j : jobs) tv[j.b] = clouds[j.b];
  std::vector<DIndex> tidx;
  tm.begin(7);
  // One-voxel cells: the clouds are voxel-grid outputs (at most one point per voxel), so the nearest neighbour of a query
  // that lies on the target surface is found in the 3 x 3 x 3 voxel block around it — nine (z, y) rows whose three cells are
  // one contiguous run each (icp.cu, nearest_block27).  The general row search remains the fallback for queries farther
  // than one voxel from the target.  (Round 1 measured the general search alone: 4 x 2 x 2-voxel cells were its best
  // setting because it is bound by its per-row bookkeeping; the block search has none.)
  build_index_batch(c, tv, (float)p.resolution, 0, 0, 0, tidx);
  // reach grids of the targets (icp.cu): queries without a target point in range are answered without a search
  std::vector<DReach> reach;
  {
    const double r_icp = p.max_correspondence_distance, r_score = std::sqrt(std::max(p.max_correspondence_distance, 0.0));
    build_reach_batch(c, tidx, (int)std::ceil(std::max(r_icp, r_score) / p.resolution) + 1, reach);
  }
  std::vector<const float*> t0(P);
  for (int i = 0; i < P; ++i) t0[i] = rs[i].T;
  std::vector<IcpOut> icp(P);
  IcpNeighbours icp_nn;
  if (p.refine_transform) {
    icp_batch(c, clouds, tidx, reach, jobs, t0, p.max_correspondence_distance, p.max_iterations, p.transform_epsilon, icp, nullptr, &icp_nn);
  } else {
    for (int i = 0; i < P; ++i) {
      memcpy(icp[i].T, rs[i].T, sizeof(float) * 16);
      icp[i].iterations = 0;
      icp[i].converged = 0;
    }
  }
  tm.end(7);

  tm.begin(8);
  std::vector<const float*> tf(P);
  for (int i = 0; i < P; ++i) tf[i] = icp[i].T;
  std::vector<double> scores;
  score_batch(c, clouds, tidx, reach, jobs, tf, p.max_correspondence_distance, scores, p.refine_transform ? &icp_nn : nullptr);
  tm.end(8);

  for (int i = 0; i < P; ++i) {
    memcpy(out[i].T, icp[i].T, sizeof(float) * 16);
    out[i].confidence = 1. / scores[i];
    out[i].n_corr = corr[i].n;
    out[i].n_inliers = rs[i].n_inliers;
    out[i].icp_iterations = icp[i].iterations;
    out[i].icp_converged = icp[i].converged;
  }
  c.sync();
}

int desc_dim(const mm3d_params& p)
{
  switch (p.descriptor_type) {
    case MM3D_DESC_SHOT: return 1344;
    case MM3D_DESC_PFH: return 125;
    case MM3D_DESC_PFHRGB: return 250;
    case MM3D_DESC_RSD: return 2;
    case MM3D_DESC_SC3D: return 1980;
    default: return 33;
  }
}

std::vector<FeatView> feat_views(const std::vector<MapFeat>& f)
{
  std::vector<FeatView> v(f.size());
  for (size_t m = 0; m < f.size(); ++m) v[m] = FeatView{f[m].cloud.view(), f[m].keypoints.view(), f[m].desc.p};
  return v;
}

}  // namespace mm3d

namespace {

// returns number of transforms written
int estimate_from_views(Ctx& c, const std::vector<CloudView>& raw, const mm3d_params& p, float* out_transforms, float* stage_ms)
{
  const int M = (int)raw.size();
  if (M == 0) return 0;
  if (M == 1) {
    const float id[16] = {1, 0, 0, 0, 0, 1, 0, 0, 0, 0, 1, 0, 0, 0, 0, 1};
    memcpy(out_transforms, id, sizeof(id));
    return 1;
  }
  std::vector<MapFeat> f;
  compute_features(c, raw, p, f, stage_ms);
  std::vector<PairJob> jobs;
  for (int i = 0; i < M - 1; ++i)
    for (int j = i + 1; j < M; ++j)
      if (f[i].keypoints.n > 0 && f[j].keypoints.n > 0) jobs.push_back(PairJob{i, j});
  std::vector<PairOut> po;
  register_pairs(c, feat_views(f), desc_dim(p), jobs, p, po, stage_ms);
  std::vector<HostEstimate> est(jobs.size());
  for (size_t k = 0; k < jobs.size(); ++k) {
    est[k].source_idx = (size_t)jobs[k].a;
    est[k].target_idx = (size_t)jobs[k].b;
    memcpy(est[k].T, po[k].T, sizeof(float) * 16);
    est[k].confidence = po[k].confidence;
  }
  std::vector<std::vector<float>> g = compute_global_transforms(est, p.confidence_threshold, nullptr, nullptr, nullptr, nullptr);
  for (size_t i = 0; i < g.size(); ++i) to_colmajor(g[i].data(), out_transforms + 16 * i);
  HostProf& hp = host_prof();
  if (hp.on) {
    fprintf(stderr, "[mm3d host] buffer allocations %ld calls %.2f ms (%.1f MB), cudaFreeAsync %ld calls %.2f ms, sync %ld calls %.2f ms, "
            "small copies %ld calls %.2f ms; block cache holds %.1f MB\n", hp.n_alloc, hp.alloc_ms, hp.alloc_bytes / 1e6, hp.n_free, hp.free_ms,
            hp.n_sync, hp.sync_ms, hp.n_copy, hp.copy_ms, c.cache->held_bytes / 1e6);
    const bool on = hp.on;
    hp = HostProf();
    hp.on = on;
  }
  return (int)g.size();
}

int bad_layout(mm3d_ctx* ctx)
{
  if (ctx) ctx->c.err = "malformed mm3d_layout (include/mm3d.h)";
  return MM3D_ERR_ARG;
}

}  // namespace

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

extern "C" {

void mm3d_params_default(mm3d_params* p)
{
  p->resolution = 0.1;
  p->descriptor_radius = p->resolution * 8.0;
  p->outliers_min_neighbours = 50;
  p->normal_radius = p->resolution * 6.0;
  p->keypoint_type = MM3D_KP_SIFT;
  p->keypoint_threshold = 5.0;
  p->descriptor_type = MM3D_DESC_PFH;
  p->estimation_method = MM3D_EST_MATCHING;
  p->refine_transform = 1;
  p->inlier_threshold = p->resolution * 5.0;
  p->max_correspondence_distance = p->inlier_threshold * 2.0;
  p->max_iterations = 500;
  p->matching_k = 5;
  p->transform_epsilon = 1e-2;
  p->confidence_threshold = 0.0;
  p->output_resolution = 0.05;
}

int mm3d_create(mm3d_ctx** ctx, int device, void* cuda_stream)
{
  if (!ctx) return MM3D_ERR_ARG;
  *ctx = nullptr;
  int count = 0;
  if (cudaGetDeviceCount(&count) != cudaSuccess || device < 0 || device >= count) {
    cudaGetLastError();
    return MM3D_ERR_CUDA;  // no CPU fallback: without a device the library refuses to run
  }
  std::unique_ptr<mm3d_ctx> h(new mm3d_ctx);
  h->c.device = device;
  if (cudaSetDevice(device) != cudaSuccess) return MM3D_ERR_CUDA;
  if (cuda_stream) {
    h->c.stream = (cudaStream_t)cuda_stream;
    h->c.own_stream = false;
  } else {
    if (cudaStreamCreateWithFlags(&h->c.stream, cudaStreamNonBlocking) != cudaSuccess) return MM3D_ERR_CUDA;
    h->c.own_stream = true;
  }
  h->c.cache->device = device;
  h->c.cache->stream = h->c.stream;
  // keep freed blocks in the pool: the path allocates and frees per stage
  cudaMemPool_t pool;
  if (cudaDeviceGetDefaultMemPool(&pool, device) == cudaSuccess) {
    uint64_t thr = UINT64_MAX;
    cudaMemPoolSetAttribute(pool, cudaMemPoolAttrReleaseThreshold, &thr);
  }
  *ctx = h.release();
  return MM3D_OK;
}

void mm3d_destroy(mm3d_ctx* ctx)
{
  if (!ctx) return;
  cudaSetDevice(ctx->c.device);
  cudaStreamSynchronize(ctx->c.stream);
  ctx->c.cache->trim();        // cached blocks go back while the stream still exists
  ctx->c.cache->stream = nullptr;  // blocks returned by buffers that outlive the context are freed with the last reference
  if (ctx->c.knn_stats) cudaFree(ctx->c.knn_stats);
  staging_release(ctx->c);
  for (cudaEvent_t e : ctx->c.event_pool) cudaEventDestroy(e);
  for (KernelSample& s : ctx->c.samples) { cudaEventDestroy(s.e0); cudaEventDestroy(s.e1); }
  if (ctx->c.own_stream) cudaStreamDestroy(ctx->c.stream);
  delete ctx;
}

const char* mm3d_last_error(mm3d_ctx* ctx) { return ctx ? ctx->c.err.c_str() : "null context"; }
void mm3d_free(void* p) { mm3d::host_out_free(p); }
long long mm3d_kernel_launches(mm3d_ctx* ctx) { return ctx ? ctx->c.launches : 0; }

int mm3d_estimate_maps_transforms(mm3d_ctx* ctx, int n_maps, const float* const* clouds, const uint64_t* n_points, const mm3d_params* params,
                                  float* out_transforms, int* n_out)
{
  return mm3d_estimate_maps_transforms_layout(ctx, n_maps, (const void* const*)clouds, n_points, &kPackedLayout, params, out_transforms, n_out);
}

int mm3d_estimate_maps_transforms_layout(mm3d_ctx* ctx, int n_maps, const void* const* clouds, const uint64_t* n_points,
                                         const mm3d_layout* layout, const mm3d_params* params, float* out_transforms, int* n_out)
{
  if (!n_out) return MM3D_ERR_ARG;
  *n_out = 0;
  if (!layout_valid(layout)) return bad_layout(ctx);
  // the degenerate cases never touch the device (map_merging.cpp:192-197)
  if (n_maps == 0) return MM3D_OK;
  if (n_maps == 1) {
    const float id[16] = {1, 0, 0, 0, 0, 1, 0, 0, 0, 0, 1, 0, 0, 0, 0, 1};
    memcpy(out_transforms, id, sizeof(id));
    *n_out = 1;
    return MM3D_OK;
  }
  MM_TRY(ctx)
  if (ctx->team) {  // mm3d_create_multi: maps and pairs sharded over the context's devices (dist.cu)
    *n_out = team_estimate(ctx, n_maps, clouds, n_points, *layout, *params, out_transforms);
    return MM3D_OK;
  }
  std::vector<DCloud> d = upload_clouds(c, std::vector<const void*>(clouds, clouds + n_maps), std::vector<uint64_t>(n_points, n_points + n_maps), *layout);
  std::vector<CloudView> v(n_maps);
  for (int m = 0; m < n_maps; ++m) v[m] = d[m].view();
  *n_out = estimate_from_views(c, v, *params, out_transforms, nullptr);
  c.sync();
  MM_CATCH
}

int mm3d_compose_maps(mm3d_ctx* ctx, int n_maps, const float* const* clouds, const uint64_t* n_points, int n_transforms,
                      const float* transforms, double resolution, float** out, uint64_t* n_out)
{
  return mm3d_compose_maps_layout(ctx, n_maps, (const void* const*)clouds, n_points, &kPackedLayout, n_transforms, transforms, resolution,
                                  &kPackedLayout, (void**)out, n_out);
}

int mm3d_compose_maps_layout(mm3d_ctx* ctx, int n_maps, const void* const* clouds, const uint64_t* n_points, const mm3d_layout* in_layout,
                             int n_transforms, const float* transforms, double resolution, const mm3d_layout* out_layout, void** out,
                             uint64_t* n_out)
{
  if (!out || !n_out) return MM3D_ERR_ARG;
  *out = nullptr;
  *n_out = 0;
  if (!layout_valid(in_layout) || !layout_valid(out_layout)) return bad_layout(ctx);
  if (n_maps == 0) return 1;  // nullptr result
  if (n_maps != n_transforms) {
    if (ctx) ctx->c.err = "composeMaps: clouds and transforms size must be the same.";
    return MM3D_ERR_ARG;
  }
  // all-empty input needs no device either (test_map_merging.cpp:34-40, leaf size 0.0)
  bool any = false;
  for (int m = 0; m < n_maps; ++m)
    if (clouds[m] && n_points[m] > 0) any = true;
  if (!any) {
    *out = malloc(16);
    return MM3D_OK;
  }
  MM_TRY(ctx)
  if (ctx->team) {
    team_compose(ctx, n_maps, clouds, n_points, *in_layout, transforms, resolution, *out_layout, out, n_out);
    return MM3D_OK;
  }
  std::vector<const void*> src;
  std::vector<uint64_t> cnt;
  std::vector<std::vector<float>> tr;
  for (int m = 0; m < n_maps; ++m) {
    float rm[16];
    from_colmajor(transforms + 16 * m, rm);
    bool zero = true;  // Eigen isZero(): every |a_ij| <= 1e-5
    for (int k = 0; k < 16; ++k)
      if (!(std::fabs(rm[k]) <= 1e-5f)) zero = false;
    if (zero || !clouds[m] || n_points[m] == 0) continue;
    src.push_back(clouds[m]);
    cnt.push_back(n_points[m]);
    tr.emplace_back(rm, rm + 16);
  }
  std::vector<DCloud> d = upload_clouds(c, src, cnt, *in_layout);
  std::vector<CloudView> v;
  std::vector<const float*> tp;
  for (size_t i = 0; i < d.size(); ++i) {
    v.push_back(d[i].view());
    tp.push_back(tr[i].data());
  }
  DCloud cat;
  transform_concat(c, v, tp, cat);
  std::vector<DCloud> res;
  voxel_downsample_batch(c, {cat.view()}, (float)resolution, res, nullptr);
  *out = download_records(c, res[0].pts.p, (size_t)res[0].n, *out_layout);
  *n_out = (uint64_t)res[0].n;
  c.sync();
  MM_CATCH
}

int mm3d_downsample(mm3d_ctx* ctx, const float* pts, uint64_t n, double resolution, float** out, uint64_t* n_out)
{
  if (!out || !n_out) return MM3D_ERR_ARG;
  MM_TRY(ctx)
  DCloud d = upload_cloud(c, pts, n);
  std::vector<DCloud> res;
  voxel_downsample_batch(c, {d.view()}, (float)resolution, res, nullptr);
  *out = (float*)host_copy(c, res[0].pts.p, (size_t)res[0].n);
  *n_out = (uint64_t)res[0].n;
  c.sync();
  MM_CATCH
}

int mm3d_remove_outliers(mm3d_ctx* ctx, const float* pts, uint64_t n, double radius, int min_neighbours, double index_leaf, float** out,
                         uint64_t* n_out, int32_t* counts)
{
  if (!out || !n_out) return MM3D_ERR_ARG;
  MM_TRY(ctx)
  DCloud d = upload_cloud(c, pts, n);
  std::vector<DIndex> idx;
  build_index_batch(c, {d.view()}, (float)auto_leaf(index_leaf, radius, 8.0), 2, 0, 0, idx);
  std::vector<DCloud> res;
  std::vector<DBuf<int>> cnt;
  remove_outliers_batch(c, {d.view()}, idx, radius, min_neighbours, res, counts ? &cnt : nullptr);
  *out = (float*)host_copy(c, res[0].pts.p, (size_t)res[0].n);
  *n_out = (uint64_t)res[0].n;
  if (counts && d.n) cnt[0].download(c, counts, d.n);
  c.sync();
  MM_CATCH
}

int mm3d_normals(mm3d_ctx* ctx, const float* pts, uint64_t n, double radius, double index_leaf, float** normals)
{
  if (!normals) return MM3D_ERR_ARG;
  MM_TRY(ctx)
  DCloud d = upload_cloud(c, pts, n);
  std::vector<DIndex> idx;
  build_index_batch(c, {d.view()}, (float)auto_leaf(index_leaf, radius, 6.0), 2, 0, 0, idx);
  std::vector<DBuf<float4>> nm;
  normals_batch(c, {d.view()}, idx, radius, nm);
  *normals = (float*)host_copy(c, nm[0].p, (size_t)d.n);
  c.sync();
  MM_CATCH
}

int mm3d_keypoints(mm3d_ctx* ctx, const float* pts, uint64_t n, const float* normals, int type, double threshold, double radius,
                   double resolution, float** keypoints, uint64_t* n_keypoints, float** dog0, uint64_t* n_dog0)
{
  if (!keypoints || !n_keypoints) return MM3D_ERR_ARG;
  MM_TRY(ctx)
  if (type != MM3D_KP_SIFT && type != MM3D_KP_HARRIS) throw UnsupportedError("unsupported: unknown keypoint_type");
  DCloud d = upload_cloud(c, pts, n);
  std::vector<DCloud> kp;
  std::vector<DBuf<float>> dog;
  if (type == MM3D_KP_HARRIS) {
    // detectKeypointsHarris(points, normals, threshold, radius)  (features.cpp:94); dog0 receives the Harris response
    if (!normals) throw std::runtime_error("detectKeypoints(HARRIS) needs normals");
    DBuf<float4> nm(c, d.n);
    if (d.n) MM_CUDA(cudaMemcpyAsync(nm.p, normals, (size_t)d.n * sizeof(float4), cudaMemcpyHostToDevice, c.stream));
    std::vector<DIndex> idx;
    build_index_batch(c, {d.view()}, (float)resolution, 2, 0, 0, idx);
    harris_batch(c, {d.view()}, idx, {nm.p}, (float)threshold, (float)radius, kp, dog0 ? &dog : nullptr, nullptr);
    *keypoints = (float*)host_copy(c, kp[0].pts.p, (size_t)kp[0].n);
    *n_keypoints = (uint64_t)kp[0].n;
    if (dog0) {
      *dog0 = host_copy(c, dog[0].p, dog[0].n);
      *n_dog0 = dog[0].n;
    }
    c.sync();
    return MM3D_OK;
  }
  // detectKeypointsSIFT(points, resolution, 3, 3, threshold)  (features.cpp:92)
  sift_batch(c, {d.view()}, (float)resolution, 3, 3, (float)threshold, kp, dog0 ? &dog : nullptr);
  *keypoints = (float*)host_copy(c, kp[0].pts.p, (size_t)kp[0].n);
  *n_keypoints = (uint64_t)kp[0].n;
  if (dog0) {
    *dog0 = host_copy(c, dog[0].p, dog[0].n);
    *n_dog0 = dog[0].n;
  }
  c.sync();
  MM_CATCH
}

int mm3d_descriptors(mm3d_ctx* ctx, const float* pts, uint64_t n, const float* normals, const float* keypoints, uint64_t n_keypoints,
                     int type, double radius, double index_leaf, float** keypoints_out, uint64_t* n_out, float** descriptors, int* dim,
                     float** spfh)
{
  if (!keypoints_out || !n_out || !descriptors) return MM3D_ERR_ARG;
  MM_TRY(ctx)
  if (type < MM3D_DESC_PFH || type > MM3D_DESC_SC3D) throw UnsupportedError("unsupported: unknown descriptor_type");
  DCloud d = upload_cloud(c, pts, n);
  DBuf<float4> nm(c, d.n);
  if (d.n) MM_CUDA(cudaMemcpyAsync(nm.p, normals, (size_t)d.n * sizeof(float4), cudaMemcpyHostToDevice, c.stream));
  std::vector<DCloud> kp(1);
  kp[0] = upload_cloud(c, keypoints, n_keypoints);
  std::vector<DIndex> idx;
  build_index_batch(c, {d.view()}, (float)auto_leaf(index_leaf, radius, 8.0), 2, 0, 0, idx);
  std::vector<DBuf<float>> desc, sp;
  const int D = type == MM3D_DESC_SHOT ? 1344 : (type == MM3D_DESC_PFH ? 125 : (type == MM3D_DESC_PFHRGB ? 250 : (type == MM3D_DESC_RSD ? 2 : (type == MM3D_DESC_SC3D ? 1980 : 33))));
  if (type == MM3D_DESC_RSD || type == MM3D_DESC_SC3D) {
    if (type == MM3D_DESC_RSD) rsd_batch(c, {d.view()}, idx, {nm.p}, kp, radius, desc);
    else sc3d_batch(c, {d.view()}, idx, {nm.p}, kp, radius, desc);
    if (spfh) { sp.resize(1); }
  } else if (type == MM3D_DESC_PFH || type == MM3D_DESC_PFHRGB) {
    pfh_batch(c, {d.view()}, idx, {nm.p}, kp, radius, desc, type == MM3D_DESC_PFHRGB);
    if (spfh) { sp.resize(1); }
  } else if (type == MM3D_DESC_SHOT) shot_batch(c, {d.view()}, idx, {nm.p}, kp, radius, desc, spfh ? &sp : nullptr);  // spfh <- reference frames (K' x 9)
  else fpfh_batch(c, {d.view()}, idx, {nm.p}, kp, radius, desc, spfh ? &sp : nullptr);
  *keypoints_out = (float*)host_copy(c, kp[0].pts.p, (size_t)kp[0].n);
  *n_out = (uint64_t)kp[0].n;
  *descriptors = host_copy(c, desc[0].p, (size_t)kp[0].n * D);
  if (dim) *dim = D;
  if (spfh) *spfh = host_copy(c, sp[0].p, sp[0].n);
  c.sync();
  MM_CATCH
}

int mm3d_match(mm3d_ctx* ctx, const float* desc_src, uint64_t n_src, const float* desc_tgt, uint64_t n_tgt, int dim, uint64_t k,
               int32_t** pairs, float** distances, uint64_t* n_corr)
{
  if (!pairs || !distances || !n_corr) return MM3D_ERR_ARG;
  MM_TRY(ctx)
  DBuf<float> a(c, n_src * dim), b(c, n_tgt * dim);
  a.upload(c, desc_src, n_src * dim);
  b.upload(c, desc_tgt, n_tgt * dim);
  std::vector<DCorr> corr;
  match_batch(c, {a.p, b.p}, {(int)n_src, (int)n_tgt}, dim, {PairJob{0, 1}}, (size_t)k, corr);
  *pairs = (int32_t*)host_copy(c, corr[0].pairs.p, (size_t)corr[0].n);
  *distances = host_copy(c, corr[0].dist.p, (size_t)corr[0].n);
  *n_corr = (uint64_t)corr[0].n;
  c.sync();
  MM_CATCH
}

int mm3d_knn(mm3d_ctx* ctx, const float* a, uint64_t na, const float* b, uint64_t nb, int dim, uint64_t k, int32_t* idx, float* dist)
{
  if (!idx || !dist || dim <= 0) return MM3D_ERR_ARG;
  MM_TRY(ctx)
  const int kk = (int)std::min<uint64_t>(k, nb);
  if (na == 0 || kk == 0) return MM3D_OK;
  DBuf<float> da(c, na * dim), db(c, nb * dim);
  da.upload(c, a, na * dim);
  db.upload(c, b, nb * dim);
  DBuf<int> di(c, na * kk);
  DBuf<float> dd(c, na * kk);
  knn_problems(c, {da.p, db.p}, {(int)na, (int)nb}, dim, {KnnProblem{0, 1, (int)na, kk, di.p, dd.p}});
  std::vector<int> hi(na * kk);
  std::vector<float> hd(na * kk);
  di.download(c, hi.data(), hi.size());
  dd.download(c, hd.data(), hd.size());
  c.sync();
  for (uint64_t r = 0; r < na; ++r)
    for (uint64_t t = 0; t < k; ++t) {
      idx[r * k + t] = t < (uint64_t)kk ? hi[r * kk + t] : -1;
      dist[r * k + t] = t < (uint64_t)kk ? hd[r * kk + t] : 0.f;
    }
  MM_CATCH
}

int mm3d_knn_tc_audit(mm3d_ctx* ctx, const float* a, uint64_t na, const float* b, uint64_t nb, int dim, uint64_t k, int32_t* idx, float* dist,
                      float* acc, float* norm_a, float* norm_b, float* err_store)
{
  if (!idx || !dist || !acc || !norm_a || !norm_b || !err_store) return MM3D_ERR_ARG;
  MM_TRY(ctx)
  if (dim != 33 || k == 0 || k > 5 || na == 0 || nb < k) throw UnsupportedError("unsupported: the audit covers 33-dimensional descriptors and k <= 5");
  DBuf<float> da(c, na * dim), db(c, nb * dim);
  da.upload(c, a, na * dim);
  db.upload(c, b, nb * dim);
  DBuf<int> di(c, na * k);
  DBuf<float> dd(c, na * k);
  KnnAudit au;
  knn_tc_batch(c, {da.p, db.p}, {(int)na, (int)nb}, dim, {KnnProblem{0, 1, (int)na, (int)k, di.p, dd.p}}, &au);
  di.download(c, idx, na * k);
  dd.download(c, dist, na * k);
  c.sync();
  if (au.acc.size() != na * nb) throw std::runtime_error("knn_tc_audit: no audit data");
  memcpy(acc, au.acc.data(), au.acc.size() * sizeof(float));
  memcpy(norm_a, au.norm_a.data(), au.norm_a.size() * sizeof(float));
  memcpy(norm_b, au.norm_b.data(), au.norm_b.size() * sizeof(float));
  *err_store = au.err_store;
  MM_CATCH
}

int mm3d_ransac(mm3d_ctx* ctx, const float* kp_src, uint64_t n_src, const float* kp_tgt, uint64_t n_tgt, const int32_t* pairs,
                uint64_t n_corr, double inlier_threshold, float* transform, int32_t** inliers, uint64_t* n_inliers, int32_t* dbg,
                double* dbg_d, float* best_model)
{
  if (!transform) return MM3D_ERR_ARG;
  MM_TRY(ctx)
  DCloud s = upload_cloud(c, kp_src, n_src), t = upload_cloud(c, kp_tgt, n_tgt);
  std::vector<DCorr> corr(1);
  corr[0].n = (int)n_corr;
  corr[0].pairs.alloc(c, n_corr);
  if (n_corr) MM_CUDA(cudaMemcpyAsync(corr[0].pairs.p, pairs, n_corr * sizeof(int2), cudaMemcpyHostToDevice, c.stream));
  std::vector<RansacOut> out;
  std::vector<std::vector<int>> inl;
  ransac_batch(c, {s.view(), t.view()}, {PairJob{0, 1}}, corr, inlier_threshold, out, &inl);
  to_colmajor(out[0].T, transform);
  if (inliers) {
    *inliers = (int32_t*)malloc(std::max<size_t>(inl[0].size(), 1) * 4);
    memcpy(*inliers, inl[0].data(), inl[0].size() * 4);
  }
  if (n_inliers) *n_inliers = inl[0].size();
  if (dbg) { dbg[0] = out[0].iterations; dbg[1] = out[0].best_count; }
  if (dbg_d) *dbg_d = out[0].sample_dist_thresh;
  if (best_model) to_colmajor(out[0].best_model, best_model);
  MM_CATCH
}

int mm3d_sac_ia(mm3d_ctx* ctx, const float* kp_src, uint64_t n_src, const float* desc_src, const float* kp_tgt, uint64_t n_tgt,
                const float* desc_tgt, int dim, double min_sample_distance, double max_correspondence_distance, int max_iterations,
                uint64_t* rand_calls, float* transform, float** errors, uint64_t* n_errors)
{
  if (!transform) return MM3D_ERR_ARG;
  MM_TRY(ctx)
  DCloud s = upload_cloud(c, kp_src, n_src), t = upload_cloud(c, kp_tgt, n_tgt);
  DBuf<float> a(c, n_src * dim), b(c, n_tgt * dim);
  a.upload(c, desc_src, n_src * dim);
  b.upload(c, desc_tgt, n_tgt * dim);
  std::vector<SacOut> so;
  sac_ia_batch(c, {s.view(), t.view()}, {a.p, b.p}, dim, {PairJob{0, 1}}, {0}, min_sample_distance, max_correspondence_distance, max_iterations,
               rand_calls ? *rand_calls : 0, so);
  to_colmajor(so[0].T, transform);
  if (rand_calls) *rand_calls = so[0].rand_calls;
  if (errors) {
    *errors = (float*)malloc(std::max<size_t>(so[0].errors.size(), 1) * 4);
    memcpy(*errors, so[0].errors.data(), so[0].errors.size() * 4);
    *n_errors = so[0].errors.size();
  }
  MM_CATCH
}

int mm3d_icp(mm3d_ctx* ctx, const float* src, uint64_t n_src, const float* tgt, uint64_t n_tgt, const float* initial_guess,
             double max_correspondence_distance, double outlier_rejection_threshold, int max_iterations, double transformation_epsilon,
             double index_leaf, float* transform, int32_t* dbg, long long** sums, uint64_t* n_sums)
{
  (void)outlier_rejection_threshold;  // set on pcl::IterativeClosestPoint but without effect (matching.cpp:206)
  if (!transform) return MM3D_ERR_ARG;
  MM_TRY(ctx)
  DCloud s = upload_cloud(c, src, n_src), t = upload_cloud(c, tgt, n_tgt);
  std::vector<DIndex> idx;
  const double leaf = auto_leaf(index_leaf, max_correspondence_distance, 10.0);
  build_index_batch(c, {CloudView{nullptr, 0}, t.view()}, (float)leaf, 0, 0, 0, idx);
  std::vector<DReach> reach;
  build_reach_batch(c, idx, (int)std::ceil(max_correspondence_distance / leaf) + 1, reach);
  float t0[16];
  from_colmajor(initial_guess, t0);
  std::vector<IcpOut> out;
  std::vector<std::vector<long long>> sd;
  icp_batch(c, {s.view(), t.view()}, idx, reach, {PairJob{0, 1}}, {t0}, max_correspondence_distance, max_iterations, transformation_epsilon,
            out, sums ? &sd : nullptr);
  to_colmajor(out[0].T, transform);
  if (dbg) { dbg[0] = out[0].iterations; dbg[1] = out[0].converged; }
  if (sums) {
    *sums = (long long*)malloc(std::max<size_t>(sd[0].size(), 1) * 8);
    memcpy(*sums, sd[0].data(), sd[0].size() * 8);
    *n_sums = sd[0].size() / 17;
  }
  MM_CATCH
}

int mm3d_score(mm3d_ctx* ctx, const float* src, uint64_t n_src, const float* tgt, uint64_t n_tgt, const float* transform,
               double max_distance, double index_leaf, double* score)
{
  if (!score) return MM3D_ERR_ARG;
  MM_TRY(ctx)
  DCloud s = upload_cloud(c, src, n_src), t = upload_cloud(c, tgt, n_tgt);
  std::vector<DIndex> idx;
  const double leaf = auto_leaf(index_leaf, std::sqrt(std::max(max_distance, 1e-12)), 10.0);
  build_index_batch(c, {CloudView{nullptr, 0}, t.view()}, (float)leaf, 0, 0, 0, idx);
  std::vector<DReach> reach;
  build_reach_batch(c, idx, (int)std::ceil(std::sqrt(std::max(max_distance, 0.0)) / leaf) + 1, reach);
  float tr[16];
  from_colmajor(transform, tr);
  std::vector<double> sc;
  score_batch(c, {s.view(), t.view()}, idx, reach, {PairJob{0, 1}}, {tr}, max_distance, sc);
  *score = sc[0];
  MM_CATCH
}

int mm3d_global_transforms(int n_pairs, const int32_t* st, const float* transforms, const double* confidences, double confidence_threshold,
                           float* out, int* n_out, int* reference_frame, int32_t* in_component, int32_t* tree_edges, int* n_tree_edges,
                           int32_t* centers, int* n_centers)
{
  if (!out || !n_out) return MM3D_ERR_ARG;
  try {
    std::vector<HostEstimate> est(n_pairs);
    for (int i = 0; i < n_pairs; ++i) {
      est[i].source_idx = (size_t)st[2 * i];
      est[i].target_idx = (size_t)st[2 * i + 1];
      from_colmajor(transforms + 16 * i, est[i].T);
      est[i].confidence = confidences[i];
    }
    std::vector<int> inc, cen;
    std::vector<std::pair<int, int>> te;
    int ref = -1;
    std::vector<std::vector<float>> g = compute_global_transforms(est, confidence_threshold, &ref, &inc, &te, &cen);
    for (size_t i = 0; i < g.size(); ++i) to_colmajor(g[i].data(), out + 16 * i);
    *n_out = (int)g.size();
    if (reference_frame) *reference_frame = ref;
    if (in_component)
      for (int i = 0; i < n_pairs; ++i) in_component[i] = inc[i];
    if (tree_edges)
      for (size_t i = 0; i < te.size(); ++i) { tree_edges[2 * i] = te[i].first; tree_edges[2 * i + 1] = te[i].second; }
    if (n_tree_edges) *n_tree_edges = (int)te.size();
    if (centers)
      for (size_t i = 0; i < cen.size(); ++i) centers[i] = cen[i];
    if (n_centers) *n_centers = (int)cen.size();
  } catch (const std::exception&) {
    return MM3D_ERR;
  }
  return MM3D_OK;
}

int mm3d_knn_stats(mm3d_ctx* ctx, uint64_t* out)
{
  if (!out) return MM3D_ERR_ARG;
  MM_TRY(ctx)
  out[0] = out[1] = out[2] = 0;
  if (c.knn_stats) {
    unsigned long long h[3];
    MM_CUDA(cudaMemcpyAsync(h, c.knn_stats, sizeof(h), cudaMemcpyDeviceToHost, c.stream));
    c.sync();
    for (int i = 0; i < 3; ++i) out[i] = h[i];
  }
  MM_CATCH
}

int mm3d_profile_begin(mm3d_ctx* ctx)
{
  MM_TRY(ctx)
  c.sync();
  for (KernelSample& s : c.samples) { c.event_pool.push_back(s.e0); c.event_pool.push_back(s.e1); }
  c.samples.clear();
  c.profiling = true;
  MM_CATCH
}

int mm3d_profile_end(mm3d_ctx* ctx, char** json)
{
  if (!json) return MM3D_ERR_ARG;
  *json = nullptr;
  MM_TRY(ctx)
  c.sync();
  c.profiling = false;
  struct Agg { std::string name; long long n = 0; double ms = 0, bytes = 0, ms_annotated = 0; };
  std::vector<Agg> agg;
  for (KernelSample& s : c.samples) {
    float ms = 0.f;
    MM_CUDA(cudaEventElapsedTime(&ms, s.e0, s.e1));
    size_t k = 0;
    for (; k < agg.size(); ++k)
      if (agg[k].name == s.name) break;
    if (k == agg.size()) { agg.emplace_back(); agg.back().name = s.name; }
    agg[k].n += 1;
    agg[k].ms += ms;
    agg[k].bytes += s.bytes;
    if (s.bytes > 0) agg[k].ms_annotated += ms;
    c.event_pool.push_back(s.e0);
    c.event_pool.push_back(s.e1);
  }
  c.samples.clear();
  std::string out = "[";
  for (size_t k = 0; k < agg.size(); ++k) {
    char buf[512];
    snprintf(buf, sizeof(buf), "%s{\"kernel\": \"%s\", \"launches\": %lld, \"ms\": %.6f, \"algorithmic_bytes\": %.1f, \"ms_annotated\": %.6f}",
             k ? ", " : "", agg[k].name.c_str(), agg[k].n, agg[k].ms, agg[k].bytes, agg[k].ms_annotated);
    out += buf;
  }
  out += "]";
  *json = (char*)malloc(out.size() + 1);
  memcpy(*json, out.c_str(), out.size() + 1);
  MM_CATCH
}

// ---- composeMaps sharded over ranks --------------------------------------------

int mm3d_compose_shard_begin(mm3d_ctx* ctx, int n_maps, const float* const* clouds, const uint64_t* n_points, int n_transforms,
                             const float* transforms, float* bbox, mm3d_shard** shard)
{
  if (!bbox || !shard) return MM3D_ERR_ARG;
  *shard = nullptr;
  if (n_maps != n_transforms) {
    if (ctx) ctx->c.err = "composeMaps: clouds and transforms size must be the same.";
    return MM3D_ERR_ARG;
  }
  MM_TRY(ctx)
  std::vector<DCloud> d;
  std::vector<std::vector<float>> tr;
  for (int m = 0; m < n_maps; ++m) {
    float rm[16];
    from_colmajor(transforms + 16 * m, rm);
    bool zero = true;
    for (int k = 0; k < 16; ++k)
      if (!(std::fabs(rm[k]) <= 1e-5f)) zero = false;
    if (zero || !clouds[m] || n_points[m] == 0) continue;
    d.push_back(upload_cloud(c, clouds[m], n_points[m]));
    tr.emplace_back(rm, rm + 16);
  }
  std::vector<CloudView> v;
  std::vector<const float*> tp;
  for (size_t i = 0; i < d.size(); ++i) {
    v.push_back(d[i].view());
    tp.push_back(tr[i].data());
  }
  std::unique_ptr<mm3d_shard> s(new mm3d_shard);
  transform_concat(c, v, tp, s->cloud);
  compose_bbox(c, s->cloud, bbox);
  *shard = s.release();
  MM_CATCH
}

int mm3d_compose_shard_size(const mm3d_shard* shard, uint64_t* n)
{
  if (!shard || !n) return MM3D_ERR_ARG;
  *n = (uint64_t)shard->cloud.n;
  return MM3D_OK;
}

int mm3d_compose_shard_histogram(mm3d_ctx* ctx, const mm3d_shard* shard, const float* global_bbox, double resolution, int n_buckets,
                                 uint64_t* hist)
{
  if (!shard || !global_bbox || !hist || n_buckets <= 0) return MM3D_ERR_ARG;
  MM_TRY(ctx)
  const KeyGeomHost g = compose_geometry(global_bbox, resolution, n_buckets);
  if (g.passthrough) return 1;  // overflow guard of pcl::VoxelGrid: the composed map is the plain concatenation
  std::vector<unsigned long long> h(n_buckets);
  compose_histogram(c, shard->cloud, g, n_buckets, h.data());
  for (int i = 0; i < n_buckets; ++i) hist[i] = h[i];
  MM_CATCH
}

int mm3d_compose_shard_partition(mm3d_ctx* ctx, const mm3d_shard* shard, const float* global_bbox, double resolution, int n_buckets, int n_ranks,
                                 const int32_t* splitters, uint64_t* send_counts, void* points_dev)
{
  if (!shard || !global_bbox || !splitters || !send_counts || n_ranks <= 0) return MM3D_ERR_ARG;
  MM_TRY(ctx)
  const KeyGeomHost g = compose_geometry(global_bbox, resolution, n_buckets);
  std::vector<int> sp(splitters, splitters + n_ranks + 1);
  std::vector<unsigned long long> cnt(n_ranks);
  compose_partition(c, shard->cloud, g, n_buckets, sp, n_ranks, cnt.data(), (float4*)points_dev);
  for (int r = 0; r < n_ranks; ++r) send_counts[r] = cnt[r];
  MM_CATCH
}

int mm3d_compose_shard_points(mm3d_ctx* ctx, const mm3d_shard* shard, float** out, uint64_t* n_out)
{
  if (!shard || !out || !n_out) return MM3D_ERR_ARG;
  MM_TRY(ctx)
  *out = (float*)host_copy(c, shard->cloud.pts.p, (size_t)shard->cloud.n);
  *n_out = (uint64_t)shard->cloud.n;
  c.sync();
  MM_CATCH
}

void mm3d_shard_free(mm3d_shard* shard) { delete shard; }

int mm3d_downsample_dev(mm3d_ctx* ctx, const void* points_dev, uint64_t n, double resolution, float** out, uint64_t* n_out)
{
  if (!out || !n_out) return MM3D_ERR_ARG;
  MM_TRY(ctx)
  std::vector<DCloud> res;
  voxel_downsample_batch(c, {CloudView{(const float4*)points_dev, (int)n}}, (float)resolution, res, nullptr);
  *out = (float*)host_copy(c, res[0].pts.p, (size_t)res[0].n);
  *n_out = (uint64_t)res[0].n;
  c.sync();
  MM_CATCH
}

// ---- resident interface -----------------------------------------------------

int mm3d_maps_upload(mm3d_ctx* ctx, int n_maps, const float* const* clouds, const uint64_t* n_points, mm3d_maps** maps)
{
  return mm3d_maps_upload_layout(ctx, n_maps, (const void* const*)clouds, n_points, &kPackedLayout, maps);
}

int mm3d_maps_upload_layout(mm3d_ctx* ctx, int n_maps, const void* const* clouds, const uint64_t* n_points, const mm3d_layout* layout,
                            mm3d_maps** maps)
{
  if (!maps) return MM3D_ERR_ARG;
  *maps = nullptr;
  if (!layout_valid(layout)) return bad_layout(ctx);
  MM_TRY(ctx)
  std::unique_ptr<mm3d_maps> h(new mm3d_maps);
  h->clouds = upload_clouds(c, std::vector<const void*>(clouds, clouds + n_maps), std::vector<uint64_t>(n_points, n_points + n_maps), *layout);
  c.sync();
  *maps = h.release();
  MM_CATCH
}

void mm3d_maps_free(mm3d_maps* maps) { delete maps; }

int mm3d_features_compute(mm3d_ctx* ctx, const mm3d_maps* maps, int first, int count, const mm3d_params* params, mm3d_features** out)
{
  if (!maps || !out || first < 0 || count < 0 || first + count > (int)maps->clouds.size()) return MM3D_ERR_ARG;
  *out = nullptr;
  MM_TRY(ctx)
  std::vector<CloudView> v(count);
  for (int m = 0; m < count; ++m) v[m] = maps->clouds[first + m].view();
  std::unique_ptr<mm3d_features> f(new mm3d_features);
  compute_features(c, v, *params, f->maps, nullptr);
  f->dim = desc_dim(*params);
  *out = f.release();
  MM_CATCH
}

int mm3d_features_count(const mm3d_features* f) { return f ? (int)f->maps.size() : 0; }

int mm3d_features_sizes(const mm3d_features* f, int32_t* n_points, int32_t* n_keypoints, int32_t* dim)
{
  if (!f) return MM3D_ERR_ARG;
  for (size_t m = 0; m < f->maps.size(); ++m) {
    if (n_points) n_points[m] = f->maps[m].cloud.n;
    if (n_keypoints) n_keypoints[m] = f->maps[m].keypoints.n;
  }
  if (dim) *dim = f->dim;
  return MM3D_OK;
}

int mm3d_features_export_dev(mm3d_ctx* ctx, const mm3d_features* f, int map, void* points_dev, void* keypoints_dev, void* descriptors_dev)
{
  if (!f || map < 0 || map >= (int)f->maps.size()) return MM3D_ERR_ARG;
  MM_TRY(ctx)
  const MapFeat& m = f->maps[map];
  if (points_dev && m.cloud.n) MM_CUDA(cudaMemcpyAsync(points_dev, m.cloud.pts.p, (size_t)m.cloud.n * 16, cudaMemcpyDeviceToDevice, c.stream));
  if (keypoints_dev && m.keypoints.n)
    MM_CUDA(cudaMemcpyAsync(keypoints_dev, m.keypoints.pts.p, (size_t)m.keypoints.n * 16, cudaMemcpyDeviceToDevice, c.stream));
  if (descriptors_dev && m.keypoints.n)
    MM_CUDA(cudaMemcpyAsync(descriptors_dev, m.desc.p, (size_t)m.keypoints.n * f->dim * 4, cudaMemcpyDeviceToDevice, c.stream));
  c.sync();
  MM_CATCH
}

int mm3d_features_export_host(mm3d_ctx* ctx, const mm3d_features* f, int map, float* points, float* keypoints, float* descriptors)
{
  if (!f || map < 0 || map >= (int)f->maps.size()) return MM3D_ERR_ARG;
  MM_TRY(ctx)
  const MapFeat& m = f->maps[map];
  if (points && m.cloud.n) MM_CUDA(cudaMemcpyAsync(points, m.cloud.pts.p, (size_t)m.cloud.n * 16, cudaMemcpyDeviceToHost, c.stream));
  if (keypoints && m.keypoints.n) MM_CUDA(cudaMemcpyAsync(keypoints, m.keypoints.pts.p, (size_t)m.keypoints.n * 16, cudaMemcpyDeviceToHost, c.stream));
  if (descriptors && m.keypoints.n)
    MM_CUDA(cudaMemcpyAsync(descriptors, m.desc.p, (size_t)m.keypoints.n * f->dim * 4, cudaMemcpyDeviceToHost, c.stream));
  c.sync();
  MM_CATCH
}

int mm3d_features_import_dev(mm3d_ctx* ctx, int n_maps, const int32_t* n_points, const void* const* points_dev, const int32_t* n_keypoints,
                             const void* const* keypoints_dev, const void* const* descriptors_dev, int dim, mm3d_features** out)
{
  if (!out) return MM3D_ERR_ARG;
  *out = nullptr;
  MM_TRY(ctx)
  std::unique_ptr<mm3d_features> f(new mm3d_features);
  f->dim = dim;
  f->maps.resize(n_maps);
  for (int m = 0; m < n_maps; ++m) {
    MapFeat& mf = f->maps[m];
    mf.cloud.n = n_points[m];
    mf.cloud.pts.alloc(c, n_points[m]);
    if (n_points[m]) MM_CUDA(cudaMemcpyAsync(mf.cloud.pts.p, points_dev[m], (size_t)n_points[m] * 16, cudaMemcpyDeviceToDevice, c.stream));
    mf.keypoints.n = n_keypoints[m];
    mf.keypoints.pts.alloc(c, n_keypoints[m]);
    mf.desc.alloc(c, (size_t)n_keypoints[m] * dim);
    if (n_keypoints[m]) {
      MM_CUDA(cudaMemcpyAsync(mf.keypoints.pts.p, keypoints_dev[m], (size_t)n_keypoints[m] * 16, cudaMemcpyDeviceToDevice, c.stream));
      MM_CUDA(cudaMemcpyAsync(mf.desc.p, descriptors_dev[m], (size_t)n_keypoints[m] * dim * 4, cudaMemcpyDeviceToDevice, c.stream));
    }
  }
  c.sync();
  *out = f.release();
  MM_CATCH
}

void mm3d_features_free(mm3d_features* f) { delete f; }

int mm3d_register_pairs(mm3d_ctx* ctx, const mm3d_features* f, int n_pairs, const int32_t* ij, const mm3d_params* params, float* transforms,
                        double* confidences, int32_t* stats)
{
  if (!f || (n_pairs > 0 && (!ij || !transforms || !confidences))) return MM3D_ERR_ARG;
  MM_TRY(ctx)
  std::vector<PairJob> jobs(n_pairs);
  for (int k = 0; k < n_pairs; ++k) {
    jobs[k] = PairJob{ij[2 * k], ij[2 * k + 1]};
    if (jobs[k].a < 0 || jobs[k].b < 0 || jobs[k].a >= (int)f->maps.size() || jobs[k].b >= (int)f->maps.size())
      throw std::runtime_error("register_pairs: pair index out of range");
  }
  std::vector<PairOut> po;
  register_pairs(c, feat_views(f->maps), f->dim, jobs, *params, po, nullptr);
  for (int k = 0; k < n_pairs; ++k) {
    to_colmajor(po[k].T, transforms + 16 * k);
    confidences[k] = po[k].confidence;
    if (stats) {
      stats[4 * k] = po[k].n_corr;
      stats[4 * k + 1] = po[k].n_inliers;
      stats[4 * k + 2] = po[k].icp_iterations;
      stats[4 * k + 3] = po[k].icp_converged;
    }
  }
  MM_CATCH
}

int mm3d_estimate_resident(mm3d_ctx* ctx, const mm3d_maps* maps, const mm3d_params* params, float* out_transforms, int* n_out,
                           float* stage_ms)
{
  if (!maps || !n_out) return MM3D_ERR_ARG;
  *n_out = 0;
  MM_TRY(ctx)
  if (stage_ms)
    for (int i = 0; i < 10; ++i) stage_ms[i] = 0.f;
  std::vector<CloudView> v(maps->clouds.size());
  for (size_t m = 0; m < v.size(); ++m) v[m] = maps->clouds[m].view();
  *n_out = estimate_from_views(c, v, *params, out_transforms, stage_ms);
  c.sync();
  MM_CATCH
}

}  // extern "C"
