// mapset.cu — a resident, ordered set of maps (include/mm3d.h, "map set") that keeps each map's raw cloud, its features and
// every pair's registration between calls, so that repeated estimateMapsTransforms / composeMaps over the latest map of each
// robot (the reference's ROS node, map_merge_node) redo only the work whose inputs changed.
//
// What stays valid, and why the result cannot change:
//   * a map's features depend on its raw cloud and the parameters only (every batched feature kernel computes each map on
//     its own), so they are kept until the cloud changes bit for bit or any parameter changes;
//   * a pair's result depends on the two maps' features and the parameters.  MATCHING seeds RANSAC with mt19937(12345) per
//     pair.  SAC_IA draws from one C rand() stream that runs through the whole row-major pair list, so its result also
//     depends on the offset at which the pair's draws start; a pair whose maps did not change is reused only when that
//     offset equals the one it was registered with.
#include <cstring>
#include <map>
#include <memory>
#include <utility>

#include "../../include/mm3d.h"
#include "mm3d_internal.cuh"
#include "pipeline.cuh"

using namespace mm3d;

namespace {

struct Slot {
  DCloud raw;          // the cloud as last updated, packed layout
  MapFeat feat;        // valid when !dirty
  bool dirty = true;   // raw changed since feat was computed
};

struct PairCache {
  float T[16];  // row-major
  double confidence;
  unsigned long long rand_start;  // SAC_IA: rand() calls made before the pair's draws
};

}  // namespace

struct mm3d_mapset {
  mm3d_ctx* ctx;
  std::vector<Slot> slots;
  bool have_params = false;  // params and pairs hold the last successful estimate
  mm3d_params params;
  std::map<std::pair<int, int>, PairCache> pairs;
};

namespace {

struct CmpJob {
  const uint4* a;
  const uint4* b;
  unsigned long long n;  // points
};

// Sets differs[blockIdx.y] when two clouds of equal size differ in any 32-bit word (bitwise: NaN payloads and signed zeros
// count).  One vote per warp and one atomic per warp that saw a difference.
__global__ void __launch_bounds__(256) mapset_compare_kernel(const CmpJob* __restrict__ jobs, int* __restrict__ differs)
{
  const CmpJob j = jobs[blockIdx.y];
  bool d = false;
  for (unsigned long long i = (unsigned long long)blockIdx.x * blockDim.x + threadIdx.x; i < j.n; i += (unsigned long long)gridDim.x * blockDim.x) {
    const uint4 x = __ldcs(j.a + i), y = __ldcs(j.b + i);
    d |= (x.x != y.x) | (x.y != y.y) | (x.z != y.z) | (x.w != y.w);
  }
  if (__any_sync(0xffffffffu, d) && (threadIdx.x & 31) == 0) atomicOr(differs + blockIdx.y, 1);
}

// differs[k] = 1 when the clouds of job k differ; one launch per 65535 jobs (gridDim.y)
void compare_clouds(Ctx& c, const std::vector<CmpJob>& jobs, std::vector<int>& differs)
{
  differs.assign(jobs.size(), 0);
  if (jobs.empty()) return;
  DBuf<CmpJob> dj = to_device(c, jobs);
  DBuf<int> dd(c, jobs.size());
  dd.zero(c);
  constexpr int kMaxY = 65535, kThreads = 256;
  for (size_t first = 0; first < jobs.size(); first += kMaxY) {
    const int count = (int)std::min<size_t>(kMaxY, jobs.size() - first);
    unsigned long long max_n = 0;
    double bytes = 0;
    for (int k = 0; k < count; ++k) {
      max_n = std::max(max_n, jobs[first + k].n);
      bytes += 32.0 * jobs[first + k].n;
    }
    const unsigned gx = (unsigned)std::min<unsigned long long>((max_n + 4 * kThreads - 1) / (4 * kThreads), 1024);
    MM_BYTES(c, bytes);
    MM_LAUNCH(c, mapset_compare_kernel, dim3(gx, count), kThreads, 0, dj.p + first, dd.p + first);
  }
  dd.download(c, differs.data(), jobs.size());
  c.sync();
}

// every field compared by value bits, so -0.0 and NaN payloads count as changes
bool same_params(const mm3d_params& a, const mm3d_params& b)
{
  auto eq = [](double x, double y) { return std::memcmp(&x, &y, sizeof(double)) == 0; };
  return eq(a.resolution, b.resolution) && eq(a.descriptor_radius, b.descriptor_radius) && a.outliers_min_neighbours == b.outliers_min_neighbours &&
         eq(a.normal_radius, b.normal_radius) && a.keypoint_type == b.keypoint_type && eq(a.keypoint_threshold, b.keypoint_threshold) &&
         a.descriptor_type == b.descriptor_type && a.estimation_method == b.estimation_method && a.refine_transform == b.refine_transform &&
         eq(a.inlier_threshold, b.inlier_threshold) && eq(a.max_correspondence_distance, b.max_correspondence_distance) &&
         a.max_iterations == b.max_iterations && a.matching_k == b.matching_k && eq(a.transform_epsilon, b.transform_epsilon) &&
         eq(a.confidence_threshold, b.confidence_threshold) && eq(a.output_resolution, b.output_resolution);
}

int arg_error(mm3d_ctx* ctx, const char* what)
{
  if (ctx) ctx->c.err = what;
  return MM3D_ERR_ARG;
}

// estimateMapsTransforms over the slots; returns the number of transforms written.  The set changes only at the end.
int mapset_estimate(Ctx& c, mm3d_mapset& s, const mm3d_params& p, float* out_transforms, int32_t* work)
{
  const int M = (int)s.slots.size();
  if (M == 0) return 0;
  if (M == 1) {  // map_merging.cpp:192-197: no device work; the slot stays dirty
    const float id[16] = {1, 0, 0, 0, 0, 1, 0, 0, 0, 0, 1, 0, 0, 0, 0, 1};
    memcpy(out_transforms, id, sizeof(id));
    return 1;
  }
  check_supported(p);  // as compute_features does in the stateless call, even when nothing is left to compute
  const bool all = !s.have_params || !same_params(s.params, p);
  std::vector<char> dirty(M);
  std::vector<int> todo;       // dirty slots
  std::vector<int> computed;   // positions in todo of the non-empty ones: an empty cloud has no keypoints and so no pairs
  std::vector<CloudView> raw;
  for (int m = 0; m < M; ++m) {
    dirty[m] = all || s.slots[m].dirty;
    if (!dirty[m]) continue;
    if (s.slots[m].raw.n > 0) {
      computed.push_back((int)todo.size());
      raw.push_back(s.slots[m].raw.view());
    }
    todo.push_back(m);
  }
  std::vector<MapFeat> fresh(todo.size());
  if (!raw.empty()) {
    std::vector<MapFeat> f;
    compute_features(c, raw, p, f, nullptr);
    for (size_t k = 0; k < computed.size(); ++k) fresh[computed[k]] = std::move(f[k]);
  }
  std::vector<FeatView> fv(M);
  for (int m = 0, t = 0; m < M; ++m) {
    const MapFeat& f = dirty[m] ? fresh[t++] : s.slots[m].feat;
    fv[m] = FeatView{f.cloud.view(), f.keypoints.view(), f.desc.p};
  }
  // src/map_merging.cpp:246-254
  std::vector<PairJob> all_pairs;
  for (int i = 0; i < M - 1; ++i)
    for (int j = i + 1; j < M; ++j)
      if (fv[i].keypoints.n > 0 && fv[j].keypoints.n > 0) all_pairs.push_back(PairJob{i, j});
  const int P = (int)all_pairs.size();
  // SAC_IA: where each pair's draws start.  Without a changed map no pair's features, and so no offset, can have moved.
  const bool walk = p.estimation_method == MM3D_EST_SAC_IA && !todo.empty();
  std::vector<unsigned long long> starts(P, 0);
  if (walk) {
    std::vector<CloudView> kps(M);
    std::vector<const float*> desc(M);
    for (int m = 0; m < M; ++m) {
      kps[m] = fv[m].keypoints;
      desc[m] = fv[m].desc;
    }
    std::vector<SacOut> none;
    sac_ia_batch(c, kps, desc, desc_dim(p), all_pairs, {}, p.inlier_threshold, p.max_correspondence_distance, p.max_iterations, 0, none, &starts);
  }
  std::vector<const PairCache*> reuse(P, nullptr);
  std::vector<PairJob> jobs;
  std::vector<int> job_of(P, -1);
  for (int k = 0; k < P; ++k) {
    const PairJob& pj = all_pairs[k];
    if (!dirty[pj.a] && !dirty[pj.b]) {
      auto it = s.pairs.find({pj.a, pj.b});
      if (it != s.pairs.end() && (!walk || it->second.rand_start == starts[k])) {
        reuse[k] = &it->second;
        continue;
      }
    }
    job_of[k] = (int)jobs.size();
    jobs.push_back(pj);
  }
  std::vector<PairOut> po;
  if (!jobs.empty()) register_pairs(c, fv, desc_dim(p), jobs, p, po, nullptr);
  std::map<std::pair<int, int>, PairCache> table;
  std::vector<HostEstimate> est(P);
  for (int k = 0; k < P; ++k) {
    PairCache pc;
    if (reuse[k]) {
      pc = *reuse[k];
    } else {
      memcpy(pc.T, po[job_of[k]].T, sizeof(pc.T));
      pc.confidence = po[job_of[k]].confidence;
      pc.rand_start = starts[k];
    }
    est[k].source_idx = (size_t)all_pairs[k].a;
    est[k].target_idx = (size_t)all_pairs[k].b;
    memcpy(est[k].T, pc.T, sizeof(pc.T));
    est[k].confidence = pc.confidence;
    table[{all_pairs[k].a, all_pairs[k].b}] = pc;
  }
  std::vector<std::vector<float>> g = compute_global_transforms(est, p.confidence_threshold, nullptr, nullptr, nullptr, nullptr);
  for (size_t i = 0; i < g.size(); ++i) to_colmajor(g[i].data(), out_transforms + 16 * i);
  // commit
  for (size_t t = 0; t < todo.size(); ++t) {
    s.slots[todo[t]].feat = std::move(fresh[t]);
    s.slots[todo[t]].dirty = false;
  }
  s.params = p;
  s.have_params = true;
  s.pairs = std::move(table);
  if (work) {
    work[0] = (int32_t)todo.size();
    work[1] = (int32_t)jobs.size();
    work[2] = (int32_t)(P - jobs.size());
  }
  return (int)g.size();
}

}  // namespace

extern "C" {

int mm3d_mapset_create(mm3d_ctx* ctx, mm3d_mapset** set)
{
  if (!ctx || !set) return MM3D_ERR_ARG;
  *set = new mm3d_mapset;
  (*set)->ctx = ctx;
  return MM3D_OK;
}

int mm3d_mapset_size(const mm3d_mapset* set) { return set ? (int)set->slots.size() : 0; }

void mm3d_mapset_free(mm3d_mapset* set) { delete set; }

int mm3d_mapset_update(mm3d_ctx* ctx, mm3d_mapset* set, int n, const int32_t* slots, const void* const* clouds, const uint64_t* n_points,
                       const mm3d_layout* layout, int32_t* changed)
{
  if (!set || n < 0 || (n > 0 && (!slots || !clouds || !n_points))) return arg_error(ctx, "mm3d_mapset_update: bad arguments");
  if (!layout_valid(layout)) return arg_error(ctx, "malformed mm3d_layout (include/mm3d.h)");
  if (ctx != set->ctx) return arg_error(ctx, "mm3d_mapset_update: the map set belongs to another context");
  for (int i = 0; i < n; ++i) {
    if (slots[i] < 0) return arg_error(ctx, "mm3d_mapset_update: negative slot index");
    for (int k = 0; k < i; ++k)
      if (slots[k] == slots[i]) return arg_error(ctx, "mm3d_mapset_update: a slot appears twice");
  }
  MM_TRY(ctx)
  std::vector<DCloud> up = upload_clouds(c, std::vector<const void*>(clouds, clouds + n), std::vector<uint64_t>(n_points, n_points + n), *layout);
  const int old = (int)set->slots.size();
  std::vector<int> differs(n, 1), cmp_of(n, -1);
  std::vector<CmpJob> jobs;
  for (int i = 0; i < n; ++i) {
    if (slots[i] >= old) continue;  // a slot the call creates
    const DCloud& r = set->slots[slots[i]].raw;
    if (r.n != up[i].n) continue;
    differs[i] = 0;
    if (r.n == 0) continue;
    cmp_of[i] = (int)jobs.size();
    jobs.push_back(CmpJob{(const uint4*)r.pts.p, (const uint4*)up[i].pts.p, (unsigned long long)r.n});
  }
  std::vector<int> cmp;
  compare_clouds(c, jobs, cmp);
  c.sync();
  // commit
  int size = old;
  for (int i = 0; i < n; ++i) size = std::max(size, slots[i] + 1);
  set->slots.resize(size);
  for (int i = 0; i < n; ++i) {
    if (cmp_of[i] >= 0) differs[i] = cmp[cmp_of[i]];
    if (differs[i]) {
      Slot& sl = set->slots[slots[i]];
      sl.raw = std::move(up[i]);
      sl.feat = MapFeat();
      sl.dirty = true;
    }
    if (changed) changed[i] = differs[i];
  }
  MM_CATCH
}

int mm3d_mapset_estimate(mm3d_ctx* ctx, mm3d_mapset* set, const mm3d_params* params, float* out_transforms, int* n_out, int32_t* work)
{
  if (!n_out) return arg_error(ctx, "mm3d_mapset_estimate: n_out is NULL");
  *n_out = 0;
  if (work) work[0] = work[1] = work[2] = 0;
  if (!set || !params || (!set->slots.empty() && !out_transforms)) return arg_error(ctx, "mm3d_mapset_estimate: bad arguments");
  if (ctx != set->ctx) return arg_error(ctx, "mm3d_mapset_estimate: the map set belongs to another context");
  MM_TRY(ctx)
  *n_out = mapset_estimate(c, *set, *params, out_transforms, work);
  c.sync();
  MM_CATCH
}

int mm3d_mapset_compose(mm3d_ctx* ctx, const mm3d_mapset* set, int n_transforms, const float* transforms, double resolution,
                        const mm3d_layout* out_layout, void** out, uint64_t* n_out)
{
  if (!out || !n_out) return arg_error(ctx, "mm3d_mapset_compose: bad arguments");
  *out = nullptr;
  *n_out = 0;
  if (!set) return arg_error(ctx, "mm3d_mapset_compose: bad arguments");
  if (!layout_valid(out_layout)) return arg_error(ctx, "malformed mm3d_layout (include/mm3d.h)");
  if (ctx != set->ctx) return arg_error(ctx, "mm3d_mapset_compose: the map set belongs to another context");
  const int M = (int)set->slots.size();
  if (M == 0) return 1;  // nullptr result
  if (M != n_transforms) return arg_error(ctx, "composeMaps: clouds and transforms size must be the same.");
  if (!transforms) return arg_error(ctx, "mm3d_mapset_compose: transforms is NULL");
  MM_TRY(ctx)
  std::vector<std::vector<float>> tr;
  std::vector<CloudView> v;
  std::vector<const float*> tp;
  const float any = 0.f;  // skip_map only tests the cloud pointer of host input for NULL
  for (int m = 0; m < M; ++m) {
    float rm[16];
    if (skip_map(transforms + 16 * m, &any, (uint64_t)set->slots[m].raw.n, rm)) continue;
    v.push_back(set->slots[m].raw.view());
    tr.emplace_back(rm, rm + 16);
  }
  for (size_t i = 0; i < tr.size(); ++i) tp.push_back(tr[i].data());
  dist_compose(c, nullptr, v, tp, resolution, *out_layout, out, n_out);
  MM_CATCH
}

}  // extern "C"
