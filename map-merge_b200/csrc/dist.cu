// dist.cu — the hot path over several GPUs, behind the C ABI (include/mm3d.h, "multi-GPU interface").
//
// estimateMapsTransforms (map_merge_3d/src/map_merging.cpp:188-275): the per-map loops (:212-242) are independent per
// map and the pair loop (:256-269) is independent per pair, so rank r runs the feature pipeline for a contiguous block of
// maps, the ranks exchange {cloud, keypoints, descriptors} of every map with NCCL (an all-gather with exact per-rank
// sizes: one in-place ncclBroadcast per root inside a group — nothing is padded), every rank deals the row-major pair list
// out with the same deterministic LPT rule, registers its share and contributes its results to one all-reduce over
// disjoint slots (bit patterns as uint64 sums: adding zeros is exact, so the gathered transforms are bit-identical to a
// single-GPU run and arrive in the reference's pair order, which the pose graph's tie-breaking depends on,
// src/graph.cpp:124).  Every rank then runs the host pose graph.
//
// composeMaps (src/map_merging.cpp:277-305): see compose.cu — two small all-reduces (bounding box, key histogram) and
// one all-to-all of raw points between the per-rank steps.
//
// Two ways to form the ranks:
//   * one process per GPU (bench.py under torchrun, an MPI job, ...): mm3d_comm_id on rank 0, the 128 bytes travel
//     through the launcher's own channel, mm3d_comm_create on every rank;
//   * one process, several GPUs (map_merge_tool, the C++ shim): mm3d_create_multi builds one sub-context + communicator per
//     device (ncclCommInitAll) and the high-level calls fan out over one host thread per device.
// NCCL is loaded with dlopen at the first multi-GPU call (libnccl.so.2: the copy a host process already loaded, e.g.
// torch's, else the system one), so the single-GPU library has no NCCL dependency.
#include <dlfcn.h>
#include <nccl.h>

#include <algorithm>
#include <chrono>
#include <cstring>
#include <mutex>
#include <numeric>
#include <thread>

#include "pipeline.cuh"

using namespace mm3d;

namespace {

struct NcclApi {
  decltype(&ncclGetUniqueId) GetUniqueId = nullptr;
  decltype(&ncclCommInitRank) CommInitRank = nullptr;
  decltype(&ncclCommInitAll) CommInitAll = nullptr;
  decltype(&ncclCommDestroy) CommDestroy = nullptr;
  decltype(&ncclAllGather) AllGather = nullptr;
  decltype(&ncclAllReduce) AllReduce = nullptr;
  decltype(&ncclBroadcast) Broadcast = nullptr;
  decltype(&ncclSend) Send = nullptr;
  decltype(&ncclRecv) Recv = nullptr;
  decltype(&ncclGroupStart) GroupStart = nullptr;
  decltype(&ncclGroupEnd) GroupEnd = nullptr;
  decltype(&ncclGetErrorString) GetErrorString = nullptr;
};

NcclApi& nccl()
{
  static NcclApi api;
  static std::once_flag once;
  static std::string error;
  std::call_once(once, [] {
    void* h = dlopen("libnccl.so.2", RTLD_NOW | RTLD_GLOBAL);
    if (!h) h = dlopen("libnccl.so", RTLD_NOW | RTLD_GLOBAL);
    if (!h) {
      error = std::string("NCCL is not available (dlopen libnccl.so.2: ") + dlerror() + ")";
      return;
    }
#define MM_SYM(name)                                                  \
  api.name = (decltype(api.name))dlsym(h, "nccl" #name);              \
  if (!api.name) error = "NCCL is missing the symbol nccl" #name;
    MM_SYM(GetUniqueId) MM_SYM(CommInitRank) MM_SYM(CommInitAll) MM_SYM(CommDestroy) MM_SYM(AllGather) MM_SYM(AllReduce)
    MM_SYM(Broadcast) MM_SYM(Send) MM_SYM(Recv) MM_SYM(GroupStart) MM_SYM(GroupEnd) MM_SYM(GetErrorString)
#undef MM_SYM
  });
  if (!error.empty()) throw UnsupportedError("unsupported: " + error);
  return api;
}

#define MM_NCCL(expr)                                                                                                        \
  do {                                                                                                                       \
    ncclResult_t _r = (expr);                                                                                                \
    if (_r != ncclSuccess)                                                                                                   \
      throw CudaError(std::string("CUDA error: NCCL ") + nccl().GetErrorString(_r) + " at " __FILE__ ":" + std::to_string(__LINE__) + \
                      " (" #expr ")");                                                                                       \
  } while (0)

}  // namespace

struct mm3d_comm {
  ncclComm_t comm = nullptr;
  int rank = 0, world = 1;
};

struct mm3d_team {
  std::vector<mm3d_ctx*> subs;  // contexts of devices 1 .. n-1 (device 0 is the owning context)
  std::vector<mm3d_comm> comms; // one per device, rank = position in the device list
  ~mm3d_team()
  {
    for (mm3d_comm& cm : comms)
      if (cm.comm) nccl().CommDestroy(cm.comm);
    for (mm3d_ctx* s : subs) mm3d_destroy(s);
  }
};

mm3d_ctx::mm3d_ctx() {}
mm3d_ctx::~mm3d_ctx() {}

namespace {

int block_per(int n_maps, int world) { return (n_maps + world - 1) / world; }
void block_of(int rank, int world, int n_maps, int* first, int* count)
{
  const int per = block_per(n_maps, world);
  *first = std::min(rank * per, n_maps);
  *count = std::max(0, std::min(per, n_maps - *first));
}

// Estimated cost of registering pair (i, j): the descriptor distance matrix plus the ICP / scoring sweeps over the source
// cloud (several iterations) and the target index.
double pair_cost(int npi, int npj, int nki, int nkj, int dim) { return (double)nki * nkj * dim * 2e-3 + 4.0 * npi + npj; }

// Who registers which pair.  Every rank has to build the neighbour index and the reach grid of each TARGET map its pairs
// name, so pairs are dealt out in chunks that share a target: the pairs of one target (ascending source), cut into chunks of
// at most a quarter of a rank's fair share of the total cost; the chunks go out longest-processing-time-first (descending
// cost, stable; each to the least loaded rank, lowest rank on ties).  A rank then touches ~8 targets instead of all of them
// (config 3 on 8 GPUs), and the granularity still balances the ranks to a few per cent.  Deterministic: every rank computes
// the same plan from the all-gathered sizes.
void lpt_assign(const std::vector<PairJob>& pairs, const std::vector<double>& cost, int world, std::vector<int>& owner)
{
  const int P = (int)pairs.size();
  owner.assign(P, 0);
  if (P == 0 || world <= 1) return;
  double total = 0;
  int max_b = 0;
  for (int k = 0; k < P; ++k) {
    total += cost[k];
    max_b = std::max(max_b, pairs[k].b);
  }
  const double cap = total / world / 4.0;
  // pairs of every target in ascending source order (the list is row-major: ascending source already)
  std::vector<std::vector<int>> by_target(max_b + 1);
  for (int k = 0; k < P; ++k) by_target[pairs[k].b].push_back(k);
  struct Chunk {
    int first, count, target;
    double cost;
  };
  std::vector<Chunk> chunks;
  std::vector<int> flat;  // pair ids, chunk after chunk
  for (int b = 0; b <= max_b; ++b) {
    const std::vector<int>& v = by_target[b];
    size_t i = 0;
    while (i < v.size()) {
      Chunk ch{(int)flat.size(), 0, b, 0.0};
      do {
        ch.cost += cost[v[i]];
        flat.push_back(v[i]);
        ++ch.count;
        ++i;
      } while (i < v.size() && ch.cost + cost[v[i]] <= cap);
      chunks.push_back(ch);
    }
  }
  std::vector<int> order(chunks.size());
  std::iota(order.begin(), order.end(), 0);
  std::stable_sort(order.begin(), order.end(), [&](int x, int y) { return chunks[x].cost > chunks[y].cost; });
  std::vector<double> load(world, 0.0);
  for (int c : order) {
    int best = 0;
    for (int r = 1; r < world; ++r)
      if (load[r] < load[best]) best = r;
    load[best] += chunks[c].cost;
    for (int t = 0; t < chunks[c].count; ++t) owner[flat[chunks[c].first + t]] = best;
  }
}

double now_ms() { return std::chrono::duration<double, std::milli>(std::chrono::steady_clock::now().time_since_epoch()).count(); }

struct Phases {
  Ctx& c;
  float* ms;
  double t0;
  Phases(Ctx& ctx, float* out) : c(ctx), ms(out), t0(0)
  {
    if (ms) {
      for (int i = 0; i < 5; ++i) ms[i] = 0.f;
      c.sync();
      t0 = now_ms();
    }
  }
  void mark(int k)
  {
    if (!ms) return;
    c.sync();
    const double t = now_ms();
    ms[k] += (float)(t - t0);
    t0 = t;
  }
};

constexpr int RES_W = 22;  // per pair: 16 transform floats, confidence (double bits), contribution count, 4 stats

// One rank's part of estimateMapsTransforms.  local = this rank's block of raw clouds (device).  Returns the number of
// transforms written (every rank gets all of them).
int dist_estimate(Ctx& c, mm3d_comm* cm, int n_maps, const std::vector<CloudView>& local, const mm3d_params& p, float* out_transforms,
                  float* phase_ms)
{
  const int W = cm ? cm->world : 1, R = cm ? cm->rank : 0;
  const int M = n_maps;
  if (M == 0) return 0;
  if (M == 1) {
    const float id[16] = {1, 0, 0, 0, 0, 1, 0, 0, 0, 0, 1, 0, 0, 0, 0, 1};
    memcpy(out_transforms, id, sizeof(id));
    return 1;
  }
  const int per = block_per(M, W);
  int first, count;
  block_of(R, W, M, &first, &count);
  if ((int)local.size() != count) throw std::runtime_error("estimateMapsTransforms (multi-GPU): this rank's block holds " + std::to_string(count) + " maps");
  Phases ph(c, phase_ms);

  // ---- A: feature pipeline of the own block
  std::vector<MapFeat> f;
  compute_features(c, local, p, f, nullptr);
  const int dim = desc_dim(p);
  ph.mark(0);

  // ---- B: sizes of every map
  std::vector<int> sz((size_t)W * per * 2, 0);
  for (int m = 0; m < count; ++m) {
    sz[((size_t)R * per + m) * 2] = f[m].cloud.n;
    sz[((size_t)R * per + m) * 2 + 1] = f[m].keypoints.n;
  }
  if (W > 1) {
    DBuf<int> dsz(c, sz.size());
    dsz.upload(c, sz.data(), sz.size());
    MM_NCCL(nccl().AllGather(dsz.p + (size_t)R * per * 2, dsz.p, (size_t)per * 2, ncclInt32, cm->comm, c.stream));
    dsz.download(c, sz.data(), sz.size());
    c.sync();
  }
  std::vector<int> npt(M), nkp(M);
  for (int m = 0; m < M; ++m) {
    const int r = std::min(m / per, W - 1), l = m - r * per;
    npt[m] = sz[((size_t)r * per + l) * 2];
    nkp[m] = sz[((size_t)r * per + l) * 2 + 1];
  }

  // ---- C: exchange {cloud, keypoints, descriptors}; per map one chunk [points | keypoints | descriptors], chunks padded to
  // 256 bytes, rank r's chunks contiguous: rank r broadcasts exactly its own region.
  std::vector<size_t> off(M + 1, 0);
  for (int m = 0; m < M; ++m) {
    const size_t floats = 4 * (size_t)npt[m] + 4 * (size_t)nkp[m] + (size_t)dim * nkp[m];
    off[m + 1] = off[m] + ((floats + 63) / 64) * 64;
  }
  DBuf<float> all(c, off[M] + 64);
  for (int m = 0; m < count; ++m) {
    float* base = all.p + off[first + m];
    if (f[m].cloud.n) MM_CUDA(cudaMemcpyAsync(base, f[m].cloud.pts.p, (size_t)f[m].cloud.n * 16, cudaMemcpyDeviceToDevice, c.stream));
    if (f[m].keypoints.n) {
      MM_CUDA(cudaMemcpyAsync(base + 4 * (size_t)f[m].cloud.n, f[m].keypoints.pts.p, (size_t)f[m].keypoints.n * 16, cudaMemcpyDeviceToDevice, c.stream));
      MM_CUDA(cudaMemcpyAsync(base + 4 * (size_t)(f[m].cloud.n + f[m].keypoints.n), f[m].desc.p, (size_t)f[m].keypoints.n * dim * 4,
                              cudaMemcpyDeviceToDevice, c.stream));
    }
  }
  if (W > 1) {
    MM_NCCL(nccl().GroupStart());
    for (int r = 0; r < W; ++r) {
      int rf, rc;
      block_of(r, W, M, &rf, &rc);
      const size_t cnt = off[rf + rc] - off[rf];
      if (cnt) MM_NCCL(nccl().Broadcast(all.p + off[rf], all.p + off[rf], cnt, ncclFloat, r, cm->comm, c.stream));
    }
    MM_NCCL(nccl().GroupEnd());
  }
  f.clear();  // the views below point into `all`
  std::vector<FeatView> views(M);
  for (int m = 0; m < M; ++m) {
    const float* base = all.p + off[m];
    views[m].cloud = CloudView{(const float4*)base, npt[m]};
    views[m].keypoints = CloudView{(const float4*)(base + 4 * (size_t)npt[m]), nkp[m]};
    views[m].desc = base + 4 * (size_t)(npt[m] + nkp[m]);
  }
  ph.mark(1);

  // ---- D: the row-major pair list (map_merging.cpp:246-254), dealt out by LPT — identical on every rank
  std::vector<PairJob> pairs;
  for (int i = 0; i < M - 1; ++i)
    for (int j = i + 1; j < M; ++j)
      if (nkp[i] > 0 && nkp[j] > 0) pairs.push_back(PairJob{i, j});
  const int P = (int)pairs.size();
  std::vector<double> cost(P);
  for (int k = 0; k < P; ++k) cost[k] = pair_cost(npt[pairs[k].a], npt[pairs[k].b], nkp[pairs[k].a], nkp[pairs[k].b], dim);
  std::vector<int> owner;
  lpt_assign(pairs, cost, W, owner);
  std::vector<PairJob> mine;
  std::vector<int> mine_k;
  for (int k = 0; k < P; ++k)
    if (owner[k] == R) {
      mine.push_back(pairs[k]);
      mine_k.push_back(k);
    }

  // ---- E: register the own share
  std::vector<PairOut> po;
  register_pairs(c, views, dim, mine, p, po, nullptr);
  ph.mark(2);

  // ---- F: results into their row-major slots
  std::vector<unsigned long long> res((size_t)std::max(P, 1) * RES_W, 0ull);
  for (size_t t = 0; t < mine.size(); ++t) {
    unsigned long long* r = &res[(size_t)mine_k[t] * RES_W];
    for (int k = 0; k < 16; ++k) {
      uint32_t b;
      memcpy(&b, &po[t].T[k], 4);
      r[k] = b;
    }
    memcpy(&r[16], &po[t].confidence, 8);
    r[17] = 1;
    r[18] = (unsigned)po[t].n_corr;
    r[19] = (unsigned)po[t].n_inliers;
    r[20] = (unsigned)po[t].icp_iterations;
    r[21] = (unsigned)po[t].icp_converged;
  }
  if (W > 1 && P > 0) {
    DBuf<unsigned long long> dres(c, res.size());
    dres.upload(c, res.data(), res.size());
    MM_NCCL(nccl().AllReduce(dres.p, dres.p, res.size(), ncclUint64, ncclSum, cm->comm, c.stream));
    dres.download(c, res.data(), res.size());
    c.sync();
  }
  ph.mark(3);

  // ---- G: pose graph (host), on every rank
  std::vector<HostEstimate> est(P);
  for (int k = 0; k < P; ++k) {
    const unsigned long long* r = &res[(size_t)k * RES_W];
    if (r[17] != 1) throw std::runtime_error("estimateMapsTransforms (multi-GPU): pair " + std::to_string(k) + " was registered " + std::to_string(r[17]) + " times");
    est[k].source_idx = (size_t)pairs[k].a;
    est[k].target_idx = (size_t)pairs[k].b;
    for (int q = 0; q < 16; ++q) {
      const uint32_t b = (uint32_t)r[q];
      memcpy(&est[k].T[q], &b, 4);
    }
    memcpy(&est[k].confidence, &r[16], 8);
  }
  std::vector<std::vector<float>> g = compute_global_transforms(est, p.confidence_threshold, nullptr, nullptr, nullptr, nullptr);
  for (size_t i = 0; i < g.size(); ++i) to_colmajor(g[i].data(), out_transforms + 16 * i);
  ph.mark(4);
  return (int)g.size();
}

// Balanced key-range splitters from the all-reduced bucket histogram: splitters[r] <= bucket < splitters[r + 1] goes to rank r.
std::vector<int> choose_splitters(const std::vector<unsigned long long>& hist, int world)
{
  const int nb = (int)hist.size();
  std::vector<unsigned long long> cum(nb);
  unsigned long long run = 0;
  for (int i = 0; i < nb; ++i) { run += hist[i]; cum[i] = run; }
  const unsigned long long total = run;
  std::vector<int> sp(world + 1, 0);
  sp[world] = nb;
  for (int r = 1; r < world; ++r) {
    const unsigned long long target = total * (unsigned long long)r / (unsigned long long)world;
    int pos = (int)(std::lower_bound(cum.begin(), cum.end(), target) - cum.begin());
    pos += total ? 1 : 0;
    sp[r] = std::min(std::max(pos, sp[r - 1]), nb);
  }
  return sp;
}

// One rank's part of composeMaps: local clouds already on the device.  Returns this rank's slice of the composed map on the
// host (host_out_alloc, records in out_layout); the slices concatenated in rank order are the reference's output bit for bit.
void dist_compose(Ctx& c, mm3d_comm* cm, const std::vector<CloudView>& local, const std::vector<const float*>& transforms_rowmajor,
                  double resolution, const mm3d_layout& out_layout, void** out, uint64_t* n_out)
{
  const int W = cm ? cm->world : 1;
  constexpr int NB = 4096;
  *out = nullptr;
  *n_out = 0;
  // MM3D_HOST_TRACE=1: host wall clock between the phases (each ends in a synchronisation of its own)
  const bool trace = host_prof().on;
  double t_prev = trace ? now_ms() : 0.0;
  auto mark = [&](const char* what) {
    if (!trace) return;
    const double t = now_ms();
    fprintf(stderr, "[mm3d compose] %s %.2f ms\n", what, t - t_prev);
    t_prev = t;
  };
  DCloud cat;
  transform_concat(c, local, transforms_rowmajor, cat);
  float bbox[6];
  compose_bbox(c, cat, bbox);
  mark("transform + concatenate + bounding box");
  unsigned long long total = (unsigned long long)cat.n;
  if (W > 1) {
    // min over ranks of (lo, -hi) and the point count
    float h[6] = {bbox[0], bbox[1], bbox[2], -bbox[3], -bbox[4], -bbox[5]};
    DBuf<float> d(c, 6);
    d.upload(c, h, 6);
    DBuf<unsigned long long> dt(c, 1);
    dt.upload(c, &total, 1);
    MM_NCCL(nccl().GroupStart());
    MM_NCCL(nccl().AllReduce(d.p, d.p, 6, ncclFloat, ncclMin, cm->comm, c.stream));
    MM_NCCL(nccl().AllReduce(dt.p, dt.p, 1, ncclUint64, ncclSum, cm->comm, c.stream));
    MM_NCCL(nccl().GroupEnd());
    d.download(c, h, 6);
    dt.download(c, &total, 1);
    c.sync();
    for (int k = 0; k < 3; ++k) { bbox[k] = h[k]; bbox[3 + k] = -h[3 + k]; }
  }
  auto to_host = [&](const float4* p, size_t n) {
    *out = download_records(c, p, n, out_layout);
    *n_out = n;
    c.sync();
    mark("copy to the host");
  };
  if (total == 0) {
    to_host(nullptr, 0);
    return;
  }
  const KeyGeomHost g = compose_geometry(bbox, resolution, NB);
  if (g.passthrough) {  // pcl::VoxelGrid's overflow guard: the composed map is the plain concatenation, rank order = map order
    to_host(cat.pts.p, (size_t)cat.n);
    return;
  }
  if (W == 1) {
    std::vector<DCloud> res;
    voxel_downsample_batch(c, {cat.view()}, (float)resolution, res, nullptr);
    if (trace) c.sync();
    mark("voxel grid");
    to_host(res[0].pts.p, (size_t)res[0].n);
    return;
  }
  std::vector<unsigned long long> hist(NB);
  compose_histogram(c, cat, g, NB, hist.data());
  {
    DBuf<unsigned long long> dh(c, NB);
    dh.upload(c, hist.data(), NB);
    MM_NCCL(nccl().AllReduce(dh.p, dh.p, NB, ncclUint64, ncclSum, cm->comm, c.stream));
    dh.download(c, hist.data(), NB);
    c.sync();
  }
  const std::vector<int> sp = choose_splitters(hist, W);
  DBuf<float4> send(c, (size_t)cat.n + 1);
  std::vector<unsigned long long> cnt(W, 0);
  compose_partition(c, cat, g, NB, sp, W, cnt.data(), send.p);
  // counts matrix: row r = what rank r sends to every rank
  std::vector<unsigned long long> mat((size_t)W * W, 0);
  {
    DBuf<unsigned long long> dm(c, mat.size());
    MM_CUDA(cudaMemcpyAsync(dm.p + (size_t)cm->rank * W, cnt.data(), W * 8, cudaMemcpyHostToDevice, c.stream));
    MM_NCCL(nccl().AllGather(dm.p + (size_t)cm->rank * W, dm.p, W, ncclUint64, cm->comm, c.stream));
    dm.download(c, mat.data(), mat.size());
    c.sync();
  }
  size_t recv_total = 0;
  for (int r = 0; r < W; ++r) recv_total += (size_t)mat[(size_t)r * W + cm->rank];
  DBuf<float4> recv(c, recv_total + 1);
  MM_NCCL(nccl().GroupStart());
  size_t so = 0, ro = 0;
  for (int r = 0; r < W; ++r) {
    const size_t ns = (size_t)cnt[r], nr = (size_t)mat[(size_t)r * W + cm->rank];
    if (ns) MM_NCCL(nccl().Send(send.p + so, ns * 4, ncclFloat, r, cm->comm, c.stream));
    if (nr) MM_NCCL(nccl().Recv(recv.p + ro, nr * 4, ncclFloat, r, cm->comm, c.stream));
    so += ns;
    ro += nr;
  }
  MM_NCCL(nccl().GroupEnd());
  std::vector<DCloud> res;
  voxel_downsample_batch(c, {CloudView{recv.p, (int)recv_total}}, (float)resolution, res, nullptr);
  to_host(res[0].pts.p, (size_t)res[0].n);
}

// composeMaps' skip rules (map_merging.cpp:293-295): zero transforms and empty clouds are left out
bool skip_map(const float* colmajor, const void* cloud, uint64_t n, float* rowmajor)
{
  from_colmajor(colmajor, rowmajor);
  bool zero = true;  // Eigen isZero(): every |a_ij| <= 1e-5
  for (int k = 0; k < 16; ++k)
    if (!(std::fabs(rowmajor[k]) <= 1e-5f)) zero = false;
  return zero || !cloud || n == 0;
}

// run fn(rank) on one host thread per device of the team; the first error wins
template <typename F>
void team_run(mm3d_ctx* master, F fn)
{
  mm3d_team& t = *master->team;
  const int n = (int)t.comms.size();
  std::vector<std::string> errors(n);
  std::vector<int> kinds(n, 0);
  std::vector<std::thread> th;
  for (int r = 0; r < n; ++r)
    th.emplace_back([&, r] {
      mm3d_ctx* h = r == 0 ? master : t.subs[r - 1];
      try {
        MM_CUDA(cudaSetDevice(h->c.device));
        fn(r, h->c, &t.comms[r]);
      } catch (const UnsupportedError& e) {
        errors[r] = e.what();
        kinds[r] = 2;
      } catch (const CudaError& e) {
        errors[r] = e.what();
        kinds[r] = 1;
        cudaGetLastError();
      } catch (const std::exception& e) {
        errors[r] = e.what();
        kinds[r] = 3;
      }
    });
  for (std::thread& x : th) x.join();
  for (int r = 0; r < n; ++r) {
    if (kinds[r] == 1) throw CudaError("device " + std::to_string(r) + ": " + errors[r]);
    if (kinds[r] == 2) throw UnsupportedError(errors[r]);
    if (kinds[r] == 3) throw std::runtime_error("device " + std::to_string(r) + ": " + errors[r]);
  }
}

}  // namespace

namespace mm3d {

int team_size(const mm3d_ctx* ctx) { return ctx && ctx->team ? (int)ctx->team->comms.size() : 1; }

// estimateMapsTransforms from host buffers over the devices of a mm3d_create_multi context; each device uploads its own block
int team_estimate(mm3d_ctx* master, int n_maps, const void* const* clouds, const uint64_t* n_points, const mm3d_layout& layout,
                  const mm3d_params& p, float* out_transforms)
{
  int n_out = 0;
  const int W = team_size(master);
  std::vector<std::vector<float>> outs(W, std::vector<float>((size_t)std::max(n_maps, 1) * 16));
  std::vector<int> counts(W, 0);
  team_run(master, [&](int r, Ctx& c, mm3d_comm* cm) {
    int first, count;
    block_of(r, W, n_maps, &first, &count);
    std::vector<DCloud> d = upload_clouds(c, std::vector<const void*>(clouds + first, clouds + first + count),
                                          std::vector<uint64_t>(n_points + first, n_points + first + count), layout);
    std::vector<CloudView> v(count);
    for (int m = 0; m < count; ++m) v[m] = d[m].view();
    counts[r] = dist_estimate(c, cm, n_maps, v, p, outs[r].data(), nullptr);
    c.sync();
  });
  n_out = counts[0];
  memcpy(out_transforms, outs[0].data(), (size_t)n_out * 16 * sizeof(float));
  return n_out;
}

// composeMaps from host buffers over the devices of a mm3d_create_multi context
void team_compose(mm3d_ctx* master, int n_maps, const void* const* clouds, const uint64_t* n_points, const mm3d_layout& in_layout,
                  const float* transforms, double resolution, const mm3d_layout& out_layout, void** out, uint64_t* n_out)
{
  const int W = team_size(master);
  std::vector<void*> parts(W, nullptr);
  std::vector<uint64_t> sizes(W, 0);
  try {
    team_run(master, [&](int r, Ctx& c, mm3d_comm* cm) {
      int first, count;
      block_of(r, W, n_maps, &first, &count);
      std::vector<const void*> src;
      std::vector<uint64_t> cnt;
      std::vector<std::vector<float>> tr;
      for (int m = first; m < first + count; ++m) {
        float rm[16];
        if (skip_map(transforms + 16 * m, clouds[m], n_points[m], rm)) continue;
        src.push_back(clouds[m]);
        cnt.push_back(n_points[m]);
        tr.emplace_back(rm, rm + 16);
      }
      std::vector<DCloud> d = upload_clouds(c, src, cnt, in_layout);
      std::vector<CloudView> v;
      std::vector<const float*> tp;
      for (size_t i = 0; i < d.size(); ++i) {
        v.push_back(d[i].view());
        tp.push_back(tr[i].data());
      }
      dist_compose(c, cm, v, tp, resolution, out_layout, &parts[r], &sizes[r]);
    });
  } catch (...) {
    for (void* p : parts) host_out_free(p);
    throw;
  }
  const size_t step = out_layout.point_step;
  uint64_t total = 0;
  for (uint64_t s : sizes) total += s;
  *out = host_out_alloc(std::max<uint64_t>(total, 1) * step);
  uint64_t o = 0;
  for (int r = 0; r < W; ++r) {
    if (sizes[r]) memcpy((unsigned char*)*out + o * step, parts[r], sizes[r] * step);
    o += sizes[r];
    host_out_free(parts[r]);
  }
  *n_out = total;
}

}  // namespace mm3d

extern "C" {

int mm3d_comm_id(void* id)
{
  if (!id) return MM3D_ERR_ARG;
  try {
    static_assert(sizeof(ncclUniqueId) <= MM3D_COMM_ID_BYTES, "ncclUniqueId does not fit");
    ncclUniqueId u;
    memset(&u, 0, sizeof(u));
    const ncclResult_t r = nccl().GetUniqueId(&u);
    if (r != ncclSuccess) return MM3D_ERR_CUDA;
    memset(id, 0, MM3D_COMM_ID_BYTES);
    memcpy(id, &u, sizeof(u));
  } catch (const UnsupportedError&) {
    return MM3D_ERR_UNSUPPORTED;
  } catch (const std::exception&) {
    return MM3D_ERR;
  }
  return MM3D_OK;
}

#define MMD_TRY(ctx) \
  if (!(ctx)) return MM3D_ERR_ARG; \
  Ctx& c = (ctx)->c; \
  try { \
    MM_CUDA(cudaSetDevice(c.device));
#define MMD_CATCH \
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

int mm3d_comm_create(mm3d_ctx* ctx, int rank, int world, const void* id, mm3d_comm** comm)
{
  if (!comm || !id || world < 1 || rank < 0 || rank >= world) return MM3D_ERR_ARG;
  *comm = nullptr;
  MMD_TRY(ctx)
  std::unique_ptr<mm3d_comm> h(new mm3d_comm);
  h->rank = rank;
  h->world = world;
  ncclUniqueId u;
  memcpy(&u, id, sizeof(u));
  MM_NCCL(nccl().CommInitRank(&h->comm, world, u, rank));
  *comm = h.release();
  MMD_CATCH
}

void mm3d_comm_destroy(mm3d_comm* comm)
{
  if (!comm) return;
  if (comm->comm) nccl().CommDestroy(comm->comm);
  delete comm;
}

int mm3d_comm_rank(const mm3d_comm* comm) { return comm ? comm->rank : 0; }
int mm3d_comm_size(const mm3d_comm* comm) { return comm ? comm->world : 1; }

int mm3d_dist_block(int rank, int world, int n_maps, int* first, int* count)
{
  if (world < 1 || rank < 0 || rank >= world || n_maps < 0 || !first || !count) return MM3D_ERR_ARG;
  block_of(rank, world, n_maps, first, count);
  return MM3D_OK;
}

int mm3d_dist_plan(int n_maps, const int32_t* n_points, const int32_t* n_keypoints, int dim, int world, int32_t* pairs, int32_t* owner,
                   int* n_pairs)
{
  if (n_maps < 0 || world < 1 || !n_points || !n_keypoints || !n_pairs) return MM3D_ERR_ARG;
  std::vector<double> cost;
  std::vector<PairJob> pj;
  int P = 0;
  for (int i = 0; i < n_maps - 1; ++i)
    for (int j = i + 1; j < n_maps; ++j)
      if (n_keypoints[i] > 0 && n_keypoints[j] > 0) {
        if (pairs) { pairs[2 * P] = i; pairs[2 * P + 1] = j; }
        pj.push_back(PairJob{i, j});
        cost.push_back(pair_cost(n_points[i], n_points[j], n_keypoints[i], n_keypoints[j], dim));
        ++P;
      }
  std::vector<int> own;
  lpt_assign(pj, cost, world, own);
  if (owner)
    for (int k = 0; k < P; ++k) owner[k] = own[k];
  *n_pairs = P;
  return MM3D_OK;
}

int mm3d_estimate_maps_transforms_dist(mm3d_ctx* ctx, mm3d_comm* comm, int n_maps, const float* const* clouds, const uint64_t* n_points,
                                       const mm3d_params* params, float* out_transforms, int* n_out)
{
  if (!n_out || !params || n_maps < 0) return MM3D_ERR_ARG;
  *n_out = 0;
  MMD_TRY(ctx)
  int first, count;
  block_of(comm ? comm->rank : 0, comm ? comm->world : 1, n_maps, &first, &count);
  std::vector<DCloud> d(count);
  std::vector<CloudView> v(count);
  for (int m = 0; m < count; ++m) {
    d[m] = upload_cloud(c, clouds[first + m], clouds[first + m] ? n_points[first + m] : 0);
    v[m] = d[m].view();
  }
  *n_out = dist_estimate(c, comm, n_maps, v, *params, out_transforms, nullptr);
  c.sync();
  MMD_CATCH
}

int mm3d_estimate_resident_dist(mm3d_ctx* ctx, mm3d_comm* comm, int n_maps, const mm3d_maps* local_maps, const mm3d_params* params,
                                float* out_transforms, int* n_out, float* phase_ms)
{
  if (!n_out || !params || !local_maps || n_maps < 0) return MM3D_ERR_ARG;
  *n_out = 0;
  MMD_TRY(ctx)
  std::vector<CloudView> v(local_maps->clouds.size());
  for (size_t m = 0; m < v.size(); ++m) v[m] = local_maps->clouds[m].view();
  *n_out = dist_estimate(c, comm, n_maps, v, *params, out_transforms, phase_ms);
  c.sync();
  MMD_CATCH
}

int mm3d_compose_maps_dist(mm3d_ctx* ctx, mm3d_comm* comm, int n_local, const float* const* clouds, const uint64_t* n_points,
                           int n_transforms, const float* transforms, double resolution, float** out, uint64_t* n_out)
{
  if (!out || !n_out || n_local < 0) return MM3D_ERR_ARG;
  *out = nullptr;
  *n_out = 0;
  if (n_local != n_transforms) {
    if (ctx) ctx->c.err = "composeMaps: clouds and transforms size must be the same.";
    return MM3D_ERR_ARG;
  }
  MMD_TRY(ctx)
  std::vector<DCloud> d;
  std::vector<std::vector<float>> tr;
  for (int m = 0; m < n_local; ++m) {
    float rm[16];
    if (skip_map(transforms + 16 * m, clouds[m], n_points[m], rm)) continue;
    d.push_back(upload_cloud(c, clouds[m], n_points[m]));
    tr.emplace_back(rm, rm + 16);
  }
  std::vector<CloudView> v;
  std::vector<const float*> tp;
  for (size_t i = 0; i < d.size(); ++i) {
    v.push_back(d[i].view());
    tp.push_back(tr[i].data());
  }
  dist_compose(c, comm, v, tp, resolution, kPackedLayout, (void**)out, n_out);
  MMD_CATCH
}

int mm3d_compose_resident_dist(mm3d_ctx* ctx, mm3d_comm* comm, const mm3d_maps* local_maps, int n_transforms, const float* transforms,
                               double resolution, float** out, uint64_t* n_out)
{
  if (!out || !n_out || !local_maps) return MM3D_ERR_ARG;
  *out = nullptr;
  *n_out = 0;
  if ((int)local_maps->clouds.size() != n_transforms) {
    if (ctx) ctx->c.err = "composeMaps: clouds and transforms size must be the same.";
    return MM3D_ERR_ARG;
  }
  MMD_TRY(ctx)
  std::vector<std::vector<float>> tr;
  std::vector<CloudView> v;
  std::vector<const float*> tp;
  float dummy = 0.f;
  for (int m = 0; m < n_transforms; ++m) {
    float rm[16];
    if (skip_map(transforms + 16 * m, &dummy, (uint64_t)local_maps->clouds[m].n, rm)) continue;
    v.push_back(local_maps->clouds[m].view());
    tr.emplace_back(rm, rm + 16);
  }
  for (size_t i = 0; i < tr.size(); ++i) tp.push_back(tr[i].data());
  dist_compose(c, comm, v, tp, resolution, kPackedLayout, (void**)out, n_out);
  MMD_CATCH
}

int mm3d_create_multi(mm3d_ctx** ctx, const int* devices, int n_devices)
{
  if (!ctx) return MM3D_ERR_ARG;
  *ctx = nullptr;
  int count = 0;
  if (cudaGetDeviceCount(&count) != cudaSuccess || count == 0) {
    cudaGetLastError();
    return MM3D_ERR_CUDA;
  }
  std::vector<int> dev;
  if (!devices || n_devices <= 0) {
    for (int d = 0; d < count; ++d) dev.push_back(d);
  } else {
    dev.assign(devices, devices + n_devices);
  }
  for (size_t i = 0; i < dev.size(); ++i) {
    if (dev[i] < 0 || dev[i] >= count) return MM3D_ERR_ARG;
    for (size_t k = 0; k < i; ++k)
      if (dev[k] == dev[i]) return MM3D_ERR_ARG;
  }
  mm3d_ctx* master = nullptr;
  int rc = mm3d_create(&master, dev[0], nullptr);
  if (rc != MM3D_OK) return rc;
  if (dev.size() == 1) {
    *ctx = master;
    return MM3D_OK;
  }
  try {
    std::unique_ptr<mm3d_team> t(new mm3d_team);
    for (size_t i = 1; i < dev.size(); ++i) {
      mm3d_ctx* s = nullptr;
      rc = mm3d_create(&s, dev[i], nullptr);
      if (rc != MM3D_OK) {
        t.reset();
        mm3d_destroy(master);
        return rc;
      }
      t->subs.push_back(s);
    }
    std::vector<ncclComm_t> comms(dev.size());
    MM_NCCL(nccl().CommInitAll(comms.data(), (int)dev.size(), dev.data()));
    t->comms.resize(dev.size());
    for (size_t i = 0; i < dev.size(); ++i) {
      t->comms[i].comm = comms[i];
      t->comms[i].rank = (int)i;
      t->comms[i].world = (int)dev.size();
    }
    master->team = std::move(t);
  } catch (const UnsupportedError&) {
    mm3d_destroy(master);
    return MM3D_ERR_UNSUPPORTED;
  } catch (const std::exception&) {
    cudaGetLastError();
    mm3d_destroy(master);
    return MM3D_ERR_CUDA;
  }
  cudaSetDevice(dev[0]);
  *ctx = master;
  return MM3D_OK;
}

int mm3d_device_count(const mm3d_ctx* ctx) { return team_size(ctx); }

}  // extern "C"
