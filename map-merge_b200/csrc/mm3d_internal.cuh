// mm3d_internal.cuh — shared declarations for the sm_100a registration library.
//
// Design (see DESIGN.md): every per-map stage runs ONCE for all maps in a 2-D
// launch (blockIdx.y = map, or = pair in the registration loop), all work is
// queued on one stream, and the host synchronises only where a stage's output
// size is needed to size the next allocation.  Neighbourhood queries go through
// a "voxel-row" index: the clouds on this path are voxel-grid outputs, i.e.
// already sorted by (z, y, x) voxel key, so a dense table of row-bucket start
// offsets turns a radius query into a walk over contiguous, ascending-index
// runs — which is also the canonical summation order the parity checker uses.
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>

#include <memory>
#include <mutex>
#include <stdexcept>
#include <string>
#include <unordered_map>
#include <vector>

#include "exact_math.h"

namespace mm3d {

// Typed errors: the C ABI maps them to MM3D_ERR_CUDA / MM3D_ERR_UNSUPPORTED (anything else is MM3D_ERR).
struct CudaError : std::runtime_error {
  using std::runtime_error::runtime_error;
};
struct UnsupportedError : std::runtime_error {
  using std::runtime_error::runtime_error;
};

#define MM_CUDA(expr)                                                                                   \
  do {                                                                                                  \
    cudaError_t _e = (expr);                                                                            \
    if (_e != cudaSuccess)                                                                              \
      throw mm3d::CudaError(std::string("CUDA error: ") + cudaGetErrorString(_e) + " at " __FILE__ ":" + \
                            std::to_string(__LINE__) + " (" #expr ")");                                 \
  } while (0)

// Optional per-kernel timing: one CUDA event pair around every launch, recorded on
// the launching stream and resolved when profiling ends (no extra synchronisation).
struct KernelSample {
  const char* name;
  double bytes;  // algorithmic bytes of this launch (inputs read once + outputs written once), 0 = not annotated
  cudaEvent_t e0, e1;
};

// MM3D_HOST_TRACE=1: host time spent inside the CUDA runtime calls of the path (where does the host wait?)
struct HostProf {
  bool on = false;
  double alloc_ms = 0, free_ms = 0, sync_ms = 0, copy_ms = 0;
  long n_alloc = 0, n_free = 0, n_sync = 0, n_copy = 0;
  size_t alloc_bytes = 0;
};
HostProf& host_prof();
double host_now_ms();

// Host memory for outputs returned through the C ABI (released by mm3d_free).  Large outputs (composed maps: tens of MB) come
// from a process-wide cache of PINNED blocks: the device-to-host copy runs at PCIe speed instead of being staged through
// the driver's bounce buffers into freshly mapped pages (config 5: 75 MB per call, 36 ms -> 1.4 ms).  Small ones are plain malloc.
void* host_out_alloc(size_t bytes);
void host_out_free(void* p);

// Device-memory block cache of one context.  The path allocates and frees thousands of stage buffers per step (c3: ~4300
// calls, ~9 GB); handing them to cudaMallocAsync / cudaFreeAsync made the step time erratic — the driver pool re-creates
// multi-GB physical chunks whenever fragmentation defeats reuse (measured: 5 .. 560 ms per step inside cudaMallocAsync).
// Freed blocks therefore return to size-class free lists here (8 classes per octave: <= 12.5 % slack) and are handed out
// again without a driver call.  Everything of a context runs on ONE stream, so reuse after free is ordered by the stream,
// exactly like the driver's stream-ordered pool.  Buffers hold a shared reference: blocks that outlive their context are
// released with the last reference.
struct BlockCache {
  std::mutex mu;
  std::unordered_map<size_t, std::vector<void*>> free_blocks;
  int device = 0;
  cudaStream_t stream = nullptr;
  size_t held_bytes = 0;
  static size_t size_class(size_t bytes)
  {
    if (bytes <= 4096) return (bytes + 255) & ~(size_t)255;
    int lg = 0;
    while (((size_t)1 << (lg + 1)) <= bytes) ++lg;
    const size_t step = (size_t)1 << (lg - 3);
    return (bytes + step - 1) & ~(step - 1);
  }
  void* get(size_t cls)
  {
    {
      std::lock_guard<std::mutex> lk(mu);
      auto it = free_blocks.find(cls);
      if (it != free_blocks.end() && !it->second.empty()) {
        void* p = it->second.back();
        it->second.pop_back();
        held_bytes -= cls;
        return p;
      }
    }
    void* p = nullptr;
    cudaError_t e = cudaMallocAsync(&p, cls, stream);
    if (e != cudaSuccess) {  // out of memory: give the cached blocks back and retry once
      cudaGetLastError();
      trim();
      e = cudaMallocAsync(&p, cls, stream);
    }
    if (e != cudaSuccess)
      throw CudaError(std::string("CUDA error: ") + cudaGetErrorString(e) + " allocating " + std::to_string(cls) + " bytes");
    return p;
  }
  void put(void* p, size_t cls)
  {
    std::lock_guard<std::mutex> lk(mu);
    free_blocks[cls].push_back(p);
    held_bytes += cls;
  }
  void trim()
  {
    std::lock_guard<std::mutex> lk(mu);
    for (auto& kv : free_blocks)
      for (void* p : kv.second) cudaFreeAsync(p, stream);
    free_blocks.clear();
    held_bytes = 0;
  }
  ~BlockCache()
  {
    // the context (and its stream) may be gone: plain cudaFree, which synchronises the device
    int cur = 0;
    cudaGetDevice(&cur);
    cudaSetDevice(device);
    for (auto& kv : free_blocks)
      for (void* p : kv.second) cudaFree(p);
    cudaSetDevice(cur);
  }
};

struct StagingRing;  // layout.cu: pinned slots for records in a caller's layout

struct Ctx {
  int device = 0;
  std::shared_ptr<BlockCache> cache = std::make_shared<BlockCache>();
  cudaStream_t stream = nullptr;
  bool own_stream = false;
  std::string err;
  long long launches = 0;  // kernels launched through this context (bench.py's gpu_launches)
  bool profiling = false;
  double next_bytes = 0.0;
  unsigned long long* knn_stats = nullptr;  // device: rows, rows that fell back to the exact scan, candidates re-ranked
  std::vector<KernelSample> samples;
  std::vector<cudaEvent_t> event_pool;
  StagingRing* staging = nullptr;  // created by the first staged upload, freed by mm3d_destroy (staging_release)
  void sync()
  {
    HostProf& hp = host_prof();
    if (!hp.on) {
      MM_CUDA(cudaStreamSynchronize(stream));
      return;
    }
    const double t0 = host_now_ms();
    MM_CUDA(cudaStreamSynchronize(stream));
    hp.sync_ms += host_now_ms() - t0;
    ++hp.n_sync;
  }
  cudaEvent_t get_event()
  {
    cudaEvent_t e;
    if (!event_pool.empty()) {
      e = event_pool.back();
      event_pool.pop_back();
    } else {
      MM_CUDA(cudaEventCreate(&e));
    }
    return e;
  }
  void before_launch(const char* name)
  {
    ++launches;
    if (!profiling) return;
    KernelSample s;
    s.name = name;
    s.bytes = next_bytes;
    s.e0 = get_event();
    s.e1 = get_event();
    MM_CUDA(cudaEventRecord(s.e0, stream));
    samples.push_back(s);
  }
  void after_launch()
  {
    next_bytes = 0.0;
    if (!profiling) return;
    MM_CUDA(cudaEventRecord(samples.back().e1, stream));
  }
};

#define MM_LAUNCH(ctx, kernel, grid, block, smem, ...)                 \
  do {                                                                 \
    (ctx).before_launch(#kernel);                                      \
    kernel<<<(grid), (block), (smem), (ctx).stream>>>(__VA_ARGS__);    \
    (ctx).after_launch();                                              \
    MM_CUDA(cudaGetLastError());                                       \
  } while (0)

// annotate the next launch with its algorithmic byte count
#define MM_BYTES(ctx, b) ((ctx).next_bytes = (double)(b))

// Stream-ordered device buffer (blocks come from the context's BlockCache).
template <typename T>
struct DBuf {
  T* p = nullptr;
  size_t n = 0;
  size_t cls = 0;                     // size class of the block behind p
  std::shared_ptr<BlockCache> cache;  // where the block returns to
  DBuf() {}
  DBuf(Ctx& c, size_t count) { alloc(c, count); }
  DBuf(const DBuf&) = delete;
  DBuf& operator=(const DBuf&) = delete;
  DBuf(DBuf&& o) noexcept : p(o.p), n(o.n), cls(o.cls), cache(std::move(o.cache)) { o.p = nullptr; o.n = 0; }
  DBuf& operator=(DBuf&& o) noexcept
  {
    if (this != &o) {
      release();
      p = o.p; n = o.n; cls = o.cls; cache = std::move(o.cache);
      o.p = nullptr; o.n = 0;
    }
    return *this;
  }
  ~DBuf() { release(); }
  void alloc(Ctx& c, size_t count)
  {
    release();
    n = count;
    if (!count) return;
    cache = c.cache;
    cls = BlockCache::size_class(count * sizeof(T));
    HostProf& hp = host_prof();
    const double t0 = hp.on ? host_now_ms() : 0.0;
    p = (T*)cache->get(cls);
    if (hp.on) {
      hp.alloc_ms += host_now_ms() - t0;
      ++hp.n_alloc;
      hp.alloc_bytes += cls;
    }
  }
  void release()
  {
    if (p && cache) cache->put(p, cls);
    p = nullptr;
    n = 0;
    cache.reset();
  }
  void zero(Ctx& c) { if (n) MM_CUDA(cudaMemsetAsync(p, 0, n * sizeof(T), c.stream)); }
  void upload(Ctx& c, const T* h, size_t count)
  {
    if (!count) return;
    HostProf& hp = host_prof();
    const double t0 = hp.on ? host_now_ms() : 0.0;
    MM_CUDA(cudaMemcpyAsync(p, h, count * sizeof(T), cudaMemcpyHostToDevice, c.stream));
    if (hp.on) { hp.copy_ms += host_now_ms() - t0; ++hp.n_copy; }
  }
  void download(Ctx& c, T* h, size_t count) const
  {
    if (!count) return;
    HostProf& hp = host_prof();
    const double t0 = hp.on ? host_now_ms() : 0.0;
    MM_CUDA(cudaMemcpyAsync(h, p, count * sizeof(T), cudaMemcpyDeviceToHost, c.stream));
    if (hp.on) { hp.copy_ms += host_now_ms() - t0; ++hp.n_copy; }
  }
};

template <typename T>
inline DBuf<T> to_device(Ctx& c, const std::vector<T>& v)
{
  DBuf<T> b(c, v.size());
  b.upload(c, v.data(), v.size());
  return b;
}

struct Seg {  // one map's slice of a concatenated array
  int off;
  int n;
};

struct CloudView {
  const float4* pts;
  int n;
};

// Voxel-grid geometry of one cloud (pcl::VoxelGrid's min_b_/div_b_).
struct VoxGeom {
  int min_b[3];
  int div_b[3];
  int passthrough;  // overflow guard hit: output = input
  int nbits;        // bits needed for a voxel key
  int nonfinite;    // points with a NaN / Inf coordinate (left out of the box; the voxel grid drops them)
};

// Neighbour index over one cloud.
struct GridView {
  const float4* pts;      // points in cell order (the cloud itself when orig == nullptr)
  const int* orig;        // original index of each slot, or nullptr = identity
  const int* cell_start;  // ncell + 1 entries
  int n;
  float inv_leaf;
  float leaf;
  int min_b[3];
  int div_v[3];
  int shift[3];
  int dim[3];
};

struct DIndex {
  GridView v;
  DBuf<int> cell_start;
  DBuf<float4> pts_sorted;
  DBuf<int> orig;
};

__host__ __device__ __forceinline__ int floor_to_int(float v) { return (int)floorf(v); }

// ---------------------------------------------------------------------------
// Device-side neighbourhood walks.
// ---------------------------------------------------------------------------
#if defined(__CUDACC__)

// Visit every point with d^2 < r2, in ascending (cell z, cell y, cell x, slot)
// order — ascending point index for a voxel-sorted cloud indexed with
// shift y = z = 0.  rv = ceil(r / leaf) + 1 voxels.  Lanes without a query pass live = false.
// (A warp-collective variant that walks the union of the lanes' windows in absolute row coordinates was
// measured on B200 and is slower: +20 % on the dense per-point kernels, 2-4x on the sparse keypoint queries.)
template <typename F>
__device__ __forceinline__ void for_each_in_radius(const GridView& g, bool live, float qx, float qy, float qz, float r2, int rv, F f)
{
  if (!live) return;
  const int vx = floor_to_int(qx * g.inv_leaf) - g.min_b[0];
  const int vy = floor_to_int(qy * g.inv_leaf) - g.min_b[1];
  const int vz = floor_to_int(qz * g.inv_leaf) - g.min_b[2];
  int zlo = vz - rv, zhi = vz + rv, ylo = vy - rv, yhi = vy + rv;
  if (zhi < 0 || yhi < 0 || vx + rv < 0 || zlo >= g.div_v[2] || ylo >= g.div_v[1] || vx - rv >= g.div_v[0]) return;
  zlo = max(zlo, 0) >> g.shift[2];
  zhi = min(zhi, g.div_v[2] - 1) >> g.shift[2];
  ylo = max(ylo, 0) >> g.shift[1];
  yhi = min(yhi, g.div_v[1] - 1) >> g.shift[1];
  const float r2v = r2 * g.inv_leaf * g.inv_leaf;  // radius^2 in voxel units (pruning only)
  for (int cz = zlo; cz <= zhi; ++cz) {
    const int z0 = cz << g.shift[2], z1 = z0 + (1 << g.shift[2]) - 1;
    const int dz = max(max(z0 - vz, vz - z1), 0);
    const float fz = (float)max(dz - 1, 0);
    for (int cy = ylo; cy <= yhi; ++cy) {
      const int y0 = cy << g.shift[1], y1 = y0 + (1 << g.shift[1]) - 1;
      const int dy = max(max(y0 - vy, vy - y1), 0);
      const float fy = (float)max(dy - 1, 0);
      const float rem = r2v - fz * fz - fy * fy;
      if (rem < 0.0f) continue;
      const int rx = (int)sqrtf(rem) + 2;
      int xlo = vx - rx, xhi = vx + rx;
      if (xhi < 0 || xlo >= g.div_v[0]) continue;
      xlo = max(xlo, 0) >> g.shift[0];
      xhi = min(xhi, g.div_v[0] - 1) >> g.shift[0];
      const int base = (cz * g.dim[1] + cy) * g.dim[0];
      const int s = g.cell_start[base + xlo], e = g.cell_start[base + xhi + 1];
      for (int k = s; k < e; ++k) {
        const float4 p = g.pts[k];
        const float d2 = em::dist2_3(qx, qy, qz, p.x, p.y, p.z);
        if (d2 < r2) f(k, p, d2);
      }
    }
  }
}

// Warp-cooperative radius query: the 32 lanes of a warp serve ONE query (all lanes pass the same arguments).
// Lanes look the (z, y) rows of the window up in parallel (32 rows per round), the rows' runs are flattened with a
// warp scan so that 32 consecutive candidates are tested per step, and the candidates that pass d^2 < r2 are
// compacted (in ascending index order) through a small shared-memory queue, so `visit` always runs with full warps.
//   visit(slot)           called by every lane that has a passing candidate `slot` (dense: lanes 0..m-1)
//   returns the number of candidates that passed
// queue: 64 ints of shared memory owned by this warp.
// ALL = true: visit is always called by all 32 lanes (slot = -1 on the lanes past the end of the last batch), so it may use
// warp collectives.
template <bool ALL = false, typename F>
__device__ __forceinline__ int warp_radius_query(const GridView& g, float qx, float qy, float qz, float r2, int rv, int* queue, F visit)
{
  const int lane = threadIdx.x & 31;
  const unsigned full = 0xffffffffu;
  const int vx = floor_to_int(qx * g.inv_leaf) - g.min_b[0];
  const int vy = floor_to_int(qy * g.inv_leaf) - g.min_b[1];
  const int vz = floor_to_int(qz * g.inv_leaf) - g.min_b[2];
  int zlo = vz - rv, zhi = vz + rv, ylo = vy - rv, yhi = vy + rv;
  if (zhi < 0 || yhi < 0 || vx + rv < 0 || zlo >= g.div_v[2] || ylo >= g.div_v[1] || vx - rv >= g.div_v[0]) return 0;
  zlo = max(zlo, 0) >> g.shift[2];
  zhi = min(zhi, g.div_v[2] - 1) >> g.shift[2];
  ylo = max(ylo, 0) >> g.shift[1];
  yhi = min(yhi, g.div_v[1] - 1) >> g.shift[1];
  const int ny = yhi - ylo + 1;
  const int n_rows = (zhi - zlo + 1) * ny;
  const unsigned ny_magic = 0xFFFFFFFFu / (unsigned)ny + 1u;
  const float r2v = r2 * g.inv_leaf * g.inv_leaf;
  int qcount = 0, passed = 0;
  for (int row0 = 0; row0 < n_rows; row0 += 32) {
    // each lane resolves one row to its candidate run [s, e)
    int s = 0, e = 0;
    const int row = row0 + lane;
    if (row < n_rows) {
      const int rq = (int)__umulhi((unsigned)row, ny_magic);  // row / ny (exact for row < 2^18, ny < 512)
      const int cz = zlo + rq, cy = ylo + (row - rq * ny);
      const int z0 = cz << g.shift[2], z1 = z0 + (1 << g.shift[2]) - 1;
      const int y0 = cy << g.shift[1], y1 = y0 + (1 << g.shift[1]) - 1;
      const float fz = (float)max(max(max(z0 - vz, vz - z1), 0) - 1, 0);
      const float fy = (float)max(max(max(y0 - vy, vy - y1), 0) - 1, 0);
      const float rem = r2v - fz * fz - fy * fy;
      if (rem >= 0.0f) {
        const int rx = (int)sqrtf(rem) + 2;
        int xlo = vx - rx, xhi = vx + rx;
        if (xhi >= 0 && xlo < g.div_v[0]) {
          xlo = max(xlo, 0) >> g.shift[0];
          xhi = min(xhi, g.div_v[0] - 1) >> g.shift[0];
          const int base = (cz * g.dim[1] + cy) * g.dim[0];
          s = g.cell_start[base + xlo];
          e = g.cell_start[base + xhi + 1];
        }
      }
    }
    // inclusive scan of the run lengths
    int incl = e - s;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
      const int t = __shfl_up_sync(full, incl, o);
      if (lane >= o) incl += t;
    }
    const int total = __shfl_sync(full, incl, 31);
    const int excl = incl - (e - s);
    for (int t0 = 0; t0 < total; t0 += 32) {
      const int t = t0 + lane;
      // owner row of flattened candidate t: smallest L with incl[L] > t
      int L = 0;
#pragma unroll
      for (int step = 16; step >= 1; step >>= 1) {
        const int v = __shfl_sync(full, incl, L + step - 1);
        if (v <= t) L += step;
      }
      L = min(L, 31);
      const int ls = __shfl_sync(full, s, L), le = __shfl_sync(full, excl, L);
      bool pass = false;
      int k = 0;
      if (t < total) {
        k = ls + (t - le);
        const float4 p = g.pts[k];
        pass = em::dist2_3(qx, qy, qz, p.x, p.y, p.z) < r2;
      }
      const unsigned m = __ballot_sync(full, pass);
      if (pass) queue[qcount + __popc(m & ((1u << lane) - 1u))] = k;
      qcount += __popc(m);
      passed += __popc(m);
      __syncwarp();
      if (qcount >= 32) {
        visit(queue[lane]);
        __syncwarp();
        const int rest = qcount - 32;
        const int moved = (lane < rest) ? queue[32 + lane] : 0;
        __syncwarp();
        if (lane < rest) queue[lane] = moved;
        qcount = rest;
        __syncwarp();
      }
    }
  }
  if (ALL) {
    if (qcount > 0) visit(lane < qcount ? queue[lane] : -1);
  } else if (lane < qcount) {
    visit(queue[lane]);
  }
  __syncwarp();
  return passed;
}

// Warp-cooperative radius walk for ORDER-FREE consumers (integer / fixed-point sums): same row lookup and flattening as
// warp_radius_query, but every batch of 32 candidates is handed to `f(valid, k, p, d2)` straight away — no compaction
// queue, no ordering guarantee.  f is called by ALL 32 lanes together (valid = this lane holds a neighbour inside the
// radius), so it may use warp collectives.  All 32 lanes must call the walk with the same arguments.
template <typename F>
__device__ __forceinline__ void warp_radius_unordered(const GridView& g, float qx, float qy, float qz, float r2, int rv, F f)
{
  const int lane = threadIdx.x & 31;
  const unsigned full = 0xffffffffu;
  const int vx = floor_to_int(qx * g.inv_leaf) - g.min_b[0];
  const int vy = floor_to_int(qy * g.inv_leaf) - g.min_b[1];
  const int vz = floor_to_int(qz * g.inv_leaf) - g.min_b[2];
  int zlo = vz - rv, zhi = vz + rv, ylo = vy - rv, yhi = vy + rv;
  if (zhi < 0 || yhi < 0 || vx + rv < 0 || zlo >= g.div_v[2] || ylo >= g.div_v[1] || vx - rv >= g.div_v[0]) return;
  zlo = max(zlo, 0) >> g.shift[2];
  zhi = min(zhi, g.div_v[2] - 1) >> g.shift[2];
  ylo = max(ylo, 0) >> g.shift[1];
  yhi = min(yhi, g.div_v[1] - 1) >> g.shift[1];
  const int ny = yhi - ylo + 1;
  const int n_rows = (zhi - zlo + 1) * ny;
  const unsigned ny_magic = 0xFFFFFFFFu / (unsigned)ny + 1u;
  const float r2v = r2 * g.inv_leaf * g.inv_leaf;
  for (int row0 = 0; row0 < n_rows; row0 += 32) {
    int s = 0, e = 0;
    const int row = row0 + lane;
    if (row < n_rows) {
      const int rq = (int)__umulhi((unsigned)row, ny_magic);  // row / ny (exact for row < 2^18, ny < 512)
      const int cz = zlo + rq, cy = ylo + (row - rq * ny);
      const int z0 = cz << g.shift[2], z1 = z0 + (1 << g.shift[2]) - 1;
      const int y0 = cy << g.shift[1], y1 = y0 + (1 << g.shift[1]) - 1;
      const float fz = (float)max(max(max(z0 - vz, vz - z1), 0) - 1, 0);
      const float fy = (float)max(max(max(y0 - vy, vy - y1), 0) - 1, 0);
      const float rem = r2v - fz * fz - fy * fy;
      if (rem >= 0.0f) {
        const int rx = (int)sqrtf(rem) + 2;
        int xlo = vx - rx, xhi = vx + rx;
        if (xhi >= 0 && xlo < g.div_v[0]) {
          xlo = max(xlo, 0) >> g.shift[0];
          xhi = min(xhi, g.div_v[0] - 1) >> g.shift[0];
          const int base = (cz * g.dim[1] + cy) * g.dim[0];
          s = g.cell_start[base + xlo];
          e = g.cell_start[base + xhi + 1];
        }
      }
    }
    int incl = e - s;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
      const int t = __shfl_up_sync(full, incl, o);
      if (lane >= o) incl += t;
    }
    const int total = __shfl_sync(full, incl, 31);
    const int excl = incl - (e - s);
    for (int t0 = 0; t0 < total; t0 += 32) {
      const int t = t0 + lane;
      int L = 0;
#pragma unroll
      for (int step = 16; step >= 1; step >>= 1) {
        const int v = __shfl_sync(full, incl, L + step - 1);
        if (v <= t) L += step;
      }
      L = min(L, 31);
      const int ls = __shfl_sync(full, s, L), le = __shfl_sync(full, excl, L);
      bool valid = false;
      int k = 0;
      float4 p = make_float4(0.f, 0.f, 0.f, 0.f);
      float d2 = 0.f;
      if (t < total) {
        k = ls + (t - le);
        p = g.pts[k];
        d2 = em::dist2_3(qx, qy, qz, p.x, p.y, p.z);
        valid = d2 < r2;
      }
      f(valid, k, p, d2);
    }
  }
}

// The same walk for a GROUP of G lanes (G = 8, 16 or 32; the groups of a warp serve different queries and may diverge from
// each other, so every collective names only the group's lanes).  gmask = the group's lanes, glane = lane index inside it.
template <int G, typename F>
__device__ __forceinline__ void group_radius_unordered(const GridView& g, unsigned gmask, int glane, float qx, float qy, float qz, float r2,
                                                       int rv, F f)
{
  const int vx = floor_to_int(qx * g.inv_leaf) - g.min_b[0];
  const int vy = floor_to_int(qy * g.inv_leaf) - g.min_b[1];
  const int vz = floor_to_int(qz * g.inv_leaf) - g.min_b[2];
  int zlo = vz - rv, zhi = vz + rv, ylo = vy - rv, yhi = vy + rv;
  if (zhi < 0 || yhi < 0 || vx + rv < 0 || zlo >= g.div_v[2] || ylo >= g.div_v[1] || vx - rv >= g.div_v[0]) return;
  zlo = max(zlo, 0) >> g.shift[2];
  zhi = min(zhi, g.div_v[2] - 1) >> g.shift[2];
  ylo = max(ylo, 0) >> g.shift[1];
  yhi = min(yhi, g.div_v[1] - 1) >> g.shift[1];
  const int ny = yhi - ylo + 1;
  const int n_rows = (zhi - zlo + 1) * ny;
  const unsigned ny_magic = 0xFFFFFFFFu / (unsigned)ny + 1u;
  const float r2v = r2 * g.inv_leaf * g.inv_leaf;
  for (int row0 = 0; row0 < n_rows; row0 += G) {
    int s = 0, e = 0;
    const int row = row0 + glane;
    if (row < n_rows) {
      const int rq = (int)__umulhi((unsigned)row, ny_magic);  // row / ny (exact for row < 2^18, ny < 512)
      const int cz = zlo + rq, cy = ylo + (row - rq * ny);
      const int z0 = cz << g.shift[2], z1 = z0 + (1 << g.shift[2]) - 1;
      const int y0 = cy << g.shift[1], y1 = y0 + (1 << g.shift[1]) - 1;
      const float fz = (float)max(max(max(z0 - vz, vz - z1), 0) - 1, 0);
      const float fy = (float)max(max(max(y0 - vy, vy - y1), 0) - 1, 0);
      const float rem = r2v - fz * fz - fy * fy;
      if (rem >= 0.0f) {
        const int rx = (int)sqrtf(rem) + 2;
        int xlo = vx - rx, xhi = vx + rx;
        if (xhi >= 0 && xlo < g.div_v[0]) {
          xlo = max(xlo, 0) >> g.shift[0];
          xhi = min(xhi, g.div_v[0] - 1) >> g.shift[0];
          const int base = (cz * g.dim[1] + cy) * g.dim[0];
          s = g.cell_start[base + xlo];
          e = g.cell_start[base + xhi + 1];
        }
      }
    }
    int incl = e - s;
#pragma unroll
    for (int o = 1; o < G; o <<= 1) {
      const int t = __shfl_up_sync(gmask, incl, o, G);
      if (glane >= o) incl += t;
    }
    const int total = __shfl_sync(gmask, incl, G - 1, G);
    const int excl = incl - (e - s);
    for (int t0 = 0; t0 < total; t0 += G) {
      const int t = t0 + glane;
      int L = 0;  // owner row of flattened candidate t: smallest L with incl[L] > t
#pragma unroll
      for (int step = G / 2; step >= 1; step >>= 1) {
        const int v = __shfl_sync(gmask, incl, L + step - 1, G);
        if (v <= t) L += step;
      }
      L = min(L, G - 1);
      const int ls = __shfl_sync(gmask, s, L, G), le = __shfl_sync(gmask, excl, L, G);
      bool valid = false;
      int k = 0;
      float4 p = make_float4(0.f, 0.f, 0.f, 0.f);
      float d2 = 0.f;
      if (t < total) {
        k = ls + (t - le);
        p = g.pts[k];
        d2 = em::dist2_3(qx, qy, qz, p.x, p.y, p.z);
        valid = d2 < r2;
      }
      f(valid, k, p, d2);
    }
  }
}

// Nearest neighbour among points with (double)d2 <= bound; ties -> lower
// original index.  Rows are visited outward from the query row so the running
// best prunes the rest.  rv = ceil(sqrt(bound) / leaf) + 1 voxels.
// guess_slot >= 0: a slot (position in g.pts) expected to be close, e.g. the answer for a slightly different query; it
// only seeds the running best (the search still visits everything that could beat or tie it), so the result is the same.
// lim0_v > 0: an upper bound (voxel units, squared) on the distance to the nearest point that is known from elsewhere (the
// reach grid); like the guess it only tightens the pruning threshold.
__device__ __forceinline__ bool nearest_bounded(const GridView& g, float qx, float qy, float qz, double bound, int rv, int* out_idx,
                                                float* out_d2, float4* out_pt, int guess_slot = -1, int* out_slot = nullptr,
                                                float lim0_v = 0.0f)
{
  const int vx = floor_to_int(qx * g.inv_leaf) - g.min_b[0];
  const int vy = floor_to_int(qy * g.inv_leaf) - g.min_b[1];
  const int vz = floor_to_int(qz * g.inv_leaf) - g.min_b[2];
  if (vz + rv < 0 || vy + rv < 0 || vx + rv < 0 || vz - rv >= g.div_v[2] || vy - rv >= g.div_v[1] || vx - rv >= g.div_v[0]) return false;
  const int zlo = max(vz - rv, 0) >> g.shift[2], zhi = min(vz + rv, g.div_v[2] - 1) >> g.shift[2];
  const int ylo = max(vy - rv, 0) >> g.shift[1], yhi = min(vy + rv, g.div_v[1] - 1) >> g.shift[1];
  const int czq = min(max(vz, 0), g.div_v[2] - 1) >> g.shift[2];
  const int cyq = min(max(vy, 0), g.div_v[1] - 1) >> g.shift[1];
  bool found = false;
  float best = 0.0f;
  int best_idx = 0x7fffffff, best_slot = -1;
  float4 best_pt = make_float4(0.f, 0.f, 0.f, 0.f);
  // pruning threshold in voxel units; starts at the bound
  float lim_v = (float)bound * g.inv_leaf * g.inv_leaf * 1.0001f + 1e-3f;
  if (lim0_v > 0.0f) lim_v = fminf(lim_v, lim0_v);
  if (guess_slot >= 0 && guess_slot < g.n) {
    const float4 p = g.pts[guess_slot];
    const float d2 = em::dist2_3(qx, qy, qz, p.x, p.y, p.z);
    if ((double)d2 <= bound) {
      found = true;
      best = d2;
      best_idx = g.orig ? g.orig[guess_slot] : guess_slot;
      best_slot = guess_slot;
      best_pt = p;
      lim_v = fminf(lim_v, d2 * g.inv_leaf * g.inv_leaf * 1.0001f + 1e-3f);
    }
  }
  const int nz = zhi - zlo + 1, ny = yhi - ylo + 1;
  // Rows are visited in zig-zag order (0, +1, -1, +2, ...).  In one direction the row distance never decreases and the
  // pruning threshold only shrinks, so a direction that is out of range or pruned once stays so: it is closed, and the
  // loop ends when both directions are closed.
  bool zc0 = false, zc1 = false;  // direction closed: 0 = towards lower rows (and the query row), 1 = towards higher rows
  for (int iz = 0; iz < 2 * nz + 1; ++iz) {
    const bool zdir = iz & 1;
    if (zdir ? zc1 : zc0) {
      if (zc0 && zc1) break;
      continue;
    }
    const int cz = czq + (zdir ? (iz + 1) / 2 : -(iz / 2));
    const int z0 = cz << g.shift[2], z1 = z0 + (1 << g.shift[2]) - 1;
    const int dz = max(max(z0 - vz, vz - z1), 0);
    const float fz = (float)max(dz - 1, 0);
    if (cz < zlo || cz > zhi || fz * fz > lim_v) {
      if (zdir) zc1 = true; else zc0 = true;
      continue;
    }
    bool yc0 = false, yc1 = false;
    for (int iy = 0; iy < 2 * ny + 1; ++iy) {
      const bool ydir = iy & 1;
      if (ydir ? yc1 : yc0) {
        if (yc0 && yc1) break;
        continue;
      }
      const int cy = cyq + (ydir ? (iy + 1) / 2 : -(iy / 2));
      const int y0 = cy << g.shift[1], y1 = y0 + (1 << g.shift[1]) - 1;
      const int dy = max(max(y0 - vy, vy - y1), 0);
      const float fy = (float)max(dy - 1, 0);
      const float rem = lim_v - fz * fz - fy * fy;
      if (cy < ylo || cy > yhi || rem < 0.0f) {
        if (ydir) yc1 = true; else yc0 = true;
        continue;
      }
      const int rx = (int)sqrtf(rem) + 2;
      int xlo = vx - rx, xhi = vx + rx;
      if (xhi < 0 || xlo >= g.div_v[0]) continue;
      xlo = max(xlo, 0) >> g.shift[0];
      xhi = min(xhi, g.div_v[0] - 1) >> g.shift[0];
      const int base = (cz * g.dim[1] + cy) * g.dim[0];
      const int s = g.cell_start[base + xlo], e = g.cell_start[base + xhi + 1];
      for (int k = s; k < e; ++k) {
        const float4 p = g.pts[k];
        const float d2 = em::dist2_3(qx, qy, qz, p.x, p.y, p.z);
        if ((double)d2 > bound) continue;
        const int oi = g.orig ? g.orig[k] : k;
        if (!found || d2 < best || (d2 == best && oi < best_idx)) {
          found = true;
          best = d2;
          best_idx = oi;
          best_slot = k;
          best_pt = p;
          lim_v = d2 * g.inv_leaf * g.inv_leaf * 1.0001f + 1e-3f;
        }
      }
    }
  }
  *out_idx = best_idx;
  *out_d2 = best;
  *out_pt = best_pt;
  if (out_slot) *out_slot = found ? best_slot : -1;
  return found;
}

__device__ __forceinline__ long long warp_sum_ll(long long v)
{
  for (int o = 16; o > 0; o >>= 1) v += __shfl_down_sync(0xffffffffu, v, o);
  return v;
}

#endif  // __CUDACC__

// ---------------------------------------------------------------------------
// Host-side batched stage entry points (one call = all maps / all pairs).
// ---------------------------------------------------------------------------
struct DCloud {
  DBuf<float4> pts;
  int n = 0;
  CloudView view() const { return CloudView{pts.p, n}; }
};

// primitives.cu
void radix_sort_pairs_batch(Ctx& c, uint32_t* keys, uint32_t* vals, uint32_t* keys_tmp, uint32_t* vals_tmp, const std::vector<Seg>& segs,
                            int nbits, uint32_t** keys_sorted, uint32_t** vals_sorted);
// exclusive scan of flags per segment; pos[i] = #set flags before i (within its segment); totals on host
void scan_flags_batch(Ctx& c, const uint32_t* flags, uint32_t* pos, const std::vector<Seg>& segs, std::vector<int>& totals);

// voxel.cu — K1
void voxel_downsample_batch(Ctx& c, const std::vector<CloudView>& in, float leaf, std::vector<DCloud>& out, std::vector<VoxGeom>* geom);
// geom_hint: voxel geometry (same leaf) of a cloud that contains these points, e.g. the voxel grid they came out of;
// saves the bounding-box pass and one host synchronisation
void build_index_batch(Ctx& c, const std::vector<CloudView>& clouds, float leaf, int sx, int sy, int sz, std::vector<DIndex>& out,
                       std::vector<int>* was_sorted = nullptr, const std::vector<VoxGeom>* geom_hint = nullptr);
void transform_concat(Ctx& c, const std::vector<CloudView>& in, const std::vector<const float*>& transforms_rowmajor_host, DCloud& out);

// features.cu — K3, K4, K5, K7
void remove_outliers_batch(Ctx& c, const std::vector<CloudView>& clouds, const std::vector<DIndex>& idx, double radius, int min_nb,
                           std::vector<DCloud>& out, std::vector<DBuf<int>>* counts);
void normals_batch(Ctx& c, const std::vector<CloudView>& clouds, const std::vector<DIndex>& idx, double radius, std::vector<DBuf<float4>>& normals);
void sift_batch(Ctx& c, const std::vector<CloudView>& clouds, float min_scale, int n_octaves, int n_scales, float min_contrast,
                std::vector<DCloud>& keypoints, std::vector<DBuf<float>>* dog0);
void harris_batch(Ctx& c, const std::vector<CloudView>& clouds, const std::vector<DIndex>& idx, const std::vector<const float4*>& normals,
                  float threshold, float radius, std::vector<DCloud>& keypoints, std::vector<DBuf<float>>* response_dbg,
                  std::vector<DCloud>* unrefined_dbg);
// keypoints are filtered in place; desc[m] = K' x 33
void fpfh_batch(Ctx& c, const std::vector<CloudView>& clouds, const std::vector<DIndex>& idx, const std::vector<const float4*>& normals,
                std::vector<DCloud>& keypoints, double radius, std::vector<DBuf<float>>& desc, std::vector<DBuf<float>>* spfh_dbg);

// shot.cu — K8; desc[m] = K' x 1344, keypoints filtered in place
void shot_batch(Ctx& c, const std::vector<CloudView>& clouds, const std::vector<DIndex>& idx, const std::vector<const float4*>& normals,
                std::vector<DCloud>& keypoints, double radius, std::vector<DBuf<float>>& desc, std::vector<DBuf<float>>* rf_dbg);

// pfh.cu — PFH 125 (the reference's default descriptor); keypoints filtered in place
void pfh_batch(Ctx& c, const std::vector<CloudView>& clouds, const std::vector<DIndex>& idx, const std::vector<const float4*>& normals,
               std::vector<DCloud>& keypoints, double radius, std::vector<DBuf<float>>& desc, bool rgb = false);

// knn_tc.cu — K9 on tensor cores: per row of map a (the first na rows), the k nearest rows of map b, exact after re-rank
void rsd_batch(Ctx& c, const std::vector<CloudView>& clouds, const std::vector<DIndex>& idx, const std::vector<const float4*>& normals,
               std::vector<DCloud>& keypoints, double radius, std::vector<DBuf<float>>& desc);
void sc3d_batch(Ctx& c, const std::vector<CloudView>& clouds, const std::vector<DIndex>& idx, const std::vector<const float4*>& normals,
                std::vector<DCloud>& keypoints, double radius, std::vector<DBuf<float>>& desc);
struct KnnProblem {
  int a, b;  // indices into desc / n_rows
  int na;
  int k;
  int* idx;     // na x k
  float* dist;  // na x k
};
struct KnnAudit {  // tests: what the tensor-core filter saw for one problem
  std::vector<float> acc, norm_a, norm_b;
  float err_store = 0.f;
};
void knn_tc_batch(Ctx& c, const std::vector<const float*>& desc, const std::vector<int>& n_rows, int D, const std::vector<KnnProblem>& probs,
                  KnnAudit* audit = nullptr);
// matching.cu: picks the tensor-core filter or an exact FP32 scan per descriptor width / k / MM3D_KNN
void knn_problems(Ctx& c, const std::vector<const float*>& desc, const std::vector<int>& n_rows, int D, const std::vector<KnnProblem>& probs);

// matching.cu — K9, K10
struct PairJob {
  int a, b;  // indices into the per-map arrays
};
struct DCorr {
  DBuf<int2> pairs;
  DBuf<float> dist;
  int n = 0;
};
void match_batch(Ctx& c, const std::vector<const float*>& desc, const std::vector<int>& nk, int dim, const std::vector<PairJob>& jobs,
                 size_t k, std::vector<DCorr>& corr);
struct RansacOut {
  float T[16];         // row-major
  float best_model[16];
  int iterations;
  int best_count;
  int n_inliers;
  double sample_dist_thresh;
};
void ransac_batch(Ctx& c, const std::vector<CloudView>& keypoints, const std::vector<PairJob>& jobs, const std::vector<DCorr>& corr,
                  double inlier_threshold, std::vector<RansacOut>& out, std::vector<std::vector<int>>* inliers);

struct SacOut {
  float T[16];  // row-major
  unsigned long long rand_calls;  // rand() calls consumed up to and including this pair
  std::vector<float> errors;      // per-iteration error metric
};
// all_pairs: the complete row-major pair list (the rand() stream runs through all of it); wanted: indices into all_pairs
void sac_ia_batch(Ctx& c, const std::vector<CloudView>& keypoints, const std::vector<const float*>& desc, int dim,
                  const std::vector<PairJob>& all_pairs, const std::vector<int>& wanted, double min_sample_distance, double max_corr_dist,
                  int max_iterations, unsigned long long rand_skip, std::vector<SacOut>& out);

// icp.cu — K11, K12
// Reach grid of a target cloud: per voxel of the (margin-extended) index grid a LOWER bound, in voxel units squared, of the
// distance from any point inside that voxel to the nearest target point (separable min-plus transform of the occupancy with
// the per-axis cost max(|d| - 1, 0)^2, saturating at 255).  A query whose voxel is farther than the search bound is
// answered without a search; for the others the bound + the voxel diagonal caps the search radius.
struct ReachView {
  const unsigned char* lb2;  // dim[0] * dim[1] * dim[2], x fastest
  int org[3];                // voxel coordinate (relative to the index grid's min_b) of cell 0: -margin
  int dim[3];
  int none;                  // value stored where no occupied voxel lies inside the margin window (= min(255, margin^2))
};
struct DReach {
  ReachView v;
  DBuf<unsigned char> lb2;
};
// one reach grid per index with points; margin = voxels of reach (>= ceil(search radius / leaf) + 1, capped at 15)
void build_reach_batch(Ctx& c, const std::vector<DIndex>& idx, int margin, std::vector<DReach>& out);
struct IcpOut {
  float T[16];  // row-major
  int iterations;
  int converged;
};
// the target slot each source point matched in its pair's last ICP iteration (-1: none): a warm start for the score's search
struct IcpNeighbours {
  DBuf<int> slots;
  std::vector<long long> offset;  // per pair job, -1 = not available
};
void icp_batch(Ctx& c, const std::vector<CloudView>& clouds, const std::vector<DIndex>& idx, const std::vector<DReach>& reach,
               const std::vector<PairJob>& jobs, const std::vector<const float*>& T0_rowmajor, double max_dist, int max_it, double eps,
               std::vector<IcpOut>& out, std::vector<std::vector<long long>>* sums_dbg, IcpNeighbours* nn_keep = nullptr);
void score_batch(Ctx& c, const std::vector<CloudView>& clouds, const std::vector<DIndex>& idx, const std::vector<DReach>& reach,
                 const std::vector<PairJob>& jobs, const std::vector<const float*>& T_rowmajor, double max_range, std::vector<double>& scores,
                 const IcpNeighbours* nn_guess = nullptr);

// compose.cu — composeMaps sharded over ranks
struct KeyGeomHost {
  float inv_leaf;
  int min_b[3];
  int div_b[3];
  unsigned long long bucket_width;
  int passthrough;
};
KeyGeomHost compose_geometry(const float* bbox, double resolution, int n_buckets);
void compose_bbox(Ctx& c, const DCloud& cloud, float* bbox_host);
void compose_histogram(Ctx& c, const DCloud& cloud, const KeyGeomHost& geom, int n_buckets, unsigned long long* hist_host);
void compose_partition(Ctx& c, const DCloud& cloud, const KeyGeomHost& geom, int n_buckets, const std::vector<int>& splitters, int n_ranks,
                       unsigned long long* counts_host, float4* out_dev);

// graph.cpp — host pose graph (a14, a15)
struct HostEstimate {
  size_t source_idx, target_idx;
  float T[16];  // row-major
  double confidence;
};
std::vector<std::vector<float>> compute_global_transforms(const std::vector<HostEstimate>& pairwise, double confidence_threshold,
                                                          int* reference_frame, std::vector<int>* in_component,
                                                          std::vector<std::pair<int, int>>* tree_edges, std::vector<int>* centers);

}  // namespace mm3d
