// voxel.cu — K1 voxel-grid downSample (sort + segmented centroid reduce), the
// voxel-row neighbour index build, and K13 transform + concatenate.
//
// Replaces pcl::VoxelGrid<PointXYZRGB> as called from
//   map_merge_3d/src/features.cpp:17-27      (downSample)
//   map_merge_3d/src/map_merging.cpp:213,302 (registration resolution / compose)
// and inside pcl::SIFTKeypoint (one re-voxelisation per octave).
#include <algorithm>

#include "mm3d_internal.cuh"

namespace mm3d {

namespace {

__device__ __forceinline__ uint32_t f2ord(float f)
{
  const uint32_t b = __float_as_uint(f);
  return (b & 0x80000000u) ? ~b : (b | 0x80000000u);
}
__host__ __device__ __forceinline__ float ord2f(uint32_t u)
{
  const uint32_t b = (u & 0x80000000u) ? (u & 0x7fffffffu) : ~u;
#if defined(__CUDA_ARCH__)
  return __uint_as_float(b);
#else
  float f;
  memcpy(&f, &b, 4);
  return f;
#endif
}

// bbox[map][8] = ordered-uint min x,y,z, max x,y,z, number of non-finite points, pad.  Non-finite points are left out
// of the box, as pcl::getMinMax3D does for clouds that are not dense [PCL-recall pcl/common/impl/common.hpp].
// Block-level reduction (warp shuffles, then shared memory): seven atomics per BLOCK.
constexpr int BBOX_STRIDE = 8;
__global__ void __launch_bounds__(256) bbox_kernel(const CloudView* __restrict__ clouds, uint32_t* __restrict__ bbox)
{
  const CloudView cv = clouds[blockIdx.y];
  if ((int)(blockIdx.x * blockDim.x) >= cv.n) return;  // block-uniform
  uint32_t mn[3] = {0xffffffffu, 0xffffffffu, 0xffffffffu}, mx[3] = {0u, 0u, 0u}, bad = 0;
  for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < cv.n; i += gridDim.x * blockDim.x) {
    const float4 p = __ldg(&cv.pts[i]);
    if (!(isfinite(p.x) && isfinite(p.y) && isfinite(p.z))) {
      ++bad;
      continue;
    }
    const uint32_t a = f2ord(p.x), b = f2ord(p.y), c = f2ord(p.z);
    mn[0] = min(mn[0], a); mx[0] = max(mx[0], a);
    mn[1] = min(mn[1], b); mx[1] = max(mx[1], b);
    mn[2] = min(mn[2], c); mx[2] = max(mx[2], c);
  }
  __shared__ uint32_t sh[8][7];
  const int lane = threadIdx.x & 31, w = threadIdx.x >> 5;
#pragma unroll
  for (int k = 0; k < 3; ++k) {
    mn[k] = __reduce_min_sync(0xffffffffu, mn[k]);
    mx[k] = __reduce_max_sync(0xffffffffu, mx[k]);
  }
  bad = __reduce_add_sync(0xffffffffu, bad);
  if (lane == 0) {
#pragma unroll
    for (int k = 0; k < 3; ++k) { sh[w][k] = mn[k]; sh[w][3 + k] = mx[k]; }
    sh[w][6] = bad;
  }
  __syncthreads();
  if (threadIdx.x < 7) {
    const int k = threadIdx.x;
    uint32_t v = sh[0][k];
    for (int ww = 1; ww < 8; ++ww) v = k < 3 ? min(v, sh[ww][k]) : (k < 6 ? max(v, sh[ww][k]) : v + sh[ww][k]);
    uint32_t* bb = bbox + blockIdx.y * BBOX_STRIDE;
    if (k < 3) atomicMin(&bb[k], v);
    else if (k < 6) atomicMax(&bb[k], v);
    else if (v) atomicAdd(&bb[6], v);
  }
}

// pcl::VoxelGrid::applyFilter geometry [PCL-recall pcl/filters/impl/voxel_grid.hpp]
__global__ void geom_kernel(const CloudView* __restrict__ clouds, const uint32_t* __restrict__ bbox, float leaf, int n_maps,
                            VoxGeom* __restrict__ geom)
{
  const int m = blockIdx.x * blockDim.x + threadIdx.x;
  if (m >= n_maps) return;
  VoxGeom g;
  for (int k = 0; k < 3; ++k) { g.min_b[k] = 0; g.div_b[k] = 0; }
  g.passthrough = 0;
  g.nbits = 0;
  g.nonfinite = clouds[m].n > 0 ? (int)bbox[m * BBOX_STRIDE + 6] : 0;
  if (clouds[m].n > g.nonfinite) {
    const float inv = 1.0f / leaf;
    float mn[3], mx[3];
    for (int k = 0; k < 3; ++k) {
      mn[k] = ord2f(bbox[m * BBOX_STRIDE + k]);
      mx[k] = ord2f(bbox[m * BBOX_STRIDE + 3 + k]);
    }
    bool pass = !(leaf > 0.0f);
    if (!pass) {
      const float ex = (mx[0] - mn[0]) * inv, ey = (mx[1] - mn[1]) * inv, ez = (mx[2] - mn[2]) * inv;
      // casts of huge floats are clamped on the device; any such value trips the guard anyway
      const long long dx = (long long)ex + 1, dy = (long long)ey + 1, dz = (long long)ez + 1;
      if (!(ex < 3e9f) || !(ey < 3e9f) || !(ez < 3e9f) || dx * dy * dz > 2147483647LL) pass = true;
    }
    g.passthrough = pass ? 1 : 0;
    // The box in voxels.  Past the guard the output is the input, but neighbour indexes over it still need the box; it is
    // left at zero when its voxel coordinates do not fit in int32.
    bool fits = leaf > 0.0f;
    for (int k = 0; k < 3; ++k) {
      const float lo = floorf(mn[k] * inv), hi = floorf(mx[k] * inv);
      fits = fits && lo >= -2147483648.0f && hi < 2147483647.0f && (long long)hi - (long long)lo < 2147483647LL;
    }
    if (!pass || fits) {
      for (int k = 0; k < 3; ++k) {
        g.min_b[k] = (int)floorf(mn[k] * inv);
        g.div_b[k] = (int)floorf(mx[k] * inv) - g.min_b[k] + 1;
      }
    }
    if (!pass) {
      const long long cells = (long long)g.div_b[0] * g.div_b[1] * g.div_b[2];
      int nb = 1;
      while (nb < 32 && (1LL << nb) < cells) ++nb;
      g.nbits = nb;
    }
  }
  geom[m] = g;
}

__global__ void __launch_bounds__(256) voxel_key_kernel(const CloudView* __restrict__ clouds, const VoxGeom* __restrict__ geom,
                                                       const Seg* __restrict__ segs, float leaf, uint32_t* __restrict__ keys,
                                                       uint32_t* __restrict__ vals)
{
  const CloudView cv = clouds[blockIdx.y];
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= cv.n) return;
  const VoxGeom g = geom[blockIdx.y];
  const int off = segs[blockIdx.y].off;
  uint32_t key = 0;
  if (!g.passthrough) {
    const float inv = 1.0f / leaf;
    const float4 p = cv.pts[i];
    const int i0 = (int)(floorf(p.x * inv) - (float)g.min_b[0]);
    const int i1 = (int)(floorf(p.y * inv) - (float)g.min_b[1]);
    const int i2 = (int)(floorf(p.z * inv) - (float)g.min_b[2]);
    key = (uint32_t)(i0 + i1 * g.div_b[0] + i2 * g.div_b[0] * g.div_b[1]);
  }
  keys[off + i] = key;
  vals[off + i] = (uint32_t)i;
}

__global__ void __launch_bounds__(256) head_flag_kernel(const uint32_t* __restrict__ keys, const Seg* __restrict__ segs,
                                                       const VoxGeom* __restrict__ geom, uint32_t* __restrict__ flags)
{
  const Seg sg = segs[blockIdx.y];
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= sg.n) return;
  uint32_t f;
  if (geom[blockIdx.y].passthrough) f = 1;
  else f = (i == 0 || keys[sg.off + i] != keys[sg.off + i - 1]) ? 1u : 0u;
  flags[sg.off + i] = f;
}

// One thread per voxel: sequential float sums over the voxel's run, in ascending
// original index (stable sort), then pcl::CentroidPoint::get
// [PCL-recall pcl/common/impl/accumulators.hpp AccumulatorXYZ / AccumulatorRGBA].
struct CentroidOut {
  float4* pts;
};
__global__ void __launch_bounds__(256) centroid_kernel(const CloudView* __restrict__ clouds, const Seg* __restrict__ segs,
                                                      const uint32_t* __restrict__ keys, const uint32_t* __restrict__ vals,
                                                      const uint32_t* __restrict__ flags, const uint32_t* __restrict__ pos,
                                                      const VoxGeom* __restrict__ geom, const CentroidOut* __restrict__ outs)
{
  const Seg sg = segs[blockIdx.y];
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= sg.n) return;
  if (!flags[sg.off + i]) return;
  const CloudView cv = clouds[blockIdx.y];
  float4* out = outs[blockIdx.y].pts;
  const uint32_t v = pos[sg.off + i];
  if (geom[blockIdx.y].passthrough) {
    out[v] = cv.pts[i];
    return;
  }
  const uint32_t key = keys[sg.off + i];
  float sx = 0.f, sy = 0.f, sz = 0.f, sr = 0.f, sgc = 0.f, sb = 0.f, sa = 0.f;
  int k = i;
  while (k < sg.n && keys[sg.off + k] == key) {
    const float4 p = cv.pts[vals[sg.off + k]];
    const uint32_t c = __float_as_uint(p.w);
    sx += p.x; sy += p.y; sz += p.z;
    sr += (float)((c >> 16) & 0xffu);
    sgc += (float)((c >> 8) & 0xffu);
    sb += (float)(c & 0xffu);
    sa += (float)((c >> 24) & 0xffu);
    ++k;
  }
  const float n = (float)(k - i);
  float4 o;
  o.x = sx / n; o.y = sy / n; o.z = sz / n;
  const uint32_t rgba = ((uint32_t)(sa / n) << 24) | ((uint32_t)(sr / n) << 16) | ((uint32_t)(sgc / n) << 8) | (uint32_t)(sb / n);
  o.w = __uint_as_float(rgba);
  out[v] = o;
}

// ---- non-finite points (pcl::VoxelGrid skips them when the cloud is not dense) -------------------------------------
struct FiniteJob {
  const float4* src;
  float4* dst;
  int n;
  int off;  // offset of this cloud in the concatenated flag / position arrays
};
__global__ void __launch_bounds__(256) finite_flag_kernel(const FiniteJob* __restrict__ jobs, uint32_t* __restrict__ flags)
{
  const FiniteJob j = jobs[blockIdx.y];
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= j.n) return;
  const float4 p = j.src[i];
  flags[j.off + i] = (isfinite(p.x) && isfinite(p.y) && isfinite(p.z)) ? 1u : 0u;
}
__global__ void __launch_bounds__(256) finite_compact_kernel(const FiniteJob* __restrict__ jobs, const uint32_t* __restrict__ flags,
                                                            const uint32_t* __restrict__ pos)
{
  const FiniteJob j = jobs[blockIdx.y];
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= j.n) return;
  if (flags[j.off + i]) j.dst[pos[j.off + i]] = j.src[i];
}

// ---- index build ------------------------------------------------------------
struct IndexGeom {
  int min_b[3];
  int div_v[3];
  int shift[3];
  int dim[3];
};

__global__ void __launch_bounds__(256) cell_key_kernel(const CloudView* __restrict__ clouds, const IndexGeom* __restrict__ ig,
                                                      const Seg* __restrict__ segs, float inv_leaf, uint32_t* __restrict__ keys,
                                                      uint32_t* __restrict__ vals)
{
  const CloudView cv = clouds[blockIdx.y];
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= cv.n) return;
  const IndexGeom g = ig[blockIdx.y];
  const float4 p = cv.pts[i];
  const int cx = (floor_to_int(p.x * inv_leaf) - g.min_b[0]) >> g.shift[0];
  const int cy = (floor_to_int(p.y * inv_leaf) - g.min_b[1]) >> g.shift[1];
  const int cz = (floor_to_int(p.z * inv_leaf) - g.min_b[2]) >> g.shift[2];
  const int off = segs[blockIdx.y].off;
  keys[off + i] = (uint32_t)(cx + g.dim[0] * (cy + g.dim[1] * cz));
  vals[off + i] = (uint32_t)i;
}

__global__ void __launch_bounds__(256) sorted_check_kernel(const uint32_t* __restrict__ keys, const Seg* __restrict__ segs,
                                                          int* __restrict__ unsorted)
{
  const Seg sg = segs[blockIdx.y];
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= sg.n || i == 0) return;
  if (keys[sg.off + i] < keys[sg.off + i - 1]) unsorted[blockIdx.y] = 1;
}

struct CellStartJob {
  const uint32_t* keys;  // sorted cell keys of this map
  int n;
  int ncell;
  int* cell_start;
};
__global__ void __launch_bounds__(256) cell_start_kernel(const CellStartJob* __restrict__ jobs)
{
  const CellStartJob j = jobs[blockIdx.y];
  const int c = blockIdx.x * blockDim.x + threadIdx.x;
  if (c > j.ncell) return;
  int lo = 0, hi = j.n;  // first slot with key >= c
  while (lo < hi) {
    const int mid = (lo + hi) >> 1;
    if (j.keys[mid] < (uint32_t)c) lo = mid + 1;
    else hi = mid;
  }
  j.cell_start[c] = lo;
}

struct GatherJob {
  const float4* src;
  const uint32_t* order;
  float4* dst;
  int* orig;
  int n;
};
__global__ void __launch_bounds__(256) gather_kernel(const GatherJob* __restrict__ jobs)
{
  const GatherJob j = jobs[blockIdx.y];
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= j.n) return;
  const uint32_t o = j.order[i];
  j.dst[i] = j.src[o];
  j.orig[i] = (int)o;
}

struct XformJob {
  const float4* src;
  float4* dst;
  int n;
  float m[12];
};
// pcl::transformPointCloud [PCL-recall pcl/common/impl/transforms.hpp]; colour copied
__global__ void __launch_bounds__(256) xform_kernel(const XformJob* __restrict__ jobs)
{
  const XformJob& j = jobs[blockIdx.y];
  for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < j.n; i += gridDim.x * blockDim.x) {
    const float4 p = j.src[i];
    float4 o;
    em::transform_point(j.m, p.x, p.y, p.z, &o.x, &o.y, &o.z);
    o.w = p.w;
    j.dst[i] = o;
  }
}

static std::vector<Seg> make_segs(const std::vector<CloudView>& in, int* total)
{
  std::vector<Seg> segs(in.size());
  int off = 0;
  for (size_t m = 0; m < in.size(); ++m) {
    segs[m].off = off;
    segs[m].n = in[m].n;
    off += in[m].n;
  }
  *total = off;
  return segs;
}

static int max_n(const std::vector<CloudView>& in)
{
  int mx = 0;
  for (const CloudView& v : in) mx = std::max(mx, v.n);
  return mx;
}

static void compute_geom(Ctx& c, const std::vector<CloudView>& in, const DBuf<CloudView>& dviews, float leaf, std::vector<VoxGeom>& geom,
                         DBuf<VoxGeom>& dgeom)
{
  const int M = (int)in.size();
  std::vector<uint32_t> init(M * BBOX_STRIDE);
  for (int m = 0; m < M; ++m)
    for (int k = 0; k < BBOX_STRIDE; ++k) init[m * BBOX_STRIDE + k] = k < 3 ? 0xffffffffu : 0u;
  DBuf<uint32_t> bbox = to_device(c, init);
  const int mx = max_n(in);
  const int blocks = std::max(1, std::min((mx + 255) / 256, 148 * 4));
  MM_LAUNCH(c, bbox_kernel, dim3(blocks, M), 256, 0, dviews.p, bbox.p);
  dgeom.alloc(c, M);
  MM_LAUNCH(c, geom_kernel, (M + 63) / 64, 64, 0, dviews.p, bbox.p, leaf, M, dgeom.p);
  geom.resize(M);
  dgeom.download(c, geom.data(), M);
  c.sync();
}

}  // namespace

void voxel_downsample_batch(Ctx& c, const std::vector<CloudView>& in_arg, float leaf, std::vector<DCloud>& out, std::vector<VoxGeom>* geom_out)
{
  const int M = (int)in_arg.size();
  out.clear();
  out.resize(M);
  if (M == 0) return;
  int total = 0;
  std::vector<Seg> segs = make_segs(in_arg, &total);
  std::vector<VoxGeom> geom(M);
  if (total == 0) {
    for (auto& g : geom) memset(&g, 0, sizeof(g));
    if (geom_out) *geom_out = geom;
    return;
  }
  DBuf<CloudView> dviews = to_device(c, in_arg);
  DBuf<VoxGeom> dgeom;
  compute_geom(c, in_arg, dviews, leaf, geom, dgeom);
  if (geom_out) *geom_out = geom;
  // Clouds with NaN / Inf coordinates (organised RGB-D clouds, is_dense == false): pcl::VoxelGrid leaves such points out of
  // the bounding box and out of the voxels.  Rare, so the common case pays only the count that rides on the bbox pass.
  std::vector<CloudView> in = in_arg;
  std::vector<DBuf<float4>> finite_copy;
  {
    std::vector<FiniteJob> fj;
    std::vector<Seg> fsegs;
    std::vector<int> fmap;
    int foff = 0, fmx = 0;
    for (int m = 0; m < M; ++m)
      if (geom[m].nonfinite > 0 && !geom[m].passthrough) {  // the overflow guard returns the input as it is, NaNs included
        fj.push_back(FiniteJob{in[m].pts, nullptr, in[m].n, foff});
        fsegs.push_back(Seg{foff, in[m].n});
        fmap.push_back(m);
        foff += in[m].n;
        fmx = std::max(fmx, in[m].n);
      }
    if (!fj.empty()) {
      DBuf<uint32_t> fflags(c, foff), fpos(c, foff);
      finite_copy.resize(fj.size());
      for (size_t t = 0; t < fj.size(); ++t) {
        finite_copy[t].alloc(c, (size_t)(fj[t].n - geom[fmap[t]].nonfinite) + 1);
        fj[t].dst = finite_copy[t].p;
      }
      DBuf<FiniteJob> dfj = to_device(c, fj);
      const dim3 fgrid((fmx + 255) / 256, (unsigned)fj.size());
      MM_LAUNCH(c, finite_flag_kernel, fgrid, 256, 0, dfj.p, fflags.p);
      std::vector<int> ftotals;
      scan_flags_batch(c, fflags.p, fpos.p, fsegs, ftotals);
      MM_LAUNCH(c, finite_compact_kernel, fgrid, 256, 0, dfj.p, fflags.p, fpos.p);
      for (size_t t = 0; t < fj.size(); ++t) in[fmap[t]] = CloudView{finite_copy[t].p, ftotals[t]};
      segs = make_segs(in, &total);
      dviews = to_device(c, in);
      if (total == 0) return;
    }
  }
  int nbits = 0;
  for (const VoxGeom& g : geom) nbits = std::max(nbits, g.nbits);
  DBuf<Seg> dsegs = to_device(c, segs);
  DBuf<uint32_t> keys(c, total), vals(c, total), keys2(c, total), vals2(c, total);
  const int mx = max_n(in);
  const dim3 grid((mx + 255) / 256, M);
  MM_BYTES(c, 24.0 * total);
  MM_LAUNCH(c, voxel_key_kernel, grid, 256, 0, dviews.p, dgeom.p, dsegs.p, leaf, keys.p, vals.p);
  uint32_t *ks, *vs;
  radix_sort_pairs_batch(c, keys.p, vals.p, keys2.p, vals2.p, segs, nbits, &ks, &vs);
  uint32_t* flags = (ks == keys.p) ? keys2.p : keys.p;  // the spare key buffer
  DBuf<uint32_t> pos(c, total);
  MM_LAUNCH(c, head_flag_kernel, grid, 256, 0, ks, dsegs.p, dgeom.p, flags);
  std::vector<int> totals;
  scan_flags_batch(c, flags, pos.p, segs, totals);
  std::vector<CentroidOut> outs(M);
  for (int m = 0; m < M; ++m) {
    out[m].n = totals[m];
    out[m].pts.alloc(c, totals[m]);
    outs[m].pts = out[m].pts.p;
  }
  DBuf<CentroidOut> douts = to_device(c, outs);
  { double b = 28.0 * total; for (int m = 0; m < M; ++m) b += 16.0 * totals[m]; MM_BYTES(c, b); }
  MM_LAUNCH(c, centroid_kernel, grid, 256, 0, dviews.p, dsegs.p, ks, vs, flags, pos.p, dgeom.p, douts.p);
}

void build_index_batch(Ctx& c, const std::vector<CloudView>& clouds, float leaf, int sx, int sy, int sz, std::vector<DIndex>& out,
                       std::vector<int>* was_sorted, const std::vector<VoxGeom>* geom_hint)
{
  const int M = (int)clouds.size();
  out.clear();
  out.resize(M);
  if (was_sorted) was_sorted->assign(M, 1);
  if (M == 0) return;
  int total = 0;
  std::vector<Seg> segs = make_segs(clouds, &total);
  const float inv_leaf = 1.0f / leaf;
  for (int m = 0; m < M; ++m) {
    GridView& v = out[m].v;
    memset(&v, 0, sizeof(v));
    v.pts = clouds[m].pts;
    v.n = clouds[m].n;
    v.inv_leaf = inv_leaf;
    v.leaf = leaf;
  }
  if (total == 0) {
    for (int m = 0; m < M; ++m) {
      out[m].cell_start.alloc(c, 1);
      out[m].cell_start.zero(c);
      out[m].v.cell_start = out[m].cell_start.p;
    }
    return;
  }
  DBuf<CloudView> dviews = to_device(c, clouds);
  std::vector<VoxGeom> geom;
  DBuf<VoxGeom> dgeom;
  bool hinted = geom_hint && (int)geom_hint->size() == M;
  if (hinted)
    for (int m = 0; m < M; ++m)
      if (clouds[m].n > 0 && ((*geom_hint)[m].passthrough || (*geom_hint)[m].div_b[0] <= 0)) hinted = false;
  if (hinted) geom = *geom_hint;
  else compute_geom(c, clouds, dviews, leaf, geom, dgeom);
  std::vector<IndexGeom> ig(M);
  for (int m = 0; m < M; ++m) {
    // Past pcl::VoxelGrid's overflow guard the index still works from the box (coarsened below like any large one), unless
    // the box's voxel coordinates do not fit in int32 or the cloud kept non-finite points, which have no cell.
    if (geom[m].passthrough && clouds[m].n > 0 && (geom[m].div_b[0] <= 0 || geom[m].nonfinite > 0))
      throw std::runtime_error(geom[m].nonfinite > 0 ? "build_index: non-finite points in a cloud past the voxel-grid overflow guard"
                                                     : "build_index: voxel coordinates of the cloud do not fit in int32");
    int sh[3] = {sx, sy, sz};
    IndexGeom& g = ig[m];
    for (;;) {
      long long cells = 1;
      for (int k = 0; k < 3; ++k) {
        g.min_b[k] = geom[m].min_b[k];
        g.div_v[k] = geom[m].div_b[k];
        g.shift[k] = sh[k];
        g.dim[k] = clouds[m].n > 0 ? ((geom[m].div_b[k] - 1) >> sh[k]) + 1 : 0;
        cells *= std::max(g.dim[k], 1);
      }
      if (cells <= (1LL << 27)) break;
      // keep the dense table bounded: coarsen x first (keeps ordered enumeration), then y/z
      if (sh[0] < 8) ++sh[0];
      else { ++sh[1]; ++sh[2]; }
    }
    GridView& v = out[m].v;
    for (int k = 0; k < 3; ++k) { v.min_b[k] = g.min_b[k]; v.div_v[k] = g.div_v[k]; v.shift[k] = g.shift[k]; v.dim[k] = g.dim[k]; }
  }
  DBuf<IndexGeom> dig = to_device(c, ig);
  DBuf<Seg> dsegs = to_device(c, segs);
  DBuf<uint32_t> keys(c, total), vals(c, total);
  const int mx = max_n(clouds);
  const dim3 grid((mx + 255) / 256, M);
  MM_LAUNCH(c, cell_key_kernel, grid, 256, 0, dviews.p, dig.p, dsegs.p, inv_leaf, keys.p, vals.p);
  DBuf<int> dunsorted(c, M);
  dunsorted.zero(c);
  MM_LAUNCH(c, sorted_check_kernel, grid, 256, 0, keys.p, dsegs.p, dunsorted.p);
  std::vector<int> unsorted(M);
  dunsorted.download(c, unsorted.data(), M);
  c.sync();
  // re-sort the maps whose points are not already in cell order
  std::vector<Seg> ssegs;
  std::vector<int> smap;
  int max_bits = 0;
  for (int m = 0; m < M; ++m)
    if (unsorted[m]) {
      ssegs.push_back(segs[m]);
      smap.push_back(m);
      long long cells = (long long)ig[m].dim[0] * ig[m].dim[1] * ig[m].dim[2];
      int nb = 1;
      while (nb < 32 && (1LL << nb) < cells) ++nb;
      max_bits = std::max(max_bits, nb);
      if (was_sorted) (*was_sorted)[m] = 0;
    }
  DBuf<uint32_t> keys2, vals2;
  const uint32_t* ks = keys.p;
  if (!ssegs.empty()) {
    keys2.alloc(c, total);
    vals2.alloc(c, total);
    // unsorted segments are sorted in place inside the concatenated arrays; the
    // result may land in either buffer, so copy the sorted segments' peers across
    uint32_t *kso, *vso;
    radix_sort_pairs_batch(c, keys.p, vals.p, keys2.p, vals2.p, ssegs, max_bits, &kso, &vso);
    std::vector<GatherJob> gj;
    for (size_t t = 0; t < smap.size(); ++t) {
      const int m = smap[t];
      out[m].pts_sorted.alloc(c, clouds[m].n);
      out[m].orig.alloc(c, clouds[m].n);
      out[m].v.pts = out[m].pts_sorted.p;
      out[m].v.orig = out[m].orig.p;
      gj.push_back(GatherJob{clouds[m].pts, vso + segs[m].off, out[m].pts_sorted.p, out[m].orig.p, clouds[m].n});
      if (kso != keys.p) MM_CUDA(cudaMemcpyAsync(keys.p + segs[m].off, kso + segs[m].off, (size_t)segs[m].n * 4, cudaMemcpyDeviceToDevice, c.stream));
    }
    DBuf<GatherJob> dgj = to_device(c, gj);
    int gmx = 0;
    for (const GatherJob& j : gj) gmx = std::max(gmx, j.n);
    MM_LAUNCH(c, gather_kernel, dim3((gmx + 255) / 256, (unsigned)gj.size()), 256, 0, dgj.p);
  }
  std::vector<CellStartJob> cj(M);
  int cmx = 0;
  for (int m = 0; m < M; ++m) {
    const int ncell = ig[m].dim[0] * ig[m].dim[1] * ig[m].dim[2];
    out[m].cell_start.alloc(c, (size_t)ncell + 1);
    out[m].v.cell_start = out[m].cell_start.p;
    cj[m] = CellStartJob{ks + segs[m].off, clouds[m].n, ncell, out[m].cell_start.p};
    cmx = std::max(cmx, ncell + 1);
  }
  DBuf<CellStartJob> dcj = to_device(c, cj);
  MM_LAUNCH(c, cell_start_kernel, dim3((cmx + 255) / 256, M), 256, 0, dcj.p);
}

void transform_concat(Ctx& c, const std::vector<CloudView>& in, const std::vector<const float*>& transforms, DCloud& out)
{
  size_t total = 0;
  for (const CloudView& v : in) total += (size_t)v.n;
  out.n = (int)total;
  out.pts.alloc(c, total);
  if (total == 0) return;
  std::vector<XformJob> jobs;
  size_t off = 0;
  int mx = 0;
  for (size_t m = 0; m < in.size(); ++m) {
    if (in[m].n == 0) continue;
    XformJob j;
    j.src = in[m].pts;
    j.dst = out.pts.p + off;
    j.n = in[m].n;
    for (int k = 0; k < 12; ++k) j.m[k] = transforms[m][k];
    jobs.push_back(j);
    off += (size_t)in[m].n;
    mx = std::max(mx, in[m].n);
  }
  DBuf<XformJob> dj = to_device(c, jobs);
  const int blocks = std::max(1, std::min((mx + 255) / 256, 148 * 8));
  MM_LAUNCH(c, xform_kernel, dim3(blocks, (unsigned)jobs.size()), 256, 0, dj.p);
}

}  // namespace mm3d
