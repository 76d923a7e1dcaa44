// icp.cu — K11 point-to-point ICP refine and K12 Euclidean transform score, all pairs at once.
//   <- map_merge_3d/src/matching.cpp:196-221 (pcl::IterativeClosestPoint, TransformationEstimationSVD,
//      DefaultConvergenceCriteria) and :259-268 (pcl::registration::TransformationValidationEuclidean)
//
// The WHOLE ICP loop of every pair is ONE persistent kernel.  Every pair carries its own tile counter: blocks pull
// 128-query tiles from whichever pair has tiles left; a tile applies the pair's previous step transform, finds each
// query's nearest target point within the correspondence distance and adds its share of {n, sum p, sum q, sum q p^T,
// sum d^2} (fixed-point int64, so the reduction is order-independent and matches the CPU checker bit for bit); the last
// tile of a pair's iteration solves Umeyama (3x3 SVD), updates the transform, tests convergence and — if the pair goes on
// — re-opens its tile counter for the next iteration.  Pairs therefore iterate independently (no grid-wide barrier: with
// one, a quarter of the warp time was spent waiting for the slowest pair of every iteration, ncu round 2), and the loop
// ends on the device when no pair is active.  The host launches once and reads the results once.
//
// Nearest-neighbour search: thread per query over the voxel-row index, pruned three ways — (1) the target's reach grid
// (a lower bound of the distance to the nearest target point per voxel) answers queries that have no target point in
// range without a search, which is most of the non-overlapping part of a pair; (2) the same bound plus the voxel
// diagonal caps the radius for the others; (3) the previous iteration's match seeds the running best.
#include <algorithm>
#include <cmath>
#include <cstring>
#include <type_traits>

#include "mm3d_internal.cuh"

namespace mm3d {

namespace {

constexpr int IB = 128;
constexpr int NSUM = 17;  // n, Sp[3], Sq[3], Sqp[9], Sd

struct IcpState {
  float final_t[16];  // accumulated ICP transform (row-major)
  float step[16];     // transformation_ of the last iteration
  double prev_mse;
  int iterations;
  int active;
  int converged;
  int pad;
};

struct IcpJob {
  GridView tgt;      // target index
  ReachView reach;   // target reach grid
  const float4* src; // source cloud
  int ns;
  float4* work;      // transformed source (input_transformed)
  long long* sums;   // NSUM
  IcpState* st;
  int* ticket;       // tiles of this pair that finished the current iteration
  int* next_tile;    // tile counter of the current iteration (>= n_tiles: nothing left / iteration being solved)
  int n_tiles;
  float t0[16];      // initial guess, row-major
  long long* sums_log;  // optional max_log x NSUM
  int* nn_slot;      // per source point: the target slot matched in the previous iteration (-1 = none)
};

struct IcpLoop {
  int n_active;  // pairs still iterating
  int pad[3];
};

// ---------------------------------------------------------------- reach grid
struct ReachJob {
  GridView g;
  ReachView r;
  unsigned char* a;  // ping
  unsigned char* b;  // pong (final)
};

__global__ void __launch_bounds__(256) reach_mark_kernel(const ReachJob* __restrict__ jobs)
{
  const ReachJob& j = jobs[blockIdx.y];
  for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < j.g.n; i += gridDim.x * blockDim.x) {
    const float4 p = j.g.pts[i];
    const int x = floor_to_int(p.x * j.g.inv_leaf) - j.g.min_b[0] - j.r.org[0];
    const int y = floor_to_int(p.y * j.g.inv_leaf) - j.g.min_b[1] - j.r.org[1];
    const int z = floor_to_int(p.z * j.g.inv_leaf) - j.g.min_b[2] - j.r.org[2];
    if (x >= 0 && y >= 0 && z >= 0 && x < j.r.dim[0] && y < j.r.dim[1] && z < j.r.dim[2])
      j.a[((size_t)z * j.r.dim[1] + y) * j.r.dim[0] + x] = 0;
  }
}

// one axis of the min-plus transform: out(c) = min over |d| <= margin of in(c + d * stride) + max(|d| - 1, 0)^2, saturating
__global__ void __launch_bounds__(256) reach_pass_kernel(const ReachJob* __restrict__ jobs, int axis, int margin, int from_a)
{
  const ReachJob& j = jobs[blockIdx.y];
  const size_t ncell = (size_t)j.r.dim[0] * j.r.dim[1] * j.r.dim[2];
  const unsigned char* in = from_a ? j.a : j.b;
  unsigned char* out = from_a ? j.b : j.a;
  for (size_t c = (size_t)blockIdx.x * blockDim.x + threadIdx.x; c < ncell; c += (size_t)gridDim.x * blockDim.x) {
    const int x = (int)(c % j.r.dim[0]);
    const int y = (int)((c / j.r.dim[0]) % j.r.dim[1]);
    const int z = (int)(c / ((size_t)j.r.dim[0] * j.r.dim[1]));
    const int pos = axis == 0 ? x : (axis == 1 ? y : z);
    const int len = j.r.dim[axis];
    const long long stride = axis == 0 ? 1 : (axis == 1 ? (long long)j.r.dim[0] : (long long)j.r.dim[0] * j.r.dim[1]);
    const int lo = max(-margin, -pos), hi = min(margin, len - 1 - pos);
    int best = 255;
    for (int d = lo; d <= hi; ++d) {
      const int f = max(abs(d) - 1, 0);
      const int v = (int)in[(long long)c + (long long)d * stride] + f * f;
      best = min(best, v);
    }
    out[c] = (unsigned char)min(best, j.r.none);
  }
}

// lower bound (voxel units, squared) for a query; returns false when the query lies outside the grid (= farther than the margin)
__device__ __forceinline__ bool reach_lookup(const GridView& g, const ReachView& r, float qx, float qy, float qz, int* lb2)
{
  const int x = floor_to_int(qx * g.inv_leaf) - g.min_b[0] - r.org[0];
  const int y = floor_to_int(qy * g.inv_leaf) - g.min_b[1] - r.org[1];
  const int z = floor_to_int(qz * g.inv_leaf) - g.min_b[2] - r.org[2];
  if (x < 0 || y < 0 || z < 0 || x >= r.dim[0] || y >= r.dim[1] || z >= r.dim[2]) return false;
  *lb2 = (int)__ldg(&r.lb2[((size_t)z * r.dim[1] + y) * r.dim[0] + x]);
  return true;
}

// Walk downhill on the reach grid from cell (x, y, z) — one axis step at a time to the neighbour with the smallest lower
// bound — until a cell with lower bound 0 (an occupied voxel in its 3 x 3 x 3 block).  The field is a min-plus transform with
// the per-axis cost max(|d| - 1, 0)^2, so while the value is positive some axis neighbour is strictly smaller: the walk
// ends after at most sum(|d_i| - 1) steps.  Returns false if it leaves the grid or stalls (saturated values).
__device__ __forceinline__ bool reach_descend(const ReachView& r, int& x, int& y, int& z, int cur)
{
  for (int step = 0; step < 48 && cur > 0; ++step) {
    int best = cur, bx = x, by = y, bz = z;
#pragma unroll
    for (int t = 0; t < 6; ++t) {
      const int nx = x + (t == 0) - (t == 1), ny = y + (t == 2) - (t == 3), nz = z + (t == 4) - (t == 5);
      if (nx < 0 || ny < 0 || nz < 0 || nx >= r.dim[0] || ny >= r.dim[1] || nz >= r.dim[2]) continue;
      const int v = (int)__ldg(&r.lb2[((size_t)nz * r.dim[1] + ny) * r.dim[0] + nx]);
      if (v < best) {
        best = v;
        bx = nx;
        by = ny;
        bz = nz;
      }
    }
    if (best >= cur) return false;
    cur = best;
    x = bx;
    y = by;
    z = bz;
  }
  return cur == 0;
}

// squared distance from the query to the nearest point of the 3 x 3 x 3 voxel block around index voxel (vx, vy, vz) — any
// point there is a real target point, so the result is an upper bound of the nearest-neighbour distance; 3e38 if none
__device__ __forceinline__ float block27_any(const GridView& g, int vx, int vy, int vz, float qx, float qy, float qz)
{
  float best = 3.0e38f;
  const int xlo = max(vx - 1, 0), xhi = min(vx + 1, g.div_v[0] - 1);
  if (xlo > xhi) return best;
  for (int t = 0; t < 9; ++t) {
    const int cz = vz + t / 3 - 1, cy = vy + t % 3 - 1;
    if (cz < 0 || cz >= g.div_v[2] || cy < 0 || cy >= g.div_v[1]) continue;
    const int base = (cz * g.dim[1] + cy) * g.dim[0];
    const int s = __ldg(&g.cell_start[base + xlo]), e = __ldg(&g.cell_start[base + xhi + 1]);
    for (int k = s; k < e; ++k) {
      const float4 p = g.pts[k];
      best = fminf(best, em::dist2_3(qx, qy, qz, p.x, p.y, p.z));
    }
  }
  return best;
}

// Gap slack of the voxel geometry, in voxels, for a query at voxel coordinates (fx, fy, fz) = fl(q * inv_leaf).  The query's
// coordinate and a point's row, floor(fl(p * inv_leaf)), are each rounded by up to half an ulp of the voxel coordinate, so
// the true gap between the query and a neighbouring row or cell can be smaller than the computed one by up to about
// |f| * 2^-23 per axis: 5e-4 voxel at 500 m from the origin with a 0.1 m leaf.  Twice that bound, summed over the axes:
__device__ __forceinline__ float voxel_slack(float fx, float fy, float fz)
{
  return (fabsf(fx) + fabsf(fy) + fabsf(fz) + 1.0f) * 2.384185791015625e-7f;  // 2^-22
}

// The 3 x 3 x 3 voxel block around the query in an index with one-voxel cells: nine (z, y) rows of three cells each, every
// row one contiguous run of points.  All nine run bounds are loaded up front (independent loads), rows are skipped when
// their slab distance already exceeds the running best.  Every point outside the block is at least one voxel away, so a
// best closer than that is the exact nearest neighbour (*certain); otherwise the caller falls back to the general search.
// Both tests take the slab distances and the one voxel less voxel_slack, so they hold at any distance from the origin.
__device__ __forceinline__ bool nearest_block27(const GridView& g, float qx, float qy, float qz, double bound, int guess_slot, int* out_idx,
                                                float* out_d2, float4* out_pt, int* out_slot, bool* certain)
{
  const float fx = qx * g.inv_leaf, fy = qy * g.inv_leaf, fz = qz * g.inv_leaf;
  const float slack = voxel_slack(fx, fy, fz);
  const float flx = floorf(fx), fly = floorf(fy), flz = floorf(fz);
  const int vx = (int)flx - g.min_b[0], vy = (int)fly - g.min_b[1], vz = (int)flz - g.min_b[2];
  const float ay = fy - fly, az = fz - flz;  // position inside the voxel, voxel units
  // least gaps to the rows below and above, voxels
  const float ylo = fmaxf(ay - slack, 0.0f), yhi = fmaxf(1.0f - ay - slack, 0.0f);
  const float zlo = fmaxf(az - slack, 0.0f), zhi = fmaxf(1.0f - az - slack, 0.0f);
  bool found = false;
  float best = 0.0f;
  int best_idx = 0x7fffffff, best_slot = -1;
  float4 best_pt = make_float4(0.f, 0.f, 0.f, 0.f);
  float bestv = 3.0e38f;  // best in voxel units, squared (row pruning)
  const float inv2 = g.inv_leaf * g.inv_leaf;
  if (guess_slot >= 0 && guess_slot < g.n) {
    const float4 p = g.pts[guess_slot];
    const float d2 = em::dist2_3(qx, qy, qz, p.x, p.y, p.z);
    if ((double)d2 <= bound) {
      found = true;
      best = d2;
      best_idx = g.orig ? g.orig[guess_slot] : guess_slot;
      best_slot = guess_slot;
      best_pt = p;
      bestv = d2 * inv2 * 1.0001f + 1e-4f;
    }
  }
  int rs[9], re[9];
  const int xlo = max(vx - 1, 0), xhi = min(vx + 1, g.div_v[0] - 1);
  const bool x_ok = xlo <= xhi;
#pragma unroll
  for (int t = 0; t < 9; ++t) {
    const int cz = vz + t / 3 - 1, cy = vy + t % 3 - 1;
    rs[t] = 0;
    re[t] = 0;
    if (x_ok && cz >= 0 && cz < g.div_v[2] && cy >= 0 && cy < g.div_v[1]) {
      const int base = (cz * g.dim[1] + cy) * g.dim[0];
      rs[t] = __ldg(&g.cell_start[base + xlo]);
      re[t] = __ldg(&g.cell_start[base + xhi + 1]);
    }
  }
#pragma unroll
  for (int t = 0; t < 9; ++t) {
    const int dz = t / 3 - 1, dy = t % 3 - 1;
    const float zd = dz < 0 ? zlo : (dz > 0 ? zhi : 0.0f);
    const float yd = dy < 0 ? ylo : (dy > 0 ? yhi : 0.0f);
    if (zd * zd + yd * yd > bestv) continue;
    for (int k = rs[t]; k < re[t]; ++k) {
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
        bestv = d2 * inv2 * 1.0001f + 1e-4f;
      }
    }
  }
  const float outside = fmaxf(1.0f - slack, 0.0f);  // least gap to a point outside the block, voxels
  *certain = found && best * inv2 < 0.999f * outside * outside;
  *out_idx = best_idx;
  *out_d2 = best;
  *out_pt = best_pt;
  *out_slot = found ? best_slot : -1;
  return found;
}

// Bounded nearest neighbour for the IB queries of one tile, in three block-wide phases so that the warps stay converged:
//   1. thread per query: the reach grid answers "nothing within the bound" for queries far from the target, the 27-voxel
//      block answers queries that lie on the target surface (the common case once two clouds are roughly aligned);
//   2. the queries neither could settle are compacted into a shared-memory list and served by WHOLE WARPS, one query per
//      warp at a time: the 32 lanes resolve the (z, y) rows of the query's window in parallel and test 32 candidates per
//      step (warp_radius_unordered), the window bounded by what phase 1 learned (reach-grid upper bound, or the best
//      point of the block).  In the thread-per-query search these few long-running queries kept whole warps busy at
//      6-12 active lanes of 32 (ncu, round 2);
//   3. every thread picks up its result.
// The result is the same as an exhaustive search: the nearest point by (d^2, original index) among those with d^2 <= bound.
struct TileNn {
  float4 q[IB];   // x, y, z, search radius^2 of the queries handed to phase 2
  int todo[IB];        // small windows
  int todo_large[IB];  // large windows
  float res_d2[IB];
  int res_slot[IB];
  int n_todo, n_todo_large;
};

__device__ __forceinline__ bool tile_nearest(TileNn& sh, const GridView& g, const ReachView& r, bool live, float qx, float qy, float qz,
                                             double bound, int guess_slot, float* out_d2, float4* out_pt, int* out_slot)
{
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  if (tid == 0) {
    sh.n_todo = 0;
    sh.n_todo_large = 0;
  }
  __syncthreads();
  bool hit = false, pending = false;
  float d2 = 0.f;
  int slot = -1;
  float4 pt = make_float4(0.f, 0.f, 0.f, 0.f);
  if (live) {
    float r2 = (float)bound;  // radius^2 phase 2 would have to search
    bool rejected = false, block_has_points = true;
    // the reach grid's bounds and phase 2's row bounds count whole cells; the true gaps may be short of them by the
    // rounding slack on each axis, at most 2 * slack along any direction
    const float slack2 = 2.0f * voxel_slack(qx * g.inv_leaf, qy * g.inv_leaf, qz * g.inv_leaf);
    if (r.lb2) {
      int lb2 = 0;
      const float bound_v = (float)bound * g.inv_leaf * g.inv_leaf;  // bound in voxel units, squared
      const bool inside = reach_lookup(g, r, qx, qy, qz, &lb2);
      // outside the grid: farther than the margin from every occupied voxel, i.e. lower bound >= none
      // (sqrt(lb) - slack2)^2 >= lb - slack2 * (lb + 1), as 2 sqrt(lb) <= lb + 1
      const float lb = inside ? (float)lb2 : (float)r.none;
      if (lb - slack2 * (lb + 1.0f) > bound_v * 1.001f + 0.01f) rejected = true;
      if (inside && lb2 < r.none) {
        const float ub = sqrtf((float)lb2) + 3.4642f + slack2;  // + twice the voxel diagonal
        r2 = fminf(r2, (ub * ub * 1.001f + 0.01f) * g.leaf * g.leaf);
      }
      block_has_points = inside && lb2 == 0;  // lower bound 0 <=> an occupied voxel inside the 3 x 3 x 3 block
      // A query off the surface: the voxel diagonal slack above makes the window (and with it the number of rows and
      // candidates phase 2 has to touch) 2-3x larger than necessary.  Walking downhill on the reach grid finds a REAL target
      // point nearby in a few steps; its distance is the tightest radius one can ask for without knowing the answer.
      if (!rejected && inside && lb2 > 0 && lb2 < r.none && guess_slot < 0 && g.shift[0] == 0 && g.shift[1] == 0 && g.shift[2] == 0) {
        int cx = floor_to_int(qx * g.inv_leaf) - g.min_b[0] - r.org[0];
        int cy = floor_to_int(qy * g.inv_leaf) - g.min_b[1] - r.org[1];
        int cz = floor_to_int(qz * g.inv_leaf) - g.min_b[2] - r.org[2];
        if (reach_descend(r, cx, cy, cz, lb2)) {
          const float dd = block27_any(g, cx + r.org[0], cy + r.org[1], cz + r.org[2], qx, qy, qz);
          if (dd < 3.0e38f) r2 = fminf(r2, dd);
        }
      }
    }
    if (!rejected) {
      bool certain = false;
      if ((block_has_points || guess_slot >= 0) && g.shift[0] == 0 && g.shift[1] == 0 && g.shift[2] == 0) {
        int idx;
        hit = nearest_block27(g, qx, qy, qz, bound, guess_slot, &idx, &d2, &pt, &slot, &certain);
        if (hit) r2 = fminf(r2, d2);  // phase 2 only has to look for something at least as close
      }
      if (!certain) {
        pending = true;
        hit = false;
        // strict < inside the walk: widen by a hair; and by the slack, which the walk's whole-cell row bounds do not have
        const float rw = sqrtf(r2 * 1.00001f + 1e-12f) + slack2 * g.leaf;
        const float r2w = rw * rw;
        sh.q[tid] = make_float4(qx, qy, qz, r2w);
        if (r2w * g.inv_leaf * g.inv_leaf <= 12.25f) sh.todo[atomicAdd(&sh.n_todo, 1)] = tid;  // radius <= 3.5 voxels: at most 11 x 11 rows
        else sh.todo_large[atomicAdd(&sh.n_todo_large, 1)] = tid;
      }
    }
  }
  __syncthreads();
  // phase 2: small windows (a few dozen rows: queries near the target surface) by groups of 8 lanes, four queries per warp
  // at a time; large windows (queries up to the correspondence distance away from the target) by whole warps
  const int n_small = sh.n_todo, n_large = sh.n_todo_large;
  auto serve = [&](auto G_, int who, unsigned gmask, int glane) {
    constexpr int G = decltype(G_)::value;
    const float4 q = sh.q[who];
    const int rv = (int)ceilf(sqrtf(q.w) * g.inv_leaf) + 1;
    float bd = 3.0e38f;
    int bi = 0x7fffffff, bs = -1;
    group_radius_unordered<G>(g, gmask, glane, q.x, q.y, q.z, q.w, rv, [&](bool valid, int k, const float4&, float dd) {
      if (valid && (double)dd <= bound) {
        const int oi = g.orig ? g.orig[k] : k;
        if (dd < bd || (dd == bd && oi < bi)) {
          bd = dd;
          bi = oi;
          bs = k;
        }
      }
    });
#pragma unroll
    for (int o = G / 2; o > 0; o >>= 1) {
      const float od = __shfl_xor_sync(gmask, bd, o, G);
      const int oi = __shfl_xor_sync(gmask, bi, o, G);
      const int os = __shfl_xor_sync(gmask, bs, o, G);
      if (od < bd || (od == bd && oi < bi)) {
        bd = od;
        bi = oi;
        bs = os;
      }
    }
    if (glane == 0) {
      sh.res_d2[who] = bd;
      sh.res_slot[who] = bs;
    }
  };
  {
    const int grp = tid >> 3, glane = tid & 7;
    const unsigned gmask = 0xffu << (lane & 24);
    for (int t = grp; t < n_small; t += IB / 8) serve(std::integral_constant<int, 8>(), sh.todo[t], gmask, glane);
  }
  __syncwarp();
  for (int t = warp; t < n_large; t += IB / 32) serve(std::integral_constant<int, 32>(), sh.todo_large[t], 0xffffffffu, lane);
  __syncthreads();
  if (pending) {
    slot = sh.res_slot[tid];
    hit = slot >= 0;
    if (hit) {
      d2 = sh.res_d2[tid];
      pt = g.pts[slot];
    }
  }
  *out_d2 = d2;
  *out_pt = pt;
  *out_slot = hit ? slot : -1;
  return hit;
}

// ---------------------------------------------------------------- ICP
__global__ void __launch_bounds__(256) icp_init_kernel(const IcpJob* __restrict__ jobs)
{
  const IcpJob& j = jobs[blockIdx.y];
  for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < j.ns; i += gridDim.x * blockDim.x) {
    const float4 p = j.src[i];
    float4 o;
    em::transform_point(j.t0, p.x, p.y, p.z, &o.x, &o.y, &o.z);  // pcl::transformPointCloud(source, initial_guess)
    o.w = p.w;
    j.work[i] = o;
    j.nn_slot[i] = -1;
  }
}

__device__ __forceinline__ void block_accumulate(long long* vals, int nvals, long long* gsums)
{
  __shared__ long long sh[IB / 32][NSUM];
  const int lane = threadIdx.x & 31, w = threadIdx.x >> 5;
  __syncthreads();  // the previous tile's readers are done with sh
  for (int k = 0; k < nvals; ++k) {
    const long long v = warp_sum_ll(vals[k]);
    if (lane == 0) sh[w][k] = v;
  }
  __syncthreads();
  if (threadIdx.x < nvals) {
    long long s = 0;
    for (int ww = 0; ww < IB / 32; ++ww) s += sh[ww][threadIdx.x];
    if (s != 0) atomicAdd((unsigned long long*)&gsums[threadIdx.x], (unsigned long long)s);
  }
}

__device__ void mat4_mul(const float* a, const float* b, float* r)
{
  for (int i = 0; i < 4; ++i)
    for (int c = 0; c < 4; ++c) {
      float acc = a[i * 4 + 0] * b[0 * 4 + c];
      acc += a[i * 4 + 1] * b[1 * 4 + c];
      acc += a[i * 4 + 2] * b[2 * 4 + c];
      acc += a[i * 4 + 3] * b[3 * 4 + c];
      r[i * 4 + c] = acc;
    }
}

// Umeyama from the finished reductions, transform update and pcl::registration::DefaultConvergenceCriteria for one pair;
// runs on one thread of the LAST tile of that pair to finish
__device__ void icp_solve(const IcpJob& j, int max_iterations, double rotation_threshold, double translation_threshold, int max_log,
                          int* n_active)
{
  IcpState& st = *j.st;
  long long s[NSUM];
  for (int k = 0; k < NSUM; ++k) {
    s[k] = (long long)atomicExch((unsigned long long*)&j.sums[k], 0ull);  // read the other tiles' atomics, reset for the next iteration
  }
  if (j.sums_log && st.iterations < max_log)
    for (int k = 0; k < NSUM; ++k) j.sums_log[(size_t)st.iterations * NSUM + k] = s[k];
  const long long cnt = s[0];
  if (cnt < 3) {  // "Not enough correspondences found": stop, not converged
    st.active = 0;
    st.converged = 0;
    __threadfence();
    atomicSub(n_active, 1);
    return;
  }
  const double n = (double)cnt;
  double pm[3], qm[3];
  for (int a = 0; a < 3; ++a) {
    pm[a] = ((double)s[1 + a] / MM3D_FIX1_SCALE) / n;
    qm[a] = ((double)s[4 + a] / MM3D_FIX1_SCALE) / n;
  }
  float sigma[9], pmf[3], qmf[3];
  for (int a = 0; a < 3; ++a) {
    pmf[a] = (float)pm[a];
    qmf[a] = (float)qm[a];
    for (int b = 0; b < 3; ++b) sigma[a * 3 + b] = (float)(((double)s[7 + a * 3 + b] / MM3D_FIX2_SCALE) / n - qm[a] * pm[b]);
  }
  float T[16];
  em::umeyama_from_sigma<float>(sigma, pmf, qmf, T);
  float nf[16];
  mat4_mul(T, st.final_t, nf);
  for (int k = 0; k < 16; ++k) {
    st.final_t[k] = nf[k];
    st.step[k] = T[k];
  }
  st.iterations += 1;
  // pcl::registration::DefaultConvergenceCriteria::hasConverged
  bool conv = false;
  if (st.iterations >= max_iterations) {
    conv = true;
  } else {
    const double cos_angle = 0.5 * (double)(T[0] + T[5] + T[10] - 1);
    const double translation_sqr = (double)(T[3] * T[3] + T[7] * T[7] + T[11] * T[11]);
    if (cos_angle >= rotation_threshold && translation_sqr <= translation_threshold) {
      conv = true;
    } else {
      const double mse = ((double)s[16] / MM3D_FIXD_SCALE) / n;
      if (fabs(mse - st.prev_mse) < 1e-12) conv = true;
      else st.prev_mse = mse;
    }
  }
  if (conv) {
    st.active = 0;
    st.converged = 1;
    __threadfence();
    atomicSub(n_active, 1);
  } else {
    __threadfence();             // the new step transform is visible before the next iteration's tiles are handed out
    atomicExch(j.next_tile, 0);  // re-open the pair
  }
}

// One 128-query tile of one pair in the current iteration.  Data that other blocks wrote in an earlier iteration (work,
// nn_slot, the step transform) is read through L2 (__ldcg): L1 is not coherent between SMs.
__device__ __forceinline__ void icp_tile(const IcpJob& j, int tile, double max_dist_sqr, int rv, int max_iterations,
                                         double rotation_threshold, double translation_threshold, int max_log, int* n_active)
{
  __shared__ float s_step[16];
  __shared__ int s_apply;
  __shared__ TileNn nn;
  __syncthreads();
  if (threadIdx.x < 16) s_step[threadIdx.x] = __ldcg(&j.st->step[threadIdx.x]);
  if (threadIdx.x == 16) s_apply = __ldcg(&j.st->iterations) > 0 ? 1 : 0;  // iterations completed so far = index of this one
  __syncthreads();
  const int apply_step = s_apply;
  long long v[NSUM];
#pragma unroll
  for (int k = 0; k < NSUM; ++k) v[k] = 0;
  const int i = tile * IB + threadIdx.x;
  const bool live = i < j.ns;
  float4 p = make_float4(0.f, 0.f, 0.f, 0.f);
  int guess = -1;
  if (live) {
    p = __ldcg(&j.work[i]);
    if (apply_step) {  // transformCloud(input_transformed, input_transformed, transformation_) of the previous iteration
      float4 o;
      em::transform_point(s_step, p.x, p.y, p.z, &o.x, &o.y, &o.z);
      o.w = p.w;
      p = o;
      j.work[i] = p;
    }
    guess = __ldcg(&j.nn_slot[i]);
  }
  float d2;
  float4 q;
  int slot;
  const bool hit = tile_nearest(nn, j.tgt, j.reach, live, p.x, p.y, p.z, max_dist_sqr, guess, &d2, &q, &slot);
  if (live) {
    j.nn_slot[i] = slot;  // the transform moves little between iterations: last iteration's match seeds the next search
    if (hit) {
      const double pp[3] = {(double)p.x, (double)p.y, (double)p.z};
      const double qq[3] = {(double)q.x, (double)q.y, (double)q.z};
      v[0] = 1;
#pragma unroll
      for (int a = 0; a < 3; ++a) {
        v[1 + a] = em::to_fix(pp[a], MM3D_FIX1_SCALE);
        v[4 + a] = em::to_fix(qq[a], MM3D_FIX1_SCALE);
#pragma unroll
        for (int b = 0; b < 3; ++b) v[7 + a * 3 + b] = em::to_fix(qq[a] * pp[b], MM3D_FIX2_SCALE);
      }
      v[16] = em::to_fix((double)d2, MM3D_FIXD_SCALE);
    }
  }
  block_accumulate(v, NSUM, j.sums);
  // last tile of this pair: solve + convergence test
  __syncthreads();
  if (threadIdx.x == 0) {
    __threadfence();
    const int ntiles = (j.ns + IB - 1) / IB;
    const int ticket = atomicAdd(j.ticket, 1);
    if (ticket == ntiles - 1) {
      *j.ticket = 0;
      __threadfence();
      icp_solve(j, max_iterations, rotation_threshold, translation_threshold, max_log, n_active);
    }
  }
}

__global__ void __launch_bounds__(IB) icp_persistent_kernel(const IcpJob* __restrict__ jobs, int n_jobs, IcpLoop* loop, double max_dist_sqr,
                                                            int rv, int max_iterations, double rotation_threshold,
                                                            double translation_threshold, int max_log)
{
  __shared__ int s_pair, s_tile;
  int cur = 0;  // all blocks walk the job list (sorted by target) from the front: neighbouring blocks share a target's tables in L2
  for (;;) {
    if (threadIdx.x == 0) {
      int pair = -1, tile = -1, scanned = 0;
      while (__ldcg(&loop->n_active) > 0) {
        const IcpJob& j = jobs[cur];
        if (__ldcg(j.next_tile) < j.n_tiles) {  // cheap look before the atomic; a stale value only costs one wasted increment
          const int t = atomicAdd(j.next_tile, 1);
          if (t < j.n_tiles) {
            __threadfence();  // what the previous iteration's tiles and its solver wrote is visible to this tile
            pair = cur;
            tile = t;
            break;
          }
        }
        cur = cur + 1 == n_jobs ? 0 : cur + 1;
        if (++scanned >= n_jobs) {  // nothing to hand out right now: the remaining pairs are between two iterations
          scanned = 0;
          __nanosleep(500);
        }
      }
      s_pair = pair;
      s_tile = tile;
    }
    __syncthreads();
    const int pair = s_pair, tile = s_tile;
    if (pair < 0) break;
    icp_tile(jobs[pair], tile, max_dist_sqr, rv, max_iterations, rotation_threshold, translation_threshold, max_log, &loop->n_active);
    __syncthreads();
  }
}

// ---------------------------------------------------------------- score
struct ScoreJob {
  GridView tgt;
  ReachView reach;
  const float4* src;
  int ns;
  float t[16];
  long long* sums;  // Sd, nr
  const int* nn_guess;  // optional: the slots matched in the last ICP iteration
};

__global__ void __launch_bounds__(IB) score_kernel(const ScoreJob* __restrict__ jobs, double max_range, int rv)
{
  const ScoreJob& j = jobs[blockIdx.y];
  if (blockIdx.x * IB >= j.ns) return;
  __shared__ TileNn nn;
  long long v[2] = {0, 0};
  const int i = blockIdx.x * IB + threadIdx.x;
  const bool live = i < j.ns;
  float x = 0.f, y = 0.f, z = 0.f;
  if (live) {
    const float4 p = j.src[i];
    em::transform_point(j.t, p.x, p.y, p.z, &x, &y, &z);
  }
  float d2;
  float4 q;
  int slot;
  // the reference compares the squared distance with the plain range
  if (tile_nearest(nn, j.tgt, j.reach, live, x, y, z, max_range, (live && j.nn_guess) ? j.nn_guess[i] : -1, &d2, &q, &slot)) {
    v[0] = em::to_fix((double)d2, MM3D_FIXD_SCALE);
    v[1] = 1;
  }
  block_accumulate(v, 2, j.sums);
}

ReachView no_reach()
{
  ReachView r;
  memset(&r, 0, sizeof(r));
  return r;
}

}  // namespace

void build_reach_batch(Ctx& c, const std::vector<DIndex>& idx, int margin, std::vector<DReach>& out)
{
  const int M = (int)idx.size();
  out.clear();
  out.resize(M);
  margin = std::max(2, std::min(margin, 15));
  std::vector<ReachJob> jobs;
  std::vector<DBuf<unsigned char>> ping(M);
  size_t max_cells = 0;
  int max_n = 0;
  for (int m = 0; m < M; ++m) {
    out[m].v = no_reach();
    const GridView& g = idx[m].v;
    if (g.n <= 0 || g.div_v[0] <= 0) continue;
    ReachView r = no_reach();
    size_t cells = 1;
    for (int k = 0; k < 3; ++k) {
      r.org[k] = -margin;
      r.dim[k] = g.div_v[k] + 2 * margin;
      cells *= (size_t)r.dim[k];
    }
    if (cells > ((size_t)1 << 30)) continue;  // absurdly sparse cloud: search without the grid
    r.none = std::min(255, margin * margin);
    out[m].lb2.alloc(c, cells);
    ping[m].alloc(c, cells);
    MM_CUDA(cudaMemsetAsync(ping[m].p, 255, cells, c.stream));
    r.lb2 = out[m].lb2.p;
    out[m].v = r;
    jobs.push_back(ReachJob{g, r, ping[m].p, out[m].lb2.p});
    max_cells = std::max(max_cells, cells);
    max_n = std::max(max_n, g.n);
  }
  if (jobs.empty()) return;
  DBuf<ReachJob> dj = to_device(c, jobs);
  const unsigned nj = (unsigned)jobs.size();
  MM_LAUNCH(c, reach_mark_kernel, dim3(std::max(1, std::min((max_n + 255) / 256, 148 * 4)), nj), 256, 0, dj.p);
  const unsigned blocks = (unsigned)std::min<size_t>((max_cells + 255) / 256, 148 * 16);
  // x: ping -> lb2, y: lb2 -> ping, z: ping -> lb2
  double bytes = 0;
  for (const ReachJob& j : jobs) bytes += 2.0 * j.r.dim[0] * j.r.dim[1] * j.r.dim[2];
  MM_BYTES(c, bytes);
  MM_LAUNCH(c, reach_pass_kernel, dim3(blocks, nj), 256, 0, dj.p, 0, margin, 1);
  MM_BYTES(c, bytes);
  MM_LAUNCH(c, reach_pass_kernel, dim3(blocks, nj), 256, 0, dj.p, 1, margin, 0);
  MM_BYTES(c, bytes);
  MM_LAUNCH(c, reach_pass_kernel, dim3(blocks, nj), 256, 0, dj.p, 2, margin, 1);
}

void icp_batch(Ctx& c, const std::vector<CloudView>& clouds, const std::vector<DIndex>& idx, const std::vector<DReach>& reach,
               const std::vector<PairJob>& jobs, const std::vector<const float*>& T0, double max_dist, int max_it, double eps,
               std::vector<IcpOut>& out, std::vector<std::vector<long long>>* sums_dbg, IcpNeighbours* nn_keep)
{
  const int P = (int)jobs.size();
  out.assign(P, IcpOut());
  if (nn_keep) nn_keep->offset.assign(P, -1);
  if (sums_dbg) { sums_dbg->clear(); sums_dbg->resize(P); }
  if (P == 0) return;
  const int max_log = sums_dbg ? 64 : 0;
  // A zero initial guess (failed RANSAC) stays zero through ICP: final * 0 == 0 (matching.cpp:220).
  std::vector<int> act;
  for (int p = 0; p < P; ++p) {
    bool zero = true;
    for (int k = 0; k < 16; ++k)
      if (T0[p][k] != 0.0f) zero = false;
    if (zero) {
      for (int k = 0; k < 16; ++k) out[p].T[k] = 0.0f;
      out[p].iterations = 0;
      out[p].converged = 0;
    } else {
      act.push_back(p);
    }
  }
  const int A = (int)act.size();
  if (A == 0) return;
  // Pairs that share a target run back to back: the blocks all start at the first job and move on together, so at any time
  // only a few targets' tables (cell starts, reach grid, points: ~17 MB per 250 k-point map) are live and stay in L2.  In
  // row-major pair order the 32 targets of config 3 (550 MB of tables) were revisited round-robin — a DRAM-latency-bound
  // gather.
  std::stable_sort(act.begin(), act.end(), [&](int x, int y) { return jobs[x].b < jobs[y].b; });
  size_t tot = 0;
  int mx = 0;
  for (int a = 0; a < A; ++a) {
    tot += (size_t)clouds[jobs[act[a]].a].n;
    mx = std::max(mx, clouds[jobs[act[a]].a].n);
  }
  DBuf<float4> work(c, tot + 1);
  DBuf<int> nn_local;
  DBuf<int>& nn = nn_keep ? nn_keep->slots : nn_local;
  nn.alloc(c, tot + 1);
  DBuf<long long> sums(c, (size_t)A * NSUM);
  sums.zero(c);
  DBuf<int> tickets(c, A);
  tickets.zero(c);
  DBuf<long long> slog;
  if (max_log) {
    slog.alloc(c, (size_t)A * max_log * NSUM);
    slog.zero(c);
  }
  std::vector<IcpState> hst(A);
  for (int a = 0; a < A; ++a) {
    memset(&hst[a], 0, sizeof(IcpState));
    for (int k = 0; k < 16; ++k) hst[a].final_t[k] = hst[a].step[k] = (k % 5 == 0) ? 1.f : 0.f;
    hst[a].prev_mse = 1.7976931348623157e308;
    // an empty source has no tile, so nothing would ever retire the pair: it starts out finished and not converged
    // ("Not enough correspondences found", the transform stays the initial guess)
    hst[a].active = clouds[jobs[act[a]].a].n > 0 ? 1 : 0;
  }
  DBuf<IcpState> dst = to_device(c, hst);
  std::vector<IcpJob> ij(A);
  size_t off = 0;
  for (int a = 0; a < A; ++a) {
    const PairJob& pj = jobs[act[a]];
    ij[a].tgt = idx[pj.b].v;
    ij[a].reach = pj.b < (int)reach.size() ? reach[pj.b].v : no_reach();
    ij[a].src = clouds[pj.a].pts;
    ij[a].ns = clouds[pj.a].n;
    ij[a].work = work.p + off;
    ij[a].nn_slot = nn.p + off;
    if (nn_keep) nn_keep->offset[act[a]] = (long long)off;
    ij[a].sums = sums.p + (size_t)a * NSUM;
    ij[a].st = dst.p + a;
    ij[a].ticket = tickets.p + a;
    for (int k = 0; k < 16; ++k) ij[a].t0[k] = T0[act[a]][k];
    ij[a].sums_log = max_log ? slog.p + (size_t)a * max_log * NSUM : nullptr;
    off += (size_t)ij[a].ns;
  }
  // per-pair tile counters: open (0) for every pair with a non-empty source, closed otherwise
  std::vector<int> hnext(A, 0);
  IcpLoop hl;
  memset(&hl, 0, sizeof(hl));
  int tiles = 0;
  double bytes = 0;
  for (int a = 0; a < A; ++a) {
    ij[a].n_tiles = (ij[a].ns + IB - 1) / IB;
    if (hst[a].active) {  // at least one iteration runs whatever max_iterations says (PCL's do-while)
      hl.n_active += 1;
      tiles += ij[a].n_tiles;
      bytes += 16.0 * (2.0 * ij[a].ns + ij[a].tgt.n);
    } else {
      hnext[a] = ij[a].n_tiles;
    }
  }
  DBuf<int> dnext = to_device(c, hnext);
  for (int a = 0; a < A; ++a) ij[a].next_tile = dnext.p + a;
  DBuf<IcpJob> dij = to_device(c, ij);
  DBuf<IcpLoop> dloop(c, 1);
  dloop.upload(c, &hl, 1);
  const int iblocks = std::max(1, std::min((mx + 255) / 256, 148 * 8));
  MM_LAUNCH(c, icp_init_kernel, dim3(iblocks, A), 256, 0, dij.p);
  const double max_dist_sqr = max_dist * max_dist;
  const float leaf = idx[jobs[act[0]].b].v.leaf;
  const int rv = (int)std::ceil(max_dist / (double)leaf) + 1;
  if (hl.n_active > 0) {
    // persistent launch: as many blocks as can be resident (blocks that find no pair active exit at once)
    int dev = 0, sms = 0, per_sm = 0;
    MM_CUDA(cudaGetDevice(&dev));
    MM_CUDA(cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev));
    MM_CUDA(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, icp_persistent_kernel, IB, 0));
    const int grid = std::max(1, std::min(sms * std::max(per_sm, 1), tiles));
    MM_BYTES(c, bytes);  // one sweep of every active pair; later iterations repeat it for the pairs still active
    MM_LAUNCH(c, icp_persistent_kernel, grid, IB, 0, dij.p, A, dloop.p, max_dist_sqr, rv, max_it, 1.0 - eps, eps, max_log);
  }
  dst.download(c, hst.data(), A);
  std::vector<long long> hlog;
  if (max_log) {
    hlog.resize((size_t)A * max_log * NSUM);
    slog.download(c, hlog.data(), hlog.size());
  }
  c.sync();
  for (int a = 0; a < A; ++a) {
    IcpOut& o = out[act[a]];
    // icp.getFinalTransformation() * initial_guess
    const float* f = hst[a].final_t;
    const float* g = T0[act[a]];
    for (int i = 0; i < 4; ++i)
      for (int cc = 0; cc < 4; ++cc) {
        float acc = f[i * 4 + 0] * g[0 * 4 + cc];
        acc += f[i * 4 + 1] * g[1 * 4 + cc];
        acc += f[i * 4 + 2] * g[2 * 4 + cc];
        acc += f[i * 4 + 3] * g[3 * 4 + cc];
        o.T[i * 4 + cc] = acc;
      }
    o.iterations = hst[a].iterations;
    o.converged = hst[a].converged;
    if (sums_dbg) {
      const int nl = std::min(hst[a].iterations + (hst[a].converged ? 0 : 1), max_log);
      (*sums_dbg)[act[a]].assign(hlog.begin() + (size_t)a * max_log * NSUM, hlog.begin() + ((size_t)a * max_log + nl) * NSUM);
    }
  }
}

void score_batch(Ctx& c, const std::vector<CloudView>& clouds, const std::vector<DIndex>& idx, const std::vector<DReach>& reach,
                 const std::vector<PairJob>& jobs, const std::vector<const float*>& T, double max_range, std::vector<double>& scores,
                 const IcpNeighbours* nn_guess)
{
  const int P = (int)jobs.size();
  scores.assign(P, 1.7976931348623157e308);
  if (P == 0) return;
  DBuf<long long> sums(c, (size_t)P * 2);
  sums.zero(c);
  std::vector<ScoreJob> sj(P);
  int mx = 0;
  // launch order = by target (blockIdx.y): the pairs of one target are scored back to back, its tables stay in L2
  std::vector<int> ord(P);
  for (int p = 0; p < P; ++p) ord[p] = p;
  std::stable_sort(ord.begin(), ord.end(), [&](int x, int y) { return jobs[x].b < jobs[y].b; });
  for (int q = 0; q < P; ++q) {
    const int p = ord[q];
    sj[q].tgt = idx[jobs[p].b].v;
    sj[q].reach = jobs[p].b < (int)reach.size() ? reach[jobs[p].b].v : no_reach();
    sj[q].src = clouds[jobs[p].a].pts;
    sj[q].ns = clouds[jobs[p].a].n;
    for (int k = 0; k < 16; ++k) sj[q].t[k] = T[p][k];
    sj[q].sums = sums.p + (size_t)p * 2;
    sj[q].nn_guess = (nn_guess && p < (int)nn_guess->offset.size() && nn_guess->offset[p] >= 0) ? nn_guess->slots.p + nn_guess->offset[p] : nullptr;
    mx = std::max(mx, sj[q].ns);
  }
  if (mx == 0) return;
  DBuf<ScoreJob> dsj = to_device(c, sj);
  const float leaf = idx[jobs[0].b].v.leaf;
  const int rv = (int)std::ceil(std::sqrt(std::max(max_range, 0.0)) / (double)leaf) + 1;
  { double b = 0; for (int p = 0; p < P; ++p) b += 16.0 * ((double)sj[p].ns + sj[p].tgt.n); MM_BYTES(c, b); }
  MM_LAUNCH(c, score_kernel, dim3((mx + IB - 1) / IB, P), IB, 0, dsj.p, max_range, rv);
  std::vector<long long> h((size_t)P * 2);
  sums.download(c, h.data(), h.size());
  c.sync();
  for (int p = 0; p < P; ++p)
    if (h[2 * p + 1] > 0) scores[p] = ((double)h[2 * p] / MM3D_FIXD_SCALE) / (double)h[2 * p + 1];
}

}  // namespace mm3d
