// matching.cu — per-pair descriptor matching and RANSAC (all pairs per launch).
//   K9  reciprocal k-NN cross-matching  <- map_merge_3d/src/matching.cpp:31-93 (the reference's own algorithm;
//       pcl::search::KdTree<DescriptorT> == exact L2 k-NN, flann::L2_Simple accumulation order)
//   K10 RANSAC + final SVD              <- src/matching.cpp:110-140
//       (pcl::registration::CorrespondenceRejectorSampleConsensus, pcl::RandomSampleConsensus,
//        pcl::SampleConsensusModelRegistration, boost::mt19937(12345))
#include <algorithm>
#include <cmath>
#include <cstdlib>
#include <cstring>
#include <string>

#include "mm3d_internal.cuh"

namespace mm3d {

namespace {

constexpr int KMAX = 16;

struct KnnJob {
  const float* A;
  int na;
  const float* B;
  int nb;
  int k;
  int* idx;     // na x k
  float* dist;  // na x k
};

// Exact FP32 k-NN of every row of A among the rows of B.  One thread owns one query row (registers); B
// streams through shared memory stored dimension-major, so one 128-bit broadcast load feeds the same
// dimension of four B rows.  Distances accumulate dimension by dimension without contraction, like
// flann::L2_Simple; ties keep the lower index.  The running top-K lives in registers (K is a template
// parameter, insertion is a fully unrolled compare/select chain).
template <int D, int K>
__global__ void __launch_bounds__(128) knn_small_kernel(const KnnJob* __restrict__ jobs)
{
  constexpr int TB = 64;
  __shared__ __align__(16) float sb[D * TB];
  const KnnJob j = jobs[blockIdx.y];
  if (blockIdx.x * blockDim.x >= j.na) return;
  const int row = blockIdx.x * blockDim.x + threadIdx.x;
  const bool live = row < j.na;
  float a[D];
#pragma unroll
  for (int t = 0; t < D; ++t) a[t] = live ? j.A[(size_t)row * D + t] : 0.f;
  float bd[K];
  int bi[K];
#pragma unroll
  for (int t = 0; t < K; ++t) {
    bd[t] = __int_as_float(0x7f800000);  // +inf
    bi[t] = -1;
  }
  for (int base = 0; base < j.nb; base += TB) {
    const int tb = min(TB, j.nb - base);
    __syncthreads();
    for (int e = threadIdx.x; e < TB * D; e += blockDim.x) {
      const int r = e / D, t = e - r * D;  // coalesced global read, transposed shared write
      sb[t * TB + r] = (r < tb) ? j.B[(size_t)(base + r) * D + t] : 0.f;
    }
    __syncthreads();
    if (!live) continue;
    for (int r0 = 0; r0 < tb; r0 += 4) {
      float acc0 = 0.f, acc1 = 0.f, acc2 = 0.f, acc3 = 0.f;
#pragma unroll
      for (int t = 0; t < D; ++t) {
        const float4 b = *reinterpret_cast<const float4*>(&sb[t * TB + r0]);
        const float d0 = a[t] - b.x, d1 = a[t] - b.y, d2 = a[t] - b.z, d3 = a[t] - b.w;
        acc0 += d0 * d0;
        acc1 += d1 * d1;
        acc2 += d2 * d2;
        acc3 += d3 * d3;
      }
      const float accs[4] = {acc0, acc1, acc2, acc3};
#pragma unroll
      for (int u = 0; u < 4; ++u) {
        const float acc = accs[u];
        if (r0 + u < tb && acc < bd[K - 1]) {
          const int id = base + r0 + u;
#pragma unroll
          for (int t = K - 1; t >= 1; --t) {
            const bool up = acc < bd[t - 1];
            const bool here = !up && acc < bd[t];
            bd[t] = up ? bd[t - 1] : (here ? acc : bd[t]);
            bi[t] = up ? bi[t - 1] : (here ? id : bi[t]);
          }
          if (acc < bd[0]) {
            bd[0] = acc;
            bi[0] = id;
          }
        }
      }
    }
  }
  if (live) {
#pragma unroll
    for (int t = 0; t < K; ++t) {
      j.idx[(size_t)row * K + t] = bi[t];
      j.dist[(size_t)row * K + t] = bi[t] >= 0 ? bd[t] : 0.f;
    }
  }
}

// Any dimension (PFH 125 ... SHOT 1344): a block owns 64 query rows and a tile of
// 32 B rows; the dimension loop runs in chunks staged through shared memory while
// each thread keeps the running sums for (its row) x (16 of the 32 B rows).
__global__ void __launch_bounds__(128) knn_generic_kernel(const KnnJob* __restrict__ jobs, int D)
{
  constexpr int QA = 64, TB = 32, DC = 32;
  __shared__ float sa[QA][DC + 1];
  __shared__ float sbm[TB][DC + 1];
  __shared__ float sd[QA][TB + 1];
  const KnnJob j = jobs[blockIdx.y];
  const int row0 = blockIdx.x * QA;
  if (row0 >= j.na) return;
  const int q = threadIdx.x & (QA - 1);  // query row within the block
  const int half = threadIdx.x >> 6;     // which 16 B rows
  const int row = row0 + q;
  float bd[KMAX];
  int bi[KMAX];
  int cnt = 0;
  const int k = j.k;
  for (int base = 0; base < j.nb; base += TB) {
    float acc[TB / 2];
#pragma unroll
    for (int r = 0; r < TB / 2; ++r) acc[r] = 0.f;
    for (int d0 = 0; d0 < D; d0 += DC) {
      const int dc = min(DC, D - d0);
      __syncthreads();
      for (int e = threadIdx.x; e < QA * DC; e += blockDim.x) {
        const int rr = e / DC, dd = e - rr * DC;
        sa[rr][dd] = (row0 + rr < j.na && dd < dc) ? j.A[(size_t)(row0 + rr) * D + d0 + dd] : 0.f;
      }
      for (int e = threadIdx.x; e < TB * DC; e += blockDim.x) {
        const int rr = e / DC, dd = e - rr * DC;
        sbm[rr][dd] = (base + rr < j.nb && dd < dc) ? j.B[(size_t)(base + rr) * D + d0 + dd] : 0.f;
      }
      __syncthreads();
      for (int dd = 0; dd < dc; ++dd) {
        const float av = sa[q][dd];
#pragma unroll
        for (int r = 0; r < TB / 2; ++r) {
          const float diff = av - sbm[half * (TB / 2) + r][dd];
          acc[r] += diff * diff;
        }
      }
    }
#pragma unroll
    for (int r = 0; r < TB / 2; ++r) sd[q][half * (TB / 2) + r] = acc[r];
    __syncthreads();
    if (half == 0 && row < j.na) {
      const int tb = min(TB, j.nb - base);
      for (int r = 0; r < tb; ++r) {
        const float v = sd[q][r];
        if (cnt == k && !(v < bd[k - 1])) continue;
        int pos = (cnt < k) ? cnt : k - 1;
        while (pos > 0 && v < bd[pos - 1]) {
          bd[pos] = bd[pos - 1];
          bi[pos] = bi[pos - 1];
          --pos;
        }
        bd[pos] = v;
        bi[pos] = base + r;
        if (cnt < k) ++cnt;
      }
    }
  }
  if (half == 0 && row < j.na)
    for (int t = 0; t < k; ++t) {
      j.idx[(size_t)row * k + t] = t < cnt ? bi[t] : -1;
      j.dist[(size_t)row * k + t] = t < cnt ? bd[t] : 0.f;
    }
}

// Any k (matching_k > 16): the reference hands matching_k straight to nearestKSearch (matching.cpp:45-60), so large values
// must work.  One thread per query row, the sorted top-k list lives in the output arrays themselves (global memory);
// same arithmetic and tie order as the kernels above.  A fallback, not a fast path.
__global__ void __launch_bounds__(128) knn_anyk_kernel(const KnnJob* __restrict__ jobs, int D)
{
  const KnnJob j = jobs[blockIdx.y];
  const int row = blockIdx.x * blockDim.x + threadIdx.x;
  if (row >= j.na) return;
  const int k = j.k;
  const float* a = j.A + (size_t)row * D;
  float* bd = j.dist + (size_t)row * k;
  int* bi = j.idx + (size_t)row * k;
  int cnt = 0;
  for (int r = 0; r < j.nb; ++r) {
    const float* b = j.B + (size_t)r * D;
    float v = 0.f;
    for (int t = 0; t < D; ++t) {
      const float diff = a[t] - __ldg(&b[t]);
      v += diff * diff;
    }
    if (cnt == k && !(v < bd[k - 1])) continue;
    int pos = (cnt < k) ? cnt : k - 1;
    while (pos > 0 && v < bd[pos - 1]) {
      bd[pos] = bd[pos - 1];
      bi[pos] = bi[pos - 1];
      --pos;
    }
    bd[pos] = v;
    bi[pos] = r;
    if (cnt < k) ++cnt;
  }
  for (int t = cnt; t < k; ++t) {
    bd[t] = 0.f;
    bi[t] = -1;
  }
}

struct CrossJob {
  const int* fwd_idx;
  const float* fwd_dist;
  const int* back_idx;
  int ns, kf, kb;
  uint32_t* flags;  // ns
  int* match;       // ns
  float* dist;      // ns
};
// matching.cpp:65-90: first forward match (ascending distance) whose backward k-NN contains i
__global__ void __launch_bounds__(256) cross_match_kernel(const CrossJob* __restrict__ jobs)
{
  const CrossJob& j = jobs[blockIdx.y];
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= j.ns) return;
  uint32_t f = 0;
  int mm = -1;
  float dd = 0.f;
  for (int t = 0; t < j.kf && !f; ++t) {
    const int m = j.fwd_idx[(size_t)i * j.kf + t];
    if (m < 0) break;
    for (int b = 0; b < j.kb; ++b)
      if (j.back_idx[(size_t)m * j.kb + b] == i) {
        f = 1;
        mm = m;
        dd = j.fwd_dist[(size_t)i * j.kf + t];
        break;
      }
  }
  j.flags[i] = f;
  j.match[i] = mm;
  j.dist[i] = dd;
}

struct CorrEmitJob {
  const uint32_t* flags;
  const uint32_t* pos;
  const int* match;
  const float* dist;
  int2* pairs;
  float* odist;
  int ns;
};
__global__ void __launch_bounds__(256) corr_emit_kernel(const CorrEmitJob* __restrict__ jobs)
{
  const CorrEmitJob& j = jobs[blockIdx.y];
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= j.ns) return;
  if (!j.flags[i]) return;
  const uint32_t o = j.pos[i];
  j.pairs[o] = make_int2(i, j.match[i]);
  j.odist[o] = j.dist[i];
}

// ---------------------------------------------------------------- RANSAC
constexpr int MAX_HYP = 1001;  // iterations_ > max_iterations_(1000) breaks after the 1001st

struct RansacJob {
  const float4* skp;
  const float4* tkp;
  const int2* corr;
  int nc;
  int* shuffled;   // nc scratch
  int* samples;    // MAX_HYP x 3 (positions into corr)
  int* n_samples;  // 1
  int* counts;     // MAX_HYP
  float* models;   // MAX_HYP x 12
  int* inliers;    // nc
  RansacOut* out;
};

struct Mt19937 {
  uint32_t* s;  // 624 words in shared memory
  int idx;
  __device__ void seed(uint32_t v)
  {
    s[0] = v;
    for (int i = 1; i < 624; ++i) s[i] = 1812433253u * (s[i - 1] ^ (s[i - 1] >> 30)) + (uint32_t)i;
    idx = 624;
  }
  __device__ uint32_t next()
  {
    if (idx >= 624) {
      for (int i = 0; i < 624; ++i) {
        const uint32_t y = (s[i] & 0x80000000u) | (s[(i + 1) % 624] & 0x7fffffffu);
        s[i] = s[(i + 397) % 624] ^ (y >> 1) ^ ((y & 1u) ? 0x9908b0dfu : 0u);
      }
      idx = 0;
    }
    uint32_t y = s[idx++];
    y ^= (y >> 11);
    y ^= (y << 7) & 0x9d2c5680u;
    y ^= (y << 15) & 0xefc60000u;
    y ^= (y >> 18);
    return y;
  }
};

// One block per pair, thread 0 works: sample-distance threshold, then the whole
// sample sequence the sequential RANSAC would draw (it depends only on the RNG
// and on source keypoint coordinates, never on inlier counts).
// stage_cap = number of correspondences whose source point (3 floats) and shuffle slot (1 int) fit in the
// dynamic shared memory of this launch; a pair with more falls back to global memory.
__global__ void __launch_bounds__(128) ransac_sample_kernel(const RansacJob* __restrict__ jobs, int stage_cap)
{
  extern __shared__ __align__(16) unsigned char rs_smem[];
  uint32_t* mt_state = reinterpret_cast<uint32_t*>(rs_smem);
  float* sx = reinterpret_cast<float*>(rs_smem + 624 * 4);
  float* sy = sx + stage_cap;
  float* sz = sy + stage_cap;
  int* sshuf = reinterpret_cast<int*>(sz + stage_cap);
  const RansacJob& j = jobs[blockIdx.x];
  const int nc = j.nc;
  // all threads: stage the source keypoint of every correspondence (the sequential part only reads these)
  const bool staged = nc <= stage_cap;
  int* shuffled = staged ? sshuf : j.shuffled;
  if (staged)
    for (int i = threadIdx.x; i < nc; i += blockDim.x) {
      const float4 p = j.skp[j.corr[i].x];
      sx[i] = p.x; sy[i] = p.y; sz[i] = p.z;
    }
  for (int i = threadIdx.x; i < nc; i += blockDim.x) shuffled[i] = i;
  __syncthreads();
  if (threadIdx.x != 0) return;
  auto src_pt = [&](int pos, float* x, float* y, float* z) {
    if (staged) { *x = sx[pos]; *y = sy[pos]; *z = sz[pos]; }
    else { const float4 p = j.skp[j.corr[pos].x]; *x = p.x; *y = p.y; *z = p.z; }
  };
  j.out->sample_dist_thresh = 0.0;
  if (nc < 3) {
    *j.n_samples = 0;
    return;
  }
  // computeSampleDistanceThreshold: PCA of the source correspondences
  float a[9] = {0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f};
  for (int i = 0; i < nc; ++i) {
    float px, py, pz;
    src_pt(i, &px, &py, &pz);
    a[0] += px * px; a[1] += px * py; a[2] += px * pz;
    a[3] += py * py; a[4] += py * pz; a[5] += pz * pz;
    a[6] += px; a[7] += py; a[8] += pz;
  }
  const float n = (float)nc;
  for (int k = 0; k < 9; ++k) a[k] /= n;
  float cov[9];
  cov[0] = a[0] - a[6] * a[6];
  cov[1] = a[1] - a[6] * a[7];
  cov[2] = a[2] - a[6] * a[8];
  cov[4] = a[3] - a[7] * a[7];
  cov[5] = a[4] - a[7] * a[8];
  cov[8] = a[5] - a[8] * a[8];
  cov[3] = cov[1]; cov[6] = cov[2]; cov[7] = cov[5];
  float ev[3];
  em::eigen33_values(cov, ev);
  double thr = (double)((sqrtf(ev[0]) + sqrtf(ev[1])) + sqrtf(ev[2])) / 3.0;
  thr *= thr;
  j.out->sample_dist_thresh = thr;

  Mt19937 rng;
  rng.s = mt_state;
  rng.seed(12345u);
  int ns = 0;
  for (int h = 0; h < MAX_HYP; ++h) {
    bool good = false;
    int s0 = 0, s1 = 0, s2 = 0;
    for (int iter = 0; iter < 1000; ++iter) {
      for (int i = 0; i < 3; ++i) {
        const uint32_t rnd = rng.next() >> 1;  // uniform_int<>(0, INT_MAX) on mt19937
        const int o = i + (int)(rnd % (uint32_t)(nc - i));
        const int t = shuffled[i];
        shuffled[i] = shuffled[o];
        shuffled[o] = t;
      }
      s0 = shuffled[0]; s1 = shuffled[1]; s2 = shuffled[2];
      float pax, pay, paz, pbx, pby, pbz, pcx, pcy, pcz;
      src_pt(s0, &pax, &pay, &paz);
      src_pt(s1, &pbx, &pby, &pbz);
      src_pt(s2, &pcx, &pcy, &pcz);
      const float ax = pbx - pax, ay = pby - pay, az = pbz - paz;
      const float bx = pcx - pax, by = pcy - pay, bz = pcz - paz;
      const float cx = pcx - pbx, cy = pcy - pby, cz = pcz - pbz;
      if ((double)(ax * ax + ay * ay + az * az) > thr && (double)(bx * bx + by * by + bz * bz) > thr &&
          (double)(cx * cx + cy * cy + cz * cz) > thr) {
        good = true;
        break;
      }
    }
    if (!good) break;
    j.samples[h * 3 + 0] = s0;
    j.samples[h * 3 + 1] = s1;
    j.samples[h * 3 + 2] = s2;
    ++ns;
  }
  *j.n_samples = ns;
}

// literal Eigen::umeyama (no scaling) over n points, sequential sums
template <typename T, typename GetS, typename GetD>
__device__ void umeyama_seq(int n, GetS src, GetD dst, T* Rt)
{
  const T one_over_n = T(1) / (T)n;
  T sm[3] = {0, 0, 0}, dm[3] = {0, 0, 0};
  for (int i = 0; i < n; ++i) {
    T s[3], d[3];
    src(i, s);
    dst(i, d);
    for (int a = 0; a < 3; ++a) { sm[a] += s[a]; dm[a] += d[a]; }
  }
  for (int a = 0; a < 3; ++a) { sm[a] *= one_over_n; dm[a] *= one_over_n; }
  T sigma[9] = {0, 0, 0, 0, 0, 0, 0, 0, 0};
  for (int i = 0; i < n; ++i) {
    T s[3], d[3];
    src(i, s);
    dst(i, d);
    for (int a = 0; a < 3; ++a) { s[a] -= sm[a]; d[a] -= dm[a]; }
    for (int r = 0; r < 3; ++r)
      for (int cc = 0; cc < 3; ++cc) sigma[r * 3 + cc] += (one_over_n * d[r]) * s[cc];
  }
  em::umeyama_from_sigma<T>(sigma, sm, dm, Rt);
}

// one warp per hypothesis: lane 0 solves the 3-point Umeyama in double, all lanes vote
__global__ void __launch_bounds__(128) ransac_score_kernel(const RansacJob* __restrict__ jobs, double thresh)
{
  const RansacJob& j = jobs[blockIdx.y];
  const int h = blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
  const int lane = threadIdx.x & 31;
  if (h >= *j.n_samples) return;
  float m[12];
  if (lane == 0) {
    const int* smp = j.samples + h * 3;
    double Rt[16];
    umeyama_seq<double>(
        3,
        [&](int i, double* o) { const float4 p = j.skp[j.corr[smp[i]].x]; o[0] = p.x; o[1] = p.y; o[2] = p.z; },
        [&](int i, double* o) { const float4 p = j.tkp[j.corr[smp[i]].y]; o[0] = p.x; o[1] = p.y; o[2] = p.z; }, Rt);
    for (int i = 0; i < 12; ++i) m[i] = (float)Rt[i];
  }
#pragma unroll
  for (int i = 0; i < 12; ++i) m[i] = __shfl_sync(0xffffffffu, m[i], 0);
  int cnt = 0;
  for (int i = lane; i < j.nc; i += 32) {
    const int2 cr = j.corr[i];
    const float4 s = j.skp[cr.x], t = j.tkp[cr.y];
    float px, py, pz;
    em::transform_point(m, s.x, s.y, s.z, &px, &py, &pz);
    const float ex = px - t.x, ey = py - t.y, ez = pz - t.z;
    if ((double)((ex * ex + ey * ey) + ez * ez) < thresh) ++cnt;
  }
  cnt = __reduce_add_sync(0xffffffffu, cnt);
  if (lane == 0) {
    j.counts[h] = cnt;
    for (int i = 0; i < 12; ++i) j.models[h * 12 + i] = m[i];
  }
}

__device__ bool is_identity4(const float* t)
{
  for (int i = 0; i < 4; ++i)
    for (int c = 0; c < 4; ++c) {
      const float v = t[i * 4 + c];
      if (i == c) {
        if (!(fabsf(v - 1.0f) <= 1e-5f * fminf(fabsf(v), 1.0f))) return false;
      } else {
        if (!(fabsf(v) <= 1e-5f)) return false;
      }
    }
  return true;
}

// replay of pcl::RandomSampleConsensus::computeModel's adaptive loop over the pre-scored hypotheses;
// fills the debug fields of the output and returns the winning hypothesis (or -1)
__device__ int ransac_replay(const RansacJob& j)
{
  RansacOut& o = *j.out;
  for (int i = 0; i < 16; ++i) { o.T[i] = 0.f; o.best_model[i] = (i % 5 == 0) ? 1.f : 0.f; }
  o.iterations = 0;
  o.best_count = -2147483647;
  o.n_inliers = 0;
  const int nc = j.nc;
  const int ns = *j.n_samples;
  if (nc < 3) return -1;
  int iterations = 0, n_best = -2147483647, best_h = -1;
  double k = 1.0;
  const double log_probability = log(1.0 - 0.99);
  const double one_over_indices = 1.0 / (double)nc;
  while ((double)iterations < k) {
    if (iterations >= ns) break;  // getSamples came back empty
    const int c = j.counts[iterations];
    if (c > n_best) {
      n_best = c;
      best_h = iterations;
      const double w = (double)n_best * one_over_indices;
      double p_no_outliers = 1.0 - w * w * w;
      p_no_outliers = fmax(2.220446049250313e-16, p_no_outliers);
      p_no_outliers = fmin(1.0 - 2.220446049250313e-16, p_no_outliers);
      k = log_probability / log(p_no_outliers);
    }
    ++iterations;
    if (iterations > 1000) break;
  }
  o.iterations = iterations;
  o.best_count = n_best;
  return best_h;
}

// replay of pcl::RandomSampleConsensus::computeModel's adaptive loop over the
// pre-scored hypotheses, then inlier selection and the final float SVD.
__global__ void __launch_bounds__(32) ransac_select_kernel(const RansacJob* __restrict__ jobs, double thresh)
{
  const RansacJob& j = jobs[blockIdx.x];
  __shared__ int s_best;
  if (threadIdx.x == 0) s_best = ransac_replay(j);
  __syncwarp();
  const int best_h = s_best;
  if (best_h >= 0) {
    // selectWithinDistance with the whole warp: ordered compaction keeps correspondence order
    float bm[12];
    for (int i = 0; i < 12; ++i) bm[i] = j.models[best_h * 12 + i];
    int ni = 0;
    for (int base = 0; base < j.nc; base += 32) {
      const int i = base + threadIdx.x;
      bool in = false;
      if (i < j.nc) {
        const int2 cr = j.corr[i];
        const float4 s = j.skp[cr.x], t = j.tkp[cr.y];
        float px, py, pz;
        em::transform_point(bm, s.x, s.y, s.z, &px, &py, &pz);
        const float ex = px - t.x, ey = py - t.y, ez = pz - t.z;
        in = (double)((ex * ex + ey * ey) + ez * ez) < thresh;
      }
      const unsigned m = __ballot_sync(0xffffffffu, in);
      if (in) j.inliers[ni + __popc(m & ((1u << threadIdx.x) - 1u))] = i;
      ni += __popc(m);
    }
    __syncwarp();
    if (threadIdx.x == 0) *j.n_samples = ni;
  }
  __syncwarp();
  if (threadIdx.x != 0) return;
  RansacOut& o = *j.out;
  if (best_h < 0) return;
  float bm[16];
  for (int i = 0; i < 12; ++i) bm[i] = j.models[best_h * 12 + i];
  bm[12] = bm[13] = bm[14] = 0.f;
  bm[15] = 1.f;
  for (int i = 0; i < 16; ++i) o.best_model[i] = bm[i];
  int ni = *j.n_samples;  // inlier count left here by the warp-wide selection below
  if (ni < 3 || is_identity4(bm)) return;  // matching.cpp:128-133 -> zero matrix, inliers cleared
  o.n_inliers = ni;
  umeyama_seq<float>(
      ni, [&](int i, float* v) { const float4 p = j.skp[j.corr[j.inliers[i]].x]; v[0] = p.x; v[1] = p.y; v[2] = p.z; },
      [&](int i, float* v) { const float4 p = j.tkp[j.corr[j.inliers[i]].y]; v[0] = p.x; v[1] = p.y; v[2] = p.z; }, o.T);
}

// ---------------------------------------------------------------- SAC_IA
// pcl::SampleConsensusInitialAlignment (map_merge_3d/src/matching.cpp:142-194).  The random choices (C rand(), a
// process-global stream in the reference) are drawn on the host for ALL pairs in row-major order; the device scores
// every iteration's hypothesis: float Umeyama on the 3 sampled pairs, then TruncatedError over the transformed source
// keypoints (nearest target keypoint, squared distance), summed sequentially in float like the reference.
struct SacJob {
  const float4* skp;
  int ns;
  const float4* tkp;
  GridView tgt;          // index over the target keypoints
  const int* knn_idx;    // ns x kk nearest target features per source feature
  int kk;
  const int* samples;    // n_it x 3 source keypoint indices
  const int* choice;     // n_it x 3 index into the k-NN list
  float* errors;         // n_it
  float* models;         // n_it x 16 (row-major)
};

__global__ void __launch_bounds__(128) sac_hypothesis_kernel(const SacJob* __restrict__ jobs, int n_jobs, int n_it, float thr, int rv,
                                                            float* __restrict__ scratch, int scratch_stride)
{
  __shared__ float T[16];
  float* terms = scratch + (size_t)blockIdx.x * scratch_stride;
  for (int h = blockIdx.x; h < n_jobs * n_it; h += gridDim.x) {
    const SacJob& j = jobs[h / n_it];
    const int it = h % n_it;
    __syncthreads();
    if (threadIdx.x == 0) {
      const int* smp = j.samples + it * 3;
      const int* ch = j.choice + it * 3;
      int corr[3];
      for (int i = 0; i < 3; ++i) corr[i] = j.knn_idx[(size_t)smp[i] * j.kk + min(ch[i], j.kk - 1)];
      float Rt[16];
      umeyama_seq<float>(
          3, [&](int i, float* o) { const float4 p = j.skp[smp[i]]; o[0] = p.x; o[1] = p.y; o[2] = p.z; },
          [&](int i, float* o) { const float4 p = j.tkp[corr[i]]; o[0] = p.x; o[1] = p.y; o[2] = p.z; }, Rt);
      for (int i = 0; i < 16; ++i) {
        T[i] = Rt[i];
        j.models[(size_t)it * 16 + i] = Rt[i];
      }
    }
    __syncthreads();
    for (int i = threadIdx.x; i < j.ns; i += blockDim.x) {
      const float4 p = j.skp[i];
      float x, y, z;
      em::transform_point(T, p.x, p.y, p.z, &x, &y, &z);
      int idx;
      float d2;
      float4 q;
      float term = 1.0f;
      if (nearest_bounded(j.tgt, x, y, z, (double)thr, rv, &idx, &d2, &q)) term = (d2 <= thr) ? (d2 / thr) : 1.0f;
      terms[i] = term;
    }
    __syncthreads();
    if (threadIdx.x == 0) {
      float error = 0.f;
      for (int i = 0; i < j.ns; ++i) error += terms[i];
      j.errors[it] = error;
    }
  }
}

}  // namespace

// Exact k-NN for a list of (query map, target map) problems: per row of desc[a] (the first na rows), the k nearest rows of
// desc[b], sorted by (distance, index); k <= number of rows of b.
//   * 33-dimensional descriptors (FPFH, the BASELINE configs): tcgen05 distance GEMM as a filter + exact FP32 re-rank
//     (knn_tc.cu) — bit-identical to the FP32 scan and faster;
//   * other dimensions default to the FP32 scan kernels; any k above 16 to the any-k fallback.
// MM3D_KNN=tc forces the tensor-core path for every dimension, MM3D_KNN=exact the scan.
void knn_problems(Ctx& c, const std::vector<const float*>& desc, const std::vector<int>& nk, int dim, const std::vector<KnnProblem>& probs)
{
  if (probs.empty()) return;
  std::vector<KnnJob> kj;
  int max_rows = 0, kmax = 0;
  bool uniform_k = true;
  for (const KnnProblem& q : probs) {
    if (q.na <= 0) continue;
    kj.push_back(KnnJob{desc[q.a], q.na, desc[q.b], nk[q.b], q.k, q.idx, q.dist});
    max_rows = std::max(max_rows, q.na);
    kmax = std::max(kmax, q.k);
    if (q.k != probs[0].k) uniform_k = false;
  }
  if (kj.empty() || max_rows == 0) return;
  const char* knn_env = std::getenv("MM3D_KNN");
  const std::string knn_mode = knn_env ? knn_env : "";
  const bool k_fits = kmax <= KMAX;  // == KMAXTC
  bool nb_fits = true;  // the tensor-core kernel keeps 16-bit column indices in its pending lists
  for (const KnnProblem& q : probs)
    if (nk[q.b] > 65535) nb_fits = false;
  const bool use_tc = k_fits && nb_fits && (knn_mode == "tc" || (knn_mode != "exact" && dim == 33));
  if (use_tc) {
    knn_tc_batch(c, desc, nk, dim, probs);
    return;
  }
  DBuf<KnnJob> dkj = to_device(c, kj);
  { double b = 0; for (const KnnJob& q : kj) b += 4.0 * dim * ((double)q.na + q.nb) + 8.0 * q.k * q.na; MM_BYTES(c, b); }
  const unsigned nj = (unsigned)kj.size();
  if (!k_fits) {
    MM_LAUNCH(c, knn_anyk_kernel, dim3((max_rows + 127) / 128, nj), 128, 0, dkj.p, dim);
  } else if (dim == 33 && uniform_k && (kmax == 5 || kmax == 1 || kmax == 8 || kmax == 10)) {
    // the register kernels need one k for the whole batch (k is clamped per problem only when a set is smaller than k)
    const dim3 grid((max_rows + 127) / 128, nj);
    if (kmax == 5) MM_LAUNCH(c, (knn_small_kernel<33, 5>), grid, 128, 0, dkj.p);
    else if (kmax == 1) MM_LAUNCH(c, (knn_small_kernel<33, 1>), grid, 128, 0, dkj.p);
    else if (kmax == 8) MM_LAUNCH(c, (knn_small_kernel<33, 8>), grid, 128, 0, dkj.p);
    else MM_LAUNCH(c, (knn_small_kernel<33, 10>), grid, 128, 0, dkj.p);
  } else {
    MM_LAUNCH(c, knn_generic_kernel, dim3((max_rows + 63) / 64, nj), 128, 0, dkj.p, dim);
  }
}

void match_batch(Ctx& c, const std::vector<const float*>& desc, const std::vector<int>& nk, int dim, const std::vector<PairJob>& jobs,
                 size_t k_in, std::vector<DCorr>& corr)
{
  const int P = (int)jobs.size();
  corr.clear();
  corr.resize(P);
  if (P == 0) return;
  // forward and backward k-NN problems, 2 per pair
  std::vector<KnnJob> kj(2 * P);
  std::vector<DBuf<int>> idxb(2 * P);
  std::vector<DBuf<float>> distb(2 * P);
  int max_rows = 0, max_ns = 0;
  for (int p = 0; p < P; ++p) {
    const int a = jobs[p].a, b = jobs[p].b;
    const int ns = nk[a], nt = nk[b];
    const int kf = (int)std::min<size_t>(k_in, (size_t)nt), kb = (int)std::min<size_t>(k_in, (size_t)ns);  // KdTreeFLANN clamps k
    idxb[2 * p].alloc(c, (size_t)ns * std::max(kf, 1));
    distb[2 * p].alloc(c, (size_t)ns * std::max(kf, 1));
    idxb[2 * p + 1].alloc(c, (size_t)nt * std::max(kb, 1));
    distb[2 * p + 1].alloc(c, (size_t)nt * std::max(kb, 1));
    kj[2 * p] = KnnJob{desc[a], (kf > 0 && k_in > 0) ? ns : 0, desc[b], nt, kf, idxb[2 * p].p, distb[2 * p].p};
    kj[2 * p + 1] = KnnJob{desc[b], (kb > 0 && k_in > 0) ? nt : 0, desc[a], ns, kb, idxb[2 * p + 1].p, distb[2 * p + 1].p};
    max_rows = std::max(max_rows, std::max(kj[2 * p].na, kj[2 * p + 1].na));
    max_ns = std::max(max_ns, ns);
  }
  std::vector<KnnProblem> probs;
  for (int p = 0; p < P; ++p) {
    const int a = jobs[p].a, b = jobs[p].b;
    if (kj[2 * p].na > 0) probs.push_back(KnnProblem{a, b, kj[2 * p].na, kj[2 * p].k, kj[2 * p].idx, kj[2 * p].dist});
    if (kj[2 * p + 1].na > 0) probs.push_back(KnnProblem{b, a, kj[2 * p + 1].na, kj[2 * p + 1].k, kj[2 * p + 1].idx, kj[2 * p + 1].dist});
  }
  knn_problems(c, desc, nk, dim, probs);
  std::vector<int> nss(P);
  for (int p = 0; p < P; ++p) nss[p] = (k_in > 0 && nk[jobs[p].b] > 0) ? nk[jobs[p].a] : 0;
  std::vector<Seg> segs(P);
  int total = 0;
  for (int p = 0; p < P; ++p) { segs[p].off = total; segs[p].n = nss[p]; total += nss[p]; }
  if (total == 0) return;
  DBuf<uint32_t> flags(c, total), pos(c, total);
  DBuf<int> match(c, total);
  DBuf<float> mdist(c, total);
  std::vector<CrossJob> cj(P);
  for (int p = 0; p < P; ++p)
    cj[p] = CrossJob{idxb[2 * p].p, distb[2 * p].p, idxb[2 * p + 1].p, nss[p], kj[2 * p].k, kj[2 * p + 1].k,
                     flags.p + segs[p].off, match.p + segs[p].off, mdist.p + segs[p].off};
  DBuf<CrossJob> dcj = to_device(c, cj);
  MM_LAUNCH(c, cross_match_kernel, dim3((max_ns + 255) / 256, P), 256, 0, dcj.p);
  std::vector<int> totals;
  scan_flags_batch(c, flags.p, pos.p, segs, totals);
  std::vector<CorrEmitJob> ej(P);
  for (int p = 0; p < P; ++p) {
    corr[p].n = totals[p];
    corr[p].pairs.alloc(c, totals[p]);
    corr[p].dist.alloc(c, totals[p]);
    ej[p] = CorrEmitJob{flags.p + segs[p].off, pos.p + segs[p].off, match.p + segs[p].off, mdist.p + segs[p].off,
                        corr[p].pairs.p, corr[p].dist.p, nss[p]};
  }
  DBuf<CorrEmitJob> dej = to_device(c, ej);
  MM_LAUNCH(c, corr_emit_kernel, dim3((max_ns + 255) / 256, P), 256, 0, dej.p);
}

void ransac_batch(Ctx& c, const std::vector<CloudView>& keypoints, const std::vector<PairJob>& jobs, const std::vector<DCorr>& corr,
                  double inlier_threshold, std::vector<RansacOut>& out, std::vector<std::vector<int>>* inliers)
{
  const int P = (int)jobs.size();
  out.assign(P, RansacOut());
  if (inliers) { inliers->clear(); inliers->resize(P); }
  if (P == 0) return;
  size_t tot_c = 0;
  for (int p = 0; p < P; ++p) tot_c += (size_t)corr[p].n;
  DBuf<int> shuffled(c, tot_c + 1), inl(c, tot_c + 1);
  DBuf<int> samples(c, (size_t)P * MAX_HYP * 3), nsamp(c, P), counts(c, (size_t)P * MAX_HYP);
  DBuf<float> models(c, (size_t)P * MAX_HYP * 12);
  DBuf<RansacOut> dout(c, P);
  std::vector<RansacJob> rj(P);
  size_t off = 0;
  for (int p = 0; p < P; ++p) {
    rj[p].skp = keypoints[jobs[p].a].pts;
    rj[p].tkp = keypoints[jobs[p].b].pts;
    rj[p].corr = corr[p].pairs.p;
    rj[p].nc = corr[p].n;
    rj[p].shuffled = shuffled.p + off;
    rj[p].inliers = inl.p + off;
    rj[p].samples = samples.p + (size_t)p * MAX_HYP * 3;
    rj[p].n_samples = nsamp.p + p;
    rj[p].counts = counts.p + (size_t)p * MAX_HYP;
    rj[p].models = models.p + (size_t)p * MAX_HYP * 12;
    rj[p].out = dout.p + p;
    off += (size_t)corr[p].n;
  }
  DBuf<RansacJob> drj = to_device(c, rj);
  const double thresh = inlier_threshold * inlier_threshold;
  int max_c = 0;
  for (int p = 0; p < P; ++p) max_c = std::max(max_c, corr[p].n);
  const int stage_cap = std::min(std::max(max_c, 1), (200 * 1024 - 624 * 4) / 16);
  const size_t rs_smem = 624 * 4 + (size_t)stage_cap * 16;
  // per device and cheap: set on every call (a process may drive several GPUs)
  MM_CUDA(cudaFuncSetAttribute(ransac_sample_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, 200 * 1024));
  MM_LAUNCH(c, ransac_sample_kernel, P, 128, rs_smem, drj.p, stage_cap);
  MM_LAUNCH(c, ransac_score_kernel, dim3((MAX_HYP + 3) / 4, P), 128, 0, drj.p, thresh);
  MM_LAUNCH(c, ransac_select_kernel, P, 32, 0, drj.p, thresh);
  dout.download(c, out.data(), P);
  std::vector<int> hinl;
  if (inliers) {
    hinl.resize(tot_c + 1);
    inl.download(c, hinl.data(), tot_c);
  }
  c.sync();
  if (inliers) {
    off = 0;
    for (int p = 0; p < P; ++p) {
      (*inliers)[p].assign(hinl.begin() + off, hinl.begin() + off + out[p].n_inliers);
      off += (size_t)corr[p].n;
    }
  }
}

// glibc rand(): TYPE_3 additive feedback generator, never seeded in the reference => seed 1
struct GlibcRand {
  int32_t r[34];
  int f, b;
  unsigned long long calls = 0;
  GlibcRand()
  {
    r[0] = 1;
    for (int i = 1; i < 31; ++i) {
      const long hi = r[i - 1] / 127773, lo = r[i - 1] % 127773;
      long word = 16807 * lo - 2836 * hi;
      if (word < 0) word += 2147483647;
      r[i] = (int32_t)word;
    }
    f = 3;
    b = 0;
    for (int i = 0; i < 310; ++i) step();
  }
  int step()
  {
    uint32_t* st = (uint32_t*)r;
    st[f] += st[b];
    const int result = (int)(st[f] >> 1);
    if (++f >= 31) f = 0;
    if (++b >= 31) b = 0;
    return result;
  }
  int next() { ++calls; return step(); }
  int index(int n) { return (int)(n * (next() / (2147483647 + 1.0))); }  // getRandomIndex
};

void sac_ia_batch(Ctx& c, const std::vector<CloudView>& keypoints, const std::vector<const float*>& desc, int dim,
                  const std::vector<PairJob>& all_pairs, const std::vector<int>& wanted, double min_sample_distance, double max_corr_dist,
                  int max_iterations, unsigned long long rand_skip, std::vector<SacOut>& out, std::vector<unsigned long long>* starts)
{
  out.assign(wanted.size(), SacOut());
  for (SacOut& o : out) {
    for (int k = 0; k < 16; ++k) o.T[k] = (k % 5 == 0) ? 1.f : 0.f;  // align() leaves the identity guess when nothing is scored
    o.rand_calls = 0;
  }
  if (starts) starts->assign(all_pairs.size(), rand_skip);
  if ((wanted.empty() && !starts) || max_iterations <= 0) return;
  const int M = (int)keypoints.size();
  const int n_it = max_iterations;
  // host copies of the keypoints: the sample selection is sequential and touches only a few points per draw
  std::vector<std::vector<float4>> hk(M);
  std::vector<char> needed(M, 0);
  for (const PairJob& p : all_pairs) needed[p.a] = 1;
  for (int m = 0; m < M; ++m)
    if (needed[m] && keypoints[m].n) {
      hk[m].resize(keypoints[m].n);
      MM_CUDA(cudaMemcpyAsync(hk[m].data(), keypoints[m].pts, (size_t)keypoints[m].n * sizeof(float4), cudaMemcpyDeviceToHost, c.stream));
    }
  c.sync();
  std::vector<int> slot_of_pair(all_pairs.size(), -1);
  for (size_t w = 0; w < wanted.size(); ++w) slot_of_pair[wanted[w]] = (int)w;
  const int W = (int)wanted.size();
  std::vector<int> h_samples((size_t)W * n_it * 3, 0), h_choice((size_t)W * n_it * 3, 0);
  std::vector<char> runnable(W, 0);
  GlibcRand rng;
  for (unsigned long long i = 0; i < rand_skip; ++i) rng.next();
  for (size_t pi = 0; pi < all_pairs.size(); ++pi) {
    const PairJob& pj = all_pairs[pi];
    const int ns = keypoints[pj.a].n, nt = keypoints[pj.b].n;
    const int slot = slot_of_pair[pi];
    if (starts) (*starts)[pi] = rng.calls;
    if (ns < 3 || nt == 0) {
      if (slot >= 0) out[slot].rand_calls = rng.calls;
      continue;
    }
    if (slot >= 0) runnable[slot] = 1;
    const std::vector<float4>& kp = hk[pj.a];
    float msd = (float)min_sample_distance;
    for (int it = 0; it < n_it; ++it) {
      int sample[3], nsmp = 0, without = 0;
      const int max_without = 3 * ns;
      while (nsmp < 3) {
        const int idx = rng.index(ns);
        bool valid = true;
        for (int i = 0; i < nsmp; ++i) {
          const float dx = kp[idx].x - kp[sample[i]].x, dy = kp[idx].y - kp[sample[i]].y, dz = kp[idx].z - kp[sample[i]].z;
          const float dist = std::sqrt((dx * dx + dy * dy) + dz * dz);
          if (idx == sample[i] || dist < msd) { valid = false; break; }
        }
        if (valid) { sample[nsmp++] = idx; without = 0; }
        else ++without;
        if (without >= max_without) { msd *= 0.5f; without = 0; }
      }
      for (int i = 0; i < 3; ++i) {
        const int rc = rng.index(10);
        if (slot >= 0) {
          h_samples[((size_t)slot * n_it + it) * 3 + i] = sample[i];
          h_choice[((size_t)slot * n_it + it) * 3 + i] = rc;
        }
      }
    }
    if (slot >= 0) out[slot].rand_calls = rng.calls;
  }
  // feature-space 10-NN for the wanted pairs
  std::vector<KnnJob> kj(W);
  std::vector<DBuf<int>> kidx(W);
  std::vector<DBuf<float>> kdist(W);
  int max_rows = 0, max_ns = 0;
  bool uniform10 = true;
  for (int w = 0; w < W; ++w) {
    const PairJob& pj = all_pairs[wanted[w]];
    const int ns = runnable[w] ? keypoints[pj.a].n : 0, nt = keypoints[pj.b].n;
    const int kk = std::min(10, std::max(nt, 1));
    kidx[w].alloc(c, (size_t)std::max(ns, 1) * kk);
    kdist[w].alloc(c, (size_t)std::max(ns, 1) * kk);
    kj[w] = KnnJob{desc[pj.a], ns, desc[pj.b], nt, kk, kidx[w].p, kdist[w].p};
    max_rows = std::max(max_rows, ns);
    max_ns = std::max(max_ns, ns);
    if (ns > 0 && kk != 10) uniform10 = false;
  }
  if (max_rows == 0) return;
  DBuf<KnnJob> dkj = to_device(c, kj);
  if (dim == 33 && uniform10) MM_LAUNCH(c, (knn_small_kernel<33, 10>), dim3((max_rows + 127) / 128, W), 128, 0, dkj.p);
  else MM_LAUNCH(c, knn_generic_kernel, dim3((max_rows + 63) / 64, W), 128, 0, dkj.p, dim);
  // index over the target keypoints (arbitrary positions: the builder re-sorts them)
  std::vector<CloudView> tv(M, CloudView{nullptr, 0});
  for (int w = 0; w < W; ++w)
    if (runnable[w]) tv[all_pairs[wanted[w]].b] = keypoints[all_pairs[wanted[w]].b];
  const float thr = (float)max_corr_dist;
  const float leaf = std::max(0.05f, std::sqrt(std::max(thr, 1e-6f)) * 0.25f);
  std::vector<DIndex> tidx;
  build_index_batch(c, tv, leaf, 1, 1, 1, tidx);
  const int rv = (int)std::ceil(std::sqrt((double)thr) / (double)leaf) + 1;
  DBuf<int> dsamples = to_device(c, h_samples), dchoice = to_device(c, h_choice);
  DBuf<float> errors(c, (size_t)W * n_it), models(c, (size_t)W * n_it * 16);
  std::vector<SacJob> sj;
  std::vector<int> sj_slot;
  for (int w = 0; w < W; ++w) {
    if (!runnable[w]) continue;
    const PairJob& pj = all_pairs[wanted[w]];
    SacJob j;
    j.skp = keypoints[pj.a].pts;
    j.ns = keypoints[pj.a].n;
    j.tkp = keypoints[pj.b].pts;
    j.tgt = tidx[pj.b].v;
    j.knn_idx = kidx[w].p;
    j.kk = kj[w].k;
    j.samples = dsamples.p + (size_t)w * n_it * 3;
    j.choice = dchoice.p + (size_t)w * n_it * 3;
    j.errors = errors.p + (size_t)w * n_it;
    j.models = models.p + (size_t)w * n_it * 16;
    sj.push_back(j);
    sj_slot.push_back(w);
  }
  if (sj.empty()) return;
  DBuf<SacJob> dsj = to_device(c, sj);
  const int grid = std::min((int)sj.size() * n_it, 148 * 8);
  DBuf<float> scratch(c, (size_t)grid * max_ns);
  MM_LAUNCH(c, sac_hypothesis_kernel, grid, 128, 0, dsj.p, (int)sj.size(), n_it, thr, rv, scratch.p, max_ns);
  std::vector<float> herr((size_t)W * n_it), hmod((size_t)W * n_it * 16);
  errors.download(c, herr.data(), herr.size());
  models.download(c, hmod.data(), hmod.size());
  c.sync();
  for (size_t k = 0; k < sj.size(); ++k) {
    const int w = sj_slot[k];
    float lowest = 0.f;
    int best = -1;
    for (int it = 0; it < n_it; ++it) {
      const float e = herr[(size_t)w * n_it + it];
      if (it == 0 || e < lowest) { lowest = e; best = it; }
    }
    if (best >= 0) memcpy(out[w].T, &hmod[((size_t)w * n_it + best) * 16], 16 * sizeof(float));
    out[w].errors.assign(herr.begin() + (size_t)w * n_it, herr.begin() + (size_t)(w + 1) * n_it);
  }
}

}  // namespace mm3d
