// layout.cu — point records in a caller's layout (mm3d_layout) <-> the float4 clouds the pipeline reads.
//
// Input in the packed layout is copied straight from the caller's buffer.  Any other layout is staged: host threads copy
// raw records from the caller's (usually pageable) memory into pinned slots of the context, each slot is copied to a device
// slot and unpack_records writes the float4 cloud.  Outputs are packed into records on the device (pack_records) and
// copied once into the pinned output pool.  Fields move as 32-bit words, never through float arithmetic.
#include <cstring>
#include <exception>
#include <mutex>
#include <thread>

#include "../../include/mm3d.h"
#include "mm3d_internal.cuh"
#include "pipeline.cuh"

namespace mm3d {

const mm3d_layout kPackedLayout = {16, 0, 4, 8, 12, nullptr};

namespace {

constexpr int kCopyThreads = 4;
constexpr int kSlots = 2 * kCopyThreads;        // each copy thread fills its two slots alternately
constexpr size_t kSlotBytes = (size_t)8 << 20;  // >= 128 records of the largest point_step

__device__ __forceinline__ uint32_t word_of(const uint4& q, int w) { return w == 0 ? q.x : w == 1 ? q.y : w == 2 ? q.z : q.w; }

// off = byte offsets of x, y, z, rgba.  VEC: point_step % 16 == 0, so every record starts 16-byte aligned and is read in
// 16-byte blocks (a block that holds several fields is loaded once).
template <bool VEC>
__global__ void unpack_records(const unsigned char* __restrict__ src, unsigned n, int step, int4 off, uint4* __restrict__ dst)
{
  const unsigned i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  const unsigned char* r = src + (size_t)i * step;
  uint4 o;
  if (VEC) {
    const uint4* q = (const uint4*)r;
    const int bx = off.x >> 4, by = off.y >> 4, bz = off.z >> 4, bc = off.w >> 4;
    const uint4 qx = __ldg(q + bx);
    const uint4 qy = by == bx ? qx : __ldg(q + by);
    const uint4 qz = bz == bx ? qx : bz == by ? qy : __ldg(q + bz);
    const uint4 qc = bc == bx ? qx : bc == by ? qy : bc == bz ? qz : __ldg(q + bc);
    o = make_uint4(word_of(qx, (off.x >> 2) & 3), word_of(qy, (off.y >> 2) & 3), word_of(qz, (off.z >> 2) & 3), word_of(qc, (off.w >> 2) & 3));
  } else {
    const uint32_t* w = (const uint32_t*)r;
    o = make_uint4(__ldg(w + (off.x >> 2)), __ldg(w + (off.y >> 2)), __ldg(w + (off.z >> 2)), __ldg(w + (off.w >> 2)));
  }
  dst[i] = o;
}

// Each record = the template's words, then x, y, z and rgba written over them in that order.  off = word offsets.
template <bool VEC>
__global__ void pack_records(const uint4* __restrict__ src, unsigned n, int step, int4 off, const uint32_t* __restrict__ tmpl,
                             unsigned char* __restrict__ dst)
{
  const unsigned i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  const uint4 p = src[i];
  unsigned char* r = dst + (size_t)i * step;
  auto word = [&](int k) -> uint32_t {
    return k == off.w ? p.w : k == off.z ? p.z : k == off.y ? p.y : k == off.x ? p.x : __ldg(tmpl + k);
  };
  const int nw = step >> 2;
  if (VEC) {
    for (int k = 0; k < nw; k += 4) ((uint4*)r)[k >> 2] = make_uint4(word(k), word(k + 1), word(k + 2), word(k + 3));
  } else {
    for (int k = 0; k < nw; ++k) ((uint32_t*)r)[k] = word(k);
  }
}

void launch_unpack(Ctx& c, const unsigned char* src, size_t n, const mm3d_layout& l, float4* dst)
{
  const int4 off = make_int4(l.offset_x, l.offset_y, l.offset_z, l.offset_rgba);
  const unsigned blocks = (unsigned)((n + 255) / 256);
  MM_BYTES(c, n * (l.point_step + 16.0));
  if (l.point_step % 16 == 0) MM_LAUNCH(c, unpack_records<true>, blocks, 256, 0, src, (unsigned)n, (int)l.point_step, off, (uint4*)dst);
  else MM_LAUNCH(c, unpack_records<false>, blocks, 256, 0, src, (unsigned)n, (int)l.point_step, off, (uint4*)dst);
}

}  // namespace

// Pinned host slots and their device twins, allocated on the first staged upload of a context and kept until mm3d_destroy.
struct StagingRing {
  void* host[kSlots] = {};
  void* dev[kSlots] = {};
  cudaEvent_t copied[kSlots] = {};  // the slot's host-to-device copy has finished: the host may refill it
};

void staging_release(Ctx& c)
{
  StagingRing* r = c.staging;
  if (!r) return;
  for (int s = 0; s < kSlots; ++s) {
    if (r->host[s]) cudaFreeHost(r->host[s]);
    if (r->dev[s]) cudaFree(r->dev[s]);
    if (r->copied[s]) cudaEventDestroy(r->copied[s]);
  }
  delete r;
  c.staging = nullptr;
}

static StagingRing& staging(Ctx& c)
{
  if (c.staging) return *c.staging;
  c.staging = new StagingRing;
  try {
    for (int s = 0; s < kSlots; ++s) {
      MM_CUDA(cudaHostAlloc(&c.staging->host[s], kSlotBytes, cudaHostAllocPortable));
      MM_CUDA(cudaMalloc(&c.staging->dev[s], kSlotBytes));
      MM_CUDA(cudaEventCreateWithFlags(&c.staging->copied[s], cudaEventDisableTiming));
    }
  } catch (...) {
    staging_release(c);
    throw;
  }
  return *c.staging;
}

bool layout_valid(const mm3d_layout* l)
{
  if (!l || l->point_step < 16 || l->point_step > MM3D_LAYOUT_MAX_STEP || l->point_step % 4) return false;
  for (int32_t o : {l->offset_x, l->offset_y, l->offset_z, l->offset_rgba})
    if (o < 0 || o % 4 || (uint64_t)o + 4 > l->point_step) return false;
  return true;
}

bool layout_packed(const mm3d_layout& l)
{
  return l.point_step == 16 && l.offset_x == 0 && l.offset_y == 4 && l.offset_z == 8 && l.offset_rgba == 12;
}

std::vector<DCloud> upload_clouds(Ctx& c, const std::vector<const void*>& src, const std::vector<uint64_t>& n, const mm3d_layout& l)
{
  const int M = (int)src.size();
  std::vector<DCloud> out(M);
  for (int m = 0; m < M; ++m) {
    out[m].n = src[m] ? (int)n[m] : 0;
    out[m].pts.alloc(c, out[m].n);
  }
  if (layout_packed(l)) {
    for (int m = 0; m < M; ++m)
      if (out[m].n) MM_CUDA(cudaMemcpyAsync(out[m].pts.p, src[m], (size_t)out[m].n * sizeof(float4), cudaMemcpyHostToDevice, c.stream));
    return out;
  }
  const size_t step = l.point_step, per_slot = kSlotBytes / step;
  struct Chunk {
    int map;
    size_t first, count;
  };
  std::vector<Chunk> chunks;
  for (int m = 0; m < M; ++m)
    for (size_t f = 0; f < (size_t)out[m].n; f += per_slot) chunks.push_back(Chunk{m, f, std::min(per_slot, (size_t)out[m].n - f)});
  if (chunks.empty()) return out;
  StagingRing& ring = staging(c);
  const int T = (int)std::min<size_t>(kCopyThreads, chunks.size());
  std::mutex enqueue;  // the stream and the context's launch bookkeeping are shared by the copy threads
  std::vector<std::exception_ptr> err(T);
  const bool trace = host_prof().on;
  std::vector<double> copy_ms(T, 0.0), wait_ms(T, 0.0);
  const double t_start = trace ? host_now_ms() : 0.0;
  auto work = [&](int t) {
    try {
      MM_CUDA(cudaSetDevice(c.device));
      int j = 0;
      for (size_t k = t; k < chunks.size(); k += T, ++j) {
        const int s = 2 * t + (j & 1);
        const Chunk& ch = chunks[k];
        const size_t bytes = ch.count * step;
        double t0 = trace ? host_now_ms() : 0.0;
        MM_CUDA(cudaEventSynchronize(ring.copied[s]));
        if (trace) {
          const double t1 = host_now_ms();
          wait_ms[t] += t1 - t0;
          t0 = t1;
        }
        std::memcpy(ring.host[s], (const unsigned char*)src[ch.map] + ch.first * step, bytes);
        if (trace) copy_ms[t] += host_now_ms() - t0;
        std::lock_guard<std::mutex> lk(enqueue);
        MM_CUDA(cudaMemcpyAsync(ring.dev[s], ring.host[s], bytes, cudaMemcpyHostToDevice, c.stream));
        MM_CUDA(cudaEventRecord(ring.copied[s], c.stream));
        launch_unpack(c, (const unsigned char*)ring.dev[s], ch.count, l, out[ch.map].pts.p + ch.first);
      }
    } catch (...) {
      err[t] = std::current_exception();
    }
  };
  std::vector<std::thread> th;
  for (int t = 1; t < T; ++t) th.emplace_back(work, t);
  work(0);
  for (std::thread& x : th) x.join();
  for (const std::exception_ptr& e : err)
    if (e) std::rethrow_exception(e);
  if (trace) {
    double cm = 0, wm = 0;
    for (int t = 0; t < T; ++t) { cm += copy_ms[t]; wm += wait_ms[t]; }
    size_t recs = 0;
    for (const Chunk& ch : chunks) recs += ch.count;
    fprintf(stderr, "[mm3d staging] %zu records of %zu bytes in %zu slots: enqueue wall %.2f ms, host copy %.2f ms, slot waits %.2f ms "
            "(summed over %d threads)\n", recs, step, chunks.size(), host_now_ms() - t_start, cm, wm, T);
  }
  return out;
}

DCloud upload_cloud(Ctx& c, const float* pts, uint64_t n) { return std::move(upload_clouds(c, {pts}, {n}, kPackedLayout)[0]); }

void* download_records(Ctx& c, const float4* pts, size_t n, const mm3d_layout& l)
{
  const size_t step = l.point_step;
  void* h = host_out_alloc(std::max<size_t>(n * step, 1));
  try {
    if (n && layout_packed(l)) {
      MM_CUDA(cudaMemcpyAsync(h, pts, n * sizeof(float4), cudaMemcpyDeviceToHost, c.stream));
    } else if (n) {
      DBuf<uint32_t> tmpl(c, step / 4);
      if (l.record_template) tmpl.upload(c, (const uint32_t*)l.record_template, step / 4);
      else tmpl.zero(c);
      DBuf<unsigned char> rec(c, n * step);
      const int4 off = make_int4(l.offset_x / 4, l.offset_y / 4, l.offset_z / 4, l.offset_rgba / 4);
      const unsigned blocks = (unsigned)((n + 255) / 256);
      MM_BYTES(c, n * (16.0 + step));
      if (step % 16 == 0) MM_LAUNCH(c, pack_records<true>, blocks, 256, 0, (const uint4*)pts, (unsigned)n, (int)step, off, tmpl.p, rec.p);
      else MM_LAUNCH(c, pack_records<false>, blocks, 256, 0, (const uint4*)pts, (unsigned)n, (int)step, off, tmpl.p, rec.p);
      MM_CUDA(cudaMemcpyAsync(h, rec.p, n * step, cudaMemcpyDeviceToHost, c.stream));
    }
  } catch (...) {
    host_out_free(h);
    throw;
  }
  return h;
}

}  // namespace mm3d
