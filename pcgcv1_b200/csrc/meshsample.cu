// Surface sampling of a triangle mesh, grid quantisation and deduplication on the device (pcgc_mesh_sample): the training-set
// generator of pcgcv1_b200/dataset.py.  Contract in include/pcgc_b200.h; oracle/meshsample.py restates it in NumPy.
//
// Phases (profiler tags in brackets), all on the ctx stream:
//   [mesh_weight] per face: index check, a2 = |e1 x e2|, max a2 (block max, then atomicMax on the bits: a2 >= 0, so the bit order
//                 is the value order), referenced-vertex marks; then the box of the rotated referenced vertices (min / max on
//                 order-preserving bits); then w = floor(ldexp(a2, 32 - e)) in place of a2.  Integer min / max only, so the result
//                 does not depend on the order.
//   [mesh_scan]   exclusive prefix sum P of w over nt + 1 entries (P[nt] = W), CUB, uint64 (exact in any order).
//   [mesh_sample] one thread per sample: Philox draw, binary search in P, barycentric point, rotation, grid key.
//   [mesh_sort]   CUB radix sort of the keys over 3 * ceil(log2 R) bits, unique, decode to (x, y, z).
// One synchronisation at the end reads the error flags and the unique count.
// This file is built with -fmad=false (build.py PER_FILE): every multiply and add is rounded on its own, as in NumPy.
#include <cub/cub.cuh>
#include <float.h>
#include <math.h>

#include "common.cuh"
#include "philox.cuh"

namespace pcgc {

namespace {

constexpr int kThreads = 256;

enum MeshFlag : int { F_INDEX = 1, F_NONFINITE = 2, F_ZERO_WEIGHT = 4, F_BOX = 8 };

struct MeshParams {
  double lo[3];
  double scale;
  uint64_t W;
};

struct MeshStatus {      // read back by the one synchronisation of a call
  int flags;
  int n_unique;
};

inline unsigned blocks_for(int64_t n) { return (unsigned)((n + kThreads - 1) / kThreads); }

// Order-preserving map of a double onto uint64 (for min / max with integer atomics).
__device__ __forceinline__ unsigned long long ordered_bits(double x) {
  const unsigned long long b = (unsigned long long)__double_as_longlong(x);
  return (b >> 63) ? ~b : (b | 0x8000000000000000ull);
}
__device__ __forceinline__ double from_ordered(unsigned long long b) {
  return __longlong_as_double((long long)((b >> 63) ? (b & 0x7fffffffffffffffull) : ~b));
}

__device__ __forceinline__ void rotate(const double* R, const double* p, double* q) {
  for (int r = 0; r < 3; ++r) q[r] = (R[3 * r] * p[0] + R[3 * r + 1] * p[1]) + R[3 * r + 2] * p[2];
}

struct Rot { double m[9]; };

// Block-wide max (IS_MAX) or min of v; the result is valid on thread 0.  Every thread of the block must call it.
template <bool IS_MAX>
__device__ __forceinline__ unsigned long long block_reduce(unsigned long long v) {
  __shared__ unsigned long long warp_part[kThreads / 32];
  for (int o = 16; o > 0; o >>= 1) {
    const unsigned long long u = __shfl_xor_sync(0xffffffffu, v, o);
    v = IS_MAX ? (u > v ? u : v) : (u < v ? u : v);
  }
  __syncthreads();                                   // warp_part may still be read by an earlier call
  if ((threadIdx.x & 31) == 0) warp_part[threadIdx.x >> 5] = v;
  __syncthreads();
  if (threadIdx.x == 0)
    for (int w = 1; w < kThreads / 32; ++w) v = IS_MAX ? (warp_part[w] > v ? warp_part[w] : v) : (warp_part[w] < v ? warp_part[w] : v);
  return v;
}

// a2 per face, the max a2 (one atomic per block) and the referenced-vertex marks.
__global__ void __launch_bounds__(kThreads) mesh_area_kernel(const double* __restrict__ verts, int64_t nv, const int32_t* __restrict__ tris,
                                                             int64_t nt, double* __restrict__ a2_out, unsigned long long* __restrict__ amax,
                                                             uint8_t* __restrict__ ref, int* __restrict__ flags) {
  const int64_t f = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  unsigned long long bits = 0;
  if (f < nt) {
    int32_t v[3];
    bool ok = true;
    for (int k = 0; k < 3; ++k) {
      v[k] = tris[3 * f + k];
      ok = ok && v[k] >= 0 && v[k] < nv;
    }
    double a2 = 0.0;
    if (!ok) {
      atomicOr(flags, F_INDEX);
    } else {
      for (int k = 0; k < 3; ++k) ref[v[k]] = 1;
      const double* A = verts + 3 * (int64_t)v[0];
      const double* B = verts + 3 * (int64_t)v[1];
      const double* C = verts + 3 * (int64_t)v[2];
      const double e1[3] = {B[0] - A[0], B[1] - A[1], B[2] - A[2]};
      const double e2[3] = {C[0] - A[0], C[1] - A[1], C[2] - A[2]};
      const double cx = e1[1] * e2[2] - e1[2] * e2[1];
      const double cy = e1[2] * e2[0] - e1[0] * e2[2];
      const double cz = e1[0] * e2[1] - e1[1] * e2[0];
      a2 = sqrt((cx * cx + cy * cy) + cz * cz);
      if (!isfinite(a2)) { atomicOr(flags, F_NONFINITE); a2 = 0.0; }
    }
    a2_out[f] = a2;
    bits = (unsigned long long)__double_as_longlong(a2);
  }
  bits = block_reduce<true>(bits);
  if (threadIdx.x == 0) atomicMax(amax, bits);
}

// box[0..2] = ordered min, box[3..5] = ordered max of the rotated referenced vertices (one atomic per block and bound).
__global__ void __launch_bounds__(kThreads) mesh_box_kernel(const double* __restrict__ verts, int64_t nv, const uint8_t* __restrict__ ref,
                                                            Rot rot, unsigned long long* __restrict__ box) {
  const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  unsigned long long mn[3] = {~0ull, ~0ull, ~0ull}, mx[3] = {0, 0, 0};
  if (i < nv && ref[i]) {
    double q[3];
    rotate(rot.m, verts + 3 * i, q);
    for (int k = 0; k < 3; ++k) mn[k] = mx[k] = ordered_bits(q[k]);
  }
  for (int k = 0; k < 3; ++k) {
    const unsigned long long a = block_reduce<false>(mn[k]), b = block_reduce<true>(mx[k]);
    if (threadIdx.x == 0) { atomicMin(&box[k], a); atomicMax(&box[3 + k], b); }
  }
}

// w[f] = floor(ldexp(a2[f], 32 - e)), frexp(max a2) = (m, e); written over a2 (same 8 bytes).  w[nt] = 0 closes the scan input.
__global__ void __launch_bounds__(kThreads) mesh_weight_kernel(double* __restrict__ a2_w, int64_t nt, const unsigned long long* __restrict__ amax) {
  const int64_t f = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (f > nt) return;
  uint64_t w = 0;
  if (f < nt) {
    int e = 0;
    frexp(__longlong_as_double((long long)*amax), &e);
    w = (uint64_t)floor(ldexp(a2_w[f], 32 - e));
  }
  reinterpret_cast<uint64_t*>(a2_w)[f] = w;
}

// One thread: W, the box, the scale; flags for W == 0 and a degenerate or non-finite box.
__global__ void mesh_params_kernel(const uint64_t* __restrict__ P, int64_t nt, const unsigned long long* __restrict__ box, int resolution,
                                   MeshParams* __restrict__ mp, int* __restrict__ flags) {
  if (threadIdx.x != 0 || blockIdx.x != 0) return;
  MeshParams p;
  p.W = P[nt];
  double E = 0.0;
  for (int k = 0; k < 3; ++k) {
    p.lo[k] = from_ordered(box[k]);
    E = fmax(E, from_ordered(box[3 + k]) - p.lo[k]);
  }
  p.scale = (double)(resolution - 1) / E;
  if (p.W == 0) atomicOr(flags, F_ZERO_WEIGHT);
  else if (!(E > 0.0) || !isfinite(E) || !isfinite(p.scale)) atomicOr(flags, F_BOX);
  *mp = p;
}

__global__ void __launch_bounds__(kThreads) mesh_sample_kernel(const double* __restrict__ verts, const int32_t* __restrict__ tris, int64_t nt,
                                                               const uint64_t* __restrict__ P, const MeshParams* __restrict__ mp,
                                                               const int* __restrict__ flags, Rot rot, int64_t n, uint64_t seed,
                                                               int resolution, uint64_t* __restrict__ keys, double* __restrict__ samples,
                                                               int32_t* __restrict__ faces) {
  const int64_t j = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (j >= n || *flags) return;
  const MeshParams p = *mp;
  uint32_t r[4];
  philox4x32_10((uint32_t)j, (uint32_t)((uint64_t)j >> 32), (uint32_t)seed, (uint32_t)(seed >> 32), r);
  const uint64_t t = ((uint64_t)r[1] << 32) | r[0];
  const uint64_t target = __umul64hi(t, p.W);
  int64_t lo = 0, hi = nt - 1;             // the largest f with P[f] <= target (P[0] = 0 <= target)
  while (lo < hi) {
    const int64_t mid = lo + (hi - lo + 1) / 2;
    if (P[mid] <= target) lo = mid; else hi = mid - 1;
  }
  const int64_t f = lo;
  const double u1 = ((double)r[2] + 0.5) * 0x1p-32, u2 = ((double)r[3] + 0.5) * 0x1p-32;
  const double s = sqrt(u1);
  const double a = 1.0 - s, b = s * (1.0 - u2), c = s * u2;
  const double* A = verts + 3 * (int64_t)tris[3 * f];
  const double* B = verts + 3 * (int64_t)tris[3 * f + 1];
  const double* C = verts + 3 * (int64_t)tris[3 * f + 2];
  double x[3], q[3];
  for (int k = 0; k < 3; ++k) x[k] = (a * A[k] + b * B[k]) + c * C[k];
  rotate(rot.m, x, q);
  uint64_t key = 0;
  for (int k = 0; k < 3; ++k) {
    const double g = rint((q[k] - p.lo[k]) * p.scale);
    const int64_t gi = g < 0.0 ? 0 : g > (double)(resolution - 1) ? resolution - 1 : (int64_t)g;
    key = key * (uint64_t)resolution + (uint64_t)gi;
  }
  keys[j] = key;
  if (samples) for (int k = 0; k < 3; ++k) samples[3 * j + k] = q[k];
  if (faces) faces[j] = (int32_t)f;
}

__global__ void __launch_bounds__(kThreads) mesh_decode_kernel(const uint64_t* __restrict__ uniq, const MeshStatus* __restrict__ st, int64_t n,
                                                               int resolution, int32_t* __restrict__ points) {
  const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n || i >= st->n_unique || st->flags) return;
  const uint64_t k = uniq[i], R = (uint64_t)resolution;
  points[3 * i] = (int32_t)(k / (R * R));
  points[3 * i + 1] = (int32_t)((k / R) % R);
  points[3 * i + 2] = (int32_t)(k % R);
}

struct Carver {
  char* base;
  size_t off = 0;
  template <typename T> T* take(size_t count) {
    off = (off + 255) & ~(size_t)255;
    T* p = base ? reinterpret_cast<T*>(base + off) : nullptr;
    off += count * sizeof(T);
    return p;
  }
};

struct Bufs {
  MeshStatus* st;
  MeshParams* mp;
  unsigned long long* stats;     // [0] max a2 bits, [1..6] box
  double* a2w;                   // [nt + 1]: a2, then w
  uint64_t* P;                   // [nt + 1]
  uint8_t* ref;                  // [nv]
  uint64_t* keys[2];             // [n]
  void* tmp;
};

size_t carve(char* base, int64_t nv, int64_t nt, int64_t n, size_t tmp_bytes, Bufs& b) {
  Carver c{base};
  b.st = c.take<MeshStatus>(1);
  b.mp = c.take<MeshParams>(1);
  b.stats = c.take<unsigned long long>(7);
  b.a2w = c.take<double>(nt + 1);
  b.P = c.take<uint64_t>(nt + 1);
  b.ref = c.take<uint8_t>(nv);
  for (int k = 0; k < 2; ++k) b.keys[k] = c.take<uint64_t>(n);
  b.tmp = c.take<char>(tmp_bytes);
  return c.off + 256;
}

__global__ void mesh_init_kernel(MeshStatus* st, unsigned long long* stats) {
  if (threadIdx.x != 0 || blockIdx.x != 0) return;
  st->flags = 0;
  st->n_unique = 0;
  stats[0] = 0;
  for (int k = 0; k < 3; ++k) { stats[1 + k] = ~0ull; stats[4 + k] = 0; }
}

}  // namespace

struct MeshWorkspace {
  void* mem = nullptr;
  size_t cap = 0;
};

void free_mesh_workspace(MeshWorkspace* ws) {
  if (!ws) return;
  if (ws->mem) cudaFree(ws->mem);
  delete ws;
}

}  // namespace pcgc

using namespace pcgc;

#define MK(call)                                                                                                            \
  do {                                                                                                                      \
    cudaError_t e_ = (call);                                                                                                \
    if (e_ != cudaSuccess)                                                                                                  \
      return ctx_fail(ctx, e_ == cudaErrorMemoryAllocation ? PCGC_ERR_OOM : PCGC_ERR_CUDA, cudaGetErrorString(e_));         \
  } while (0)

extern "C" int pcgc_mesh_sample(pcgc_ctx* ctx, const double* verts_dev, int64_t nv, const int32_t* tris_dev, int64_t nt, const double* rot_host,
                                int64_t n, uint64_t seed, int resolution, int32_t* points_dev, int64_t* n_unique, double* samples_dev,
                                int32_t* face_dev) {
  if (!ctx) return PCGC_ERR_BAD_ARG;
  if (!verts_dev || !tris_dev || !rot_host || !points_dev || !n_unique || nv < 1 || nv > INT32_MAX || nt < 1 || nt > ((int64_t)1 << 30) ||
      n < 1 || n > ((int64_t)1 << 28) || resolution < 2 || resolution > 4096)
    return ctx_fail(ctx, PCGC_ERR_BAD_ARG, "pcgc_mesh_sample: bad argument (1 <= nt <= 2^30, 1 <= n <= 2^28, 2 <= resolution <= 4096)");
  int prev = -1;
  cudaGetDevice(&prev);
  if (prev != ctx_device(ctx)) cudaSetDevice(ctx_device(ctx)); else prev = -1;
  struct Restore { int d; ~Restore() { if (d >= 0) cudaSetDevice(d); } } restore_{prev};
  cudaStream_t s = ctx_stream(ctx);
  int64_t* launches = ctx_launches(ctx);
  MeshWorkspace*& ws = *ctx_mesh_workspace(ctx);

  int bits = 0;
  while ((1 << bits) < resolution) ++bits;
  const int end_bit = 3 * bits;
  size_t scan_bytes = 0, sort_bytes = 0, uniq_bytes = 0;
  {
    cub::DoubleBuffer<uint64_t> k(nullptr, nullptr);
    MK(cub::DeviceScan::ExclusiveSum(nullptr, scan_bytes, (uint64_t*)nullptr, (uint64_t*)nullptr, (int)(nt + 1), s));
    MK(cub::DeviceRadixSort::SortKeys(nullptr, sort_bytes, k, (int)n, 0, end_bit, s));
    MK(cub::DeviceSelect::Unique(nullptr, uniq_bytes, (uint64_t*)nullptr, (uint64_t*)nullptr, (int*)nullptr, (int)n, s));
  }
  const size_t tmp_bytes = std::max(scan_bytes, std::max(sort_bytes, uniq_bytes));
  Bufs b;
  const size_t need = carve(nullptr, nv, nt, n, tmp_bytes, b);
  if (!ws) ws = new MeshWorkspace();
  if (ws->cap < need) {
    if (ws->mem) { MK(cudaStreamSynchronize(s)); MK(cudaFree(ws->mem)); ws->mem = nullptr; ws->cap = 0; }
    const size_t want = need + need / 4;
    MK(cudaMalloc(&ws->mem, want));
    ws->cap = want;
  }
  carve(reinterpret_cast<char*>(((uintptr_t)ws->mem + 255) & ~(uintptr_t)255), nv, nt, n, tmp_bytes, b);
  Rot rot;
  for (int k = 0; k < 9; ++k) rot.m[k] = rot_host[k];

  ctx_prof_begin(ctx, "mesh_weight", 0, 100.0 * (double)nt + 33.0 * (double)nv);
  mesh_init_kernel<<<1, 32, 0, s>>>(b.st, b.stats);
  MK(cudaMemsetAsync(b.ref, 0, (size_t)nv, s));
  mesh_area_kernel<<<blocks_for(nt), kThreads, 0, s>>>(verts_dev, nv, tris_dev, nt, b.a2w, &b.stats[0], b.ref, &b.st->flags);
  mesh_box_kernel<<<blocks_for(nv), kThreads, 0, s>>>(verts_dev, nv, b.ref, rot, &b.stats[1]);
  mesh_weight_kernel<<<blocks_for(nt + 1), kThreads, 0, s>>>(b.a2w, nt, &b.stats[0]);
  ctx_prof_end(ctx);

  ctx_prof_begin(ctx, "mesh_scan", 0, 16.0 * (double)(nt + 1));
  size_t bytes = tmp_bytes;
  MK(cub::DeviceScan::ExclusiveSum(b.tmp, bytes, reinterpret_cast<const uint64_t*>(b.a2w), b.P, (int)(nt + 1), s));
  mesh_params_kernel<<<1, 32, 0, s>>>(b.P, nt, &b.stats[1], resolution, b.mp, &b.st->flags);
  ctx_prof_end(ctx);

  ctx_prof_begin(ctx, "mesh_sample", 0, (double)n * (8.0 + 8.0 * 20 + 72.0 + (samples_dev ? 24.0 : 0.0) + (face_dev ? 4.0 : 0.0)));
  mesh_sample_kernel<<<blocks_for(n), kThreads, 0, s>>>(verts_dev, tris_dev, nt, b.P, b.mp, &b.st->flags, rot, n, seed, resolution,
                                                        b.keys[0], samples_dev, face_dev);
  ctx_prof_end(ctx);

  ctx_prof_begin(ctx, "mesh_sort", 0, (double)n * (16.0 * 3 + 12.0));
  cub::DoubleBuffer<uint64_t> keys(b.keys[0], b.keys[1]);
  bytes = tmp_bytes;
  MK(cub::DeviceRadixSort::SortKeys(b.tmp, bytes, keys, (int)n, 0, end_bit, s));
  bytes = tmp_bytes;
  MK(cub::DeviceSelect::Unique(b.tmp, bytes, keys.Current(), keys.Alternate(), &b.st->n_unique, (int)n, s));
  mesh_decode_kernel<<<blocks_for(n), kThreads, 0, s>>>(keys.Alternate(), b.st, n, resolution, points_dev);
  ctx_prof_end(ctx);
  *launches += 11;     // seven kernels, the memset, and the scan, the sort and the unique as one launch each
  MK(cudaGetLastError());

  MeshStatus st;
  MK(cudaMemcpyAsync(&st, b.st, sizeof st, cudaMemcpyDeviceToHost, s));
  MK(cudaStreamSynchronize(s));
  if (st.flags & F_INDEX) return ctx_fail(ctx, PCGC_ERR_BAD_ARG, "pcgc_mesh_sample: a face index is outside [0, nv)");
  if (st.flags & F_NONFINITE) return ctx_fail(ctx, PCGC_ERR_BAD_ARG, "pcgc_mesh_sample: a face has a non-finite area (NaN / inf vertex)");
  if (st.flags & F_ZERO_WEIGHT) return ctx_fail(ctx, PCGC_ERR_BAD_ARG, "pcgc_mesh_sample: every face is degenerate (total weight 0)");
  if (st.flags & F_BOX) return ctx_fail(ctx, PCGC_ERR_BAD_ARG, "pcgc_mesh_sample: the bounding box of the rotated vertices is degenerate");
  *n_unique = st.n_unique;
  return PCGC_OK;
}
