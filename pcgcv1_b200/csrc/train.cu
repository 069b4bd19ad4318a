// Training-step primitives (SURVEY.md 8a row a22; train_hyper.py:184-214, loss.py:8-33): forward, data-gradient and
// weight-gradient of every Conv3D / Conv3DTranspose of the model, the Voxception merge, the two entropy models with "noise"
// quantisation, the BCE occupancy loss and Adam -- each a C-ABI entry point over device pointers.  The host side
// (pcgcv1_b200/training.py) strings them together; torch.autograd is only the tape that orders the backward calls.
//
// Exact FP32 on CUDA cores, deterministic:
//   * forward and data-gradient run on the gather-convolution kernel of conv_ffma.cu (fixed reduction order).  The data-gradient
//     of a layer IS a convolution of the same family: stride-1 SAME conv -> conv with the taps flipped and the channel roles
//     swapped; stride-2 conv -> the Conv3DTranspose with the SAME kernel array (they are adjoint, tests/test_oracle_golden.py);
//     Conv3DTranspose -> the stride-2 conv with the same array.  Weights arrive in the Keras layout and are re-packed on the
//     device per call (they change every step).
//   * weight-gradient: dW[tap][cg][ca] = sum_v T[s*v + tap - pad][cg] * A[v][ca] over anchor voxels v (A = output gradient for a
//     conv, = input for a transposed conv; T = the other one), computed as fixed-order partial sums over voxel ranges and a
//     second fixed-order pass over the partials (no atomics): per anchor tile for k <= 3 (wgrad_tile_kernel), per fixed run of
//     tiles for the k = 9 layers of model_simple (wgrad_slice_kernel).
#include <math.h>
#include <stdint.h>

#include <algorithm>

#include "common.cuh"
#include "det_math.h"
#include "philox.cuh"

namespace pcgc {
namespace {

#define TCK(call)                                                                                    \
  do {                                                                                               \
    cudaError_t e_ = (call);                                                                         \
    if (e_ != cudaSuccess) return ctx_fail(ctx, e_ == cudaErrorMemoryAllocation ? PCGC_ERR_OOM : PCGC_ERR_CUDA, cudaGetErrorString(e_)); \
  } while (0)

int pad_before(int k, int stride) { return stride == 1 ? (k - 1) / 2 : (k - 2) / 2; }      // TF SAME, even extents

// ---------------------------------------------------------------------------------------------- weight packing
// dst = the gather kernel's layout [KY][KX][Cin][KZ][Cout] of one tap box; src = a Keras kernel array.
//   mode 0: regular conv a -> b from src [k,k,k,a,b]
//   mode 1: the same with flipped taps and swapped channel roles (data-gradient of a stride-1 conv): conv b -> a
//   mode 2: parity class (r0,r1,r2) of a stride-2 transposed conv b -> a from src [k,k,k,a,b] (a = its Cout, b = its Cin)
struct PackArgs { int mode, k, a, b; int km[3], r[3]; };

__global__ void pack_weights_kernel(const float* __restrict__ src, float* __restrict__ dst, PackArgs p, int total) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= total) return;
  const int KZ = p.mode == 2 ? p.km[0] : p.k, KY = p.mode == 2 ? p.km[1] : p.k, KX = p.mode == 2 ? p.km[2] : p.k;
  const int cin = p.mode == 0 ? p.a : p.b, cout = p.mode == 0 ? p.b : p.a;
  int e = i;
  const int co = e % cout; e /= cout;
  const int jz = e % KZ; e /= KZ;
  const int ci = e % cin; e /= cin;
  const int jx = e % KX; const int jy = e / KX;
  (void)KY;
  int kz, ky, kx;
  if (p.mode == 0) { kz = jz; ky = jy; kx = jx; }
  else if (p.mode == 1) { kz = p.k - 1 - jz; ky = p.k - 1 - jy; kx = p.k - 1 - jx; }
  else { kz = p.r[0] + 2 * (p.km[0] - 1 - jz); ky = p.r[1] + 2 * (p.km[1] - 1 - jy); kx = p.r[2] + 2 * (p.km[2] - 1 - jx); }
  const size_t tap = ((size_t)kz * p.k + ky) * p.k + kx;
  // src [tap][a][b]: mode 0 reads [ci][co]; modes 1, 2 read [co][ci]
  const float v = p.mode == 0 ? src[(tap * p.a + ci) * p.b + co] : src[(tap * p.a + co) * p.b + ci];
  dst[i] = v;
}

// Runs y = conv(x) (+bias, relu) where the convolution is given as (family, k, stride) over a Keras kernel array.
//   family 0: regular conv cin -> cout, src [k,k,k,cin,cout];   family 1: flipped/swapped stride-1 conv (dgrad), src [k,k,k,cout,cin]
//   family 2: stride-2 transposed conv cin -> cout, src [k,k,k,cout,cin]
int run_gather_conv(pcgc_ctx* ctx, int family, int k, int stride, int cin, int cout, const float* x, int n_in, const float* w_src,
                    const float* bias, int relu, int B, float* out) {
  cudaStream_t s = ctx_stream(ctx);
  const size_t wfloats = (size_t)k * k * k * cin * cout;
  float* wbuf = ctx_workspace(ctx, 0, wfloats * (family == 2 ? 8 : 1) + 64);
  if (!wbuf) return ctx_fail(ctx, PCGC_ERR_OOM, "train: weight workspace");
  ConvCall c;
  c.in = x; c.in_n = n_in; c.in_cs = cin; c.in_co = 0;
  c.out = out; c.out_cs = cout; c.out_co = 0;
  c.bias = bias; c.res = nullptr; c.res_cs = c.res_co = 0;
  c.flags = relu ? EPI_RELU : 0; c.floor_v = 0.f; c.B = B;
  if (family != 2) {
    const int out_n = n_in / stride;
    if (out_n % 8 != 0) return ctx_fail(ctx, PCGC_ERR_BAD_ARG, "train conv: output grid must be a multiple of 8");
    PackArgs p{family, k, family == 0 ? cin : cout, family == 0 ? cout : cin, {0, 0, 0}, {0, 0, 0}};
    const int total = (int)wfloats;
    pack_weights_kernel<<<(total + 255) / 256, 256, 0, s>>>(w_src, wbuf, p, total);
    ++*ctx_launches(ctx);
    ConvDesc& d = c.d;
    d.kz = d.ky = d.kx = k; d.stride = stride; d.pz = d.py = d.px = pad_before(k, stride);
    d.ostride = 1; d.oz = d.oy = d.ox = 0; d.cin = cin; d.cout = cout; d.w = wbuf;
    c.out_n = out_n; c.tn = out_n;
    TCK(launch_conv_ffma(c, s, ctx_launches(ctx)));
    return PCGC_OK;
  }
  // stride-2 transposed conv: 8 output-parity classes, each a stride-1 gather conv over the input grid
  if (stride != 2 || n_in % 8 != 0) return ctx_fail(ctx, PCGC_ERR_BAD_ARG, "train transposed conv: stride 2 and an input grid multiple of 8 only");
  const int pb = pad_before(k, 2);
  size_t off = 0;
  for (int cls = 0; cls < 8; ++cls) {
    const int r[3] = {(cls >> 2) & 1, (cls >> 1) & 1, cls & 1};
    PackArgs p{2, k, cout, cin, {0, 0, 0}, {r[0], r[1], r[2]}};
    int q0[3], o0[3], P[3];
    for (int a = 0; a < 3; ++a) {
      p.km[a] = (k - r[a] + 1) / 2;
      q0[a] = std::max(0, (pb - r[a] + 1) / 2);
      o0[a] = 2 * q0[a] + r[a] - pb;
      P[a] = (p.km[a] - 1) - q0[a];
    }
    const int total = p.km[0] * p.km[1] * p.km[2] * cin * cout;
    float* wc = wbuf + off;
    off += (size_t)((total + 3) & ~3);
    pack_weights_kernel<<<(total + 255) / 256, 256, 0, s>>>(w_src, wc, p, total);
    ++*ctx_launches(ctx);
    ConvDesc& d = c.d;
    d.kz = p.km[0]; d.ky = p.km[1]; d.kx = p.km[2]; d.stride = 1; d.pz = P[0]; d.py = P[1]; d.px = P[2];
    d.ostride = 2; d.oz = o0[0]; d.oy = o0[1]; d.ox = o0[2]; d.cin = cin; d.cout = cout; d.w = wc;
    c.out_n = 2 * n_in; c.tn = n_in;
    TCK(launch_conv_ffma(c, s, ctx_launches(ctx)));
  }
  return PCGC_OK;
}

// ---------------------------------------------------------------------------------------------- weight gradient
// dW[tap][cg][ca] = sum over anchor voxels v of T[S*v + tap - pad][cg] * A[v][ca].
// A block owns one tile of anchor voxels (4x8x8 for stride 1, 2x4x4 for stride 2), 16 gathered channels and 16 anchor channels:
// the A tile and the haloed T brick are staged in shared memory once and feed every tap.  A thread owns up to 7 "units" = (tap,
// gathered channel, quad of anchor channels) with 4 accumulators each; per voxel a unit costs one 4-byte and one 16-byte shared
// load for 4 FMAs.  Every (tap, cg, ca) of a tile is written by exactly one thread: partial[tile][tap][cg][ca], summed over the
// tiles in a fixed order by wgrad_reduce_kernel (deterministic, no atomics).  The first version (one thread per (cg, ca) pair
// looping over all voxels straight from global memory) took 2.3 s per training step of 8 cubes.
template <int S>
__global__ void __launch_bounds__(256)
wgrad_tile_kernel(const float* __restrict__ T, const float* __restrict__ A, int na, int nt, int cg, int ca, int k, int pad,
                  float* __restrict__ partial) {
  constexpr int TZ = S == 1 ? 4 : 2, TY = S == 1 ? 8 : 4, TX = S == 1 ? 8 : 4, NV = TZ * TY * TX;
  extern __shared__ float sm[];
  const int BZ = (TZ - 1) * S + k, BY = (TY - 1) * S + k, BX = (TX - 1) * S + k;
  float* sT = sm;                                   // [BZ*BY*BX][16]
  float* sA = sm + (size_t)BZ * BY * BX * 16;      // [NV][16]
  const int tiles_x = na / TX, tiles_y = na / TY, tiles_z = na / TZ;
  int tile = blockIdx.x;
  const int bx = tile % tiles_x; tile /= tiles_x;
  const int by = tile % tiles_y; tile /= tiles_y;
  const int bz = tile % tiles_z; const int b = tile / tiles_z;
  const int g0 = blockIdx.y * 16, a0 = blockIdx.z * 16;
  const int gn = min(16, cg - g0), an = min(16, ca - a0);
  const int z0 = bz * TZ, y0 = by * TY, x0 = bx * TX;
  // stage the A tile (zero padded to 16 channels) and the T brick (zero outside the grid = SAME padding / cropped output)
  for (int i = threadIdx.x; i < NV * 16; i += 256) {
    const int c = i & 15, v = i >> 4;
    const int x = v % TX, y = (v / TX) % TY, z = v / (TX * TY);
    float val = 0.f;
    if (c < an) val = __ldg(A + ((((size_t)b * na + z0 + z) * na + y0 + y) * na + x0 + x) * ca + a0 + c);
    sA[i] = val;
  }
  const int nb = BZ * BY * BX;
  for (int i = threadIdx.x; i < nb * 16; i += 256) {
    const int c = i & 15, v = i >> 4;
    const int x = v % BX, y = (v / BX) % BY, z = v / (BX * BY);
    const int gz = z0 * S - pad + z, gy = y0 * S - pad + y, gx = x0 * S - pad + x;
    float val = 0.f;
    if (c < gn && (unsigned)gz < (unsigned)nt && (unsigned)gy < (unsigned)nt && (unsigned)gx < (unsigned)nt)
      val = __ldg(T + ((((size_t)b * nt + gz) * nt + gy) * nt + gx) * cg + g0 + c);
    sT[i] = val;
  }
  __syncthreads();
  const int taps = k * k * k, quads = (an + 3) >> 2;
  const int units = taps * gn * quads;
  float* out = partial + (size_t)blockIdx.x * taps * cg * ca;
  for (int u = threadIdx.x; u < units; u += 256) {
    const int c = u % gn;                          // gathered channel fastest: lanes read consecutive words of one brick row
    const int q = (u / gn) % quads, tap = u / (gn * quads);
    const int kz = tap / (k * k), ky = (tap / k) % k, kx = tap % k;
    float acc0 = 0.f, acc1 = 0.f, acc2 = 0.f, acc3 = 0.f;
    const float* tp = sT + ((size_t)(kz * BY + ky) * BX + kx) * 16 + c;
    const float4* ap = reinterpret_cast<const float4*>(sA) + q;
#pragma unroll 1
    for (int z = 0; z < TZ; ++z)
#pragma unroll 1
      for (int y = 0; y < TY; ++y) {
        const float* tr = tp + ((size_t)(z * S * BY + y * S) * BX) * 16;
        const float4* ar = ap + (size_t)((z * TY + y) * TX) * 4;
#pragma unroll
        for (int x = 0; x < TX; ++x) {
          const float t = tr[x * S * 16];
          const float4 a4 = ar[x * 4];
          acc0 = fmaf(t, a4.x, acc0); acc1 = fmaf(t, a4.y, acc1); acc2 = fmaf(t, a4.z, acc2); acc3 = fmaf(t, a4.w, acc3);
        }
      }
    float* o = out + ((size_t)tap * cg + g0 + c) * ca + a0 + 4 * q;
    const int left = an - 4 * q;
    o[0] = acc0;
    if (left > 1) o[1] = acc1;
    if (left > 2) o[2] = acc2;
    if (left > 3) o[3] = acc3;
  }
}

// The same dW for the 9^3 layers of model_simple (conv_1, deconv_3: SURVEY.md 8d).  The tile kernel above writes one partial per
// anchor tile (764 MB for conv_1 at batch 8) and stages 16 gathered channels even when the layer has one.  Here:
//   * the anchor tiles (2x4x8 voxels) are cut into `slices` contiguous runs; a block owns one run and a fixed set of units, keeps
//     its accumulators in registers across the run and writes ONE partial per slice: partial[slice][tap][cg][ca].  The slice
//     count is a function of the layer shape only, so the workspace does not grow with the batch;
//   * a unit = (gathered channel, quad of anchor channels, kz, ky) with all k kx-taps: per row of 8 anchor voxels it loads the
//     (8-1)*S + k gathered values of the row once and 8 float4 of A, for 8 * k * 4 FMAs;
//   * only the channels that exist are staged: at most 8 gathered channels (a 1-channel side stages 1) and ceil(ca/4) quads.
// Accumulation order of every dW element: tiles of the slice in increasing order, voxels of a tile in (z, y, x) order, then the
// slices in increasing order (reduce_rows_kernel).  No atomics: two calls return the same bits.
constexpr int WGL_TZ = 2, WGL_TY = 4, WGL_TX = 8, WGL_GN = 8, WGL_THREADS = 128, WGL_MAX_SLICES = 128;

template <int K, int S>
__global__ void __launch_bounds__(WGL_THREADS)
wgrad_slice_kernel(const float* __restrict__ T, const float* __restrict__ A, int B, int na, int nt, int cg, int ca, int pad, int slices,
                   int ychunks, float* __restrict__ partial) {
  constexpr int TZ = WGL_TZ, TY = WGL_TY, TX = WGL_TX, NV = TZ * TY * TX;
  constexpr int BZ = (TZ - 1) * S + K, BY = (TY - 1) * S + K, BX = (TX - 1) * S + K, NB = BZ * BY * BX;
  constexpr int ROW = (TX - 1) * S + K;
  extern __shared__ float4 sm4[];
  const int quads = (ca + 3) >> 2, cap = quads * 4;
  float* sA = reinterpret_cast<float*>(sm4);                 // [NV][cap]
  const int chunk = blockIdx.y / ychunks;
  const int g0 = chunk * WGL_GN, gn = min(WGL_GN, cg - g0);
  float* sT = sA + NV * cap;                                 // [NB][gn]
  const int u = (blockIdx.y % ychunks) * WGL_THREADS + threadIdx.x;
  const bool active = u < gn * quads * K * K;
  const int c = u % gn, q = (u / gn) % quads, kzy = u / (gn * quads);
  const int kz = kzy / K, ky = kzy % K;
  const int tiles_x = na / TX, tiles_y = na / TY, tiles_z = na / TZ;
  const long long tiles = (long long)B * tiles_z * tiles_y * tiles_x;
  const long long t0 = tiles * blockIdx.x / slices, t1 = tiles * (blockIdx.x + 1) / slices;
  float acc[K][4];
#pragma unroll
  for (int j = 0; j < K; ++j) acc[j][0] = acc[j][1] = acc[j][2] = acc[j][3] = 0.f;
  for (long long tile = t0; tile < t1; ++tile) {
    long long t = tile;
    const int bx = (int)(t % tiles_x); t /= tiles_x;
    const int by = (int)(t % tiles_y); t /= tiles_y;
    const int bz = (int)(t % tiles_z); const int b = (int)(t / tiles_z);
    const int z0 = bz * TZ, y0 = by * TY, x0 = bx * TX;
    __syncthreads();                                         // the previous tile's readers are done
    for (int i = threadIdx.x; i < NV * cap; i += WGL_THREADS) {
      const int ch = i % cap, v = i / cap;
      const int x = v % TX, y = (v / TX) % TY, z = v / (TX * TY);
      float val = 0.f;
      if (ch < ca) val = __ldg(A + ((((size_t)b * na + z0 + z) * na + y0 + y) * na + x0 + x) * ca + ch);
      sA[i] = val;
    }
    for (int i = threadIdx.x; i < NB * gn; i += WGL_THREADS) {
      const int ch = i % gn, v = i / gn;
      const int x = v % BX, y = (v / BX) % BY, z = v / (BX * BY);
      const int gz = z0 * S - pad + z, gy = y0 * S - pad + y, gx = x0 * S - pad + x;
      float val = 0.f;
      if ((unsigned)gz < (unsigned)nt && (unsigned)gy < (unsigned)nt && (unsigned)gx < (unsigned)nt)
        val = __ldg(T + ((((size_t)b * nt + gz) * nt + gy) * nt + gx) * cg + g0 + ch);
      sT[i] = val;
    }
    __syncthreads();
    if (active) {
#pragma unroll 1
      for (int z = 0; z < TZ; ++z)
#pragma unroll 1
        for (int y = 0; y < TY; ++y) {
          const float* tr = sT + ((size_t)((z * S + kz) * BY + y * S + ky) * BX) * gn + c;
          float tv[ROW];
#pragma unroll
          for (int i = 0; i < ROW; ++i) tv[i] = tr[i * gn];
          const float4* ar = reinterpret_cast<const float4*>(sA + (size_t)(z * TY + y) * TX * cap) + q;
#pragma unroll
          for (int x = 0; x < TX; ++x) {
            const float4 a4 = ar[x * quads];
#pragma unroll
            for (int kx = 0; kx < K; ++kx) {
              const float tt = tv[x * S + kx];
              acc[kx][0] = fmaf(tt, a4.x, acc[kx][0]); acc[kx][1] = fmaf(tt, a4.y, acc[kx][1]);
              acc[kx][2] = fmaf(tt, a4.z, acc[kx][2]); acc[kx][3] = fmaf(tt, a4.w, acc[kx][3]);
            }
          }
        }
    }
  }
  if (!active) return;
  const int left = ca - 4 * q;
  float* out = partial + (size_t)blockIdx.x * K * K * K * cg * ca;
#pragma unroll
  for (int kx = 0; kx < K; ++kx) {
    float* o = out + ((size_t)(kzy * K + kx) * cg + g0 + c) * ca + 4 * q;
    o[0] = acc[kx][0];
    if (left > 1) o[1] = acc[kx][1];
    if (left > 2) o[2] = acc[kx][2];
    if (left > 3) o[3] = acc[kx][3];
  }
}

// dw[i] = sum over splits (fixed order) of partial[split][i]; transposed = 0: dw layout [tap][cg][ca] as is.
__global__ void wgrad_reduce_kernel(const float* __restrict__ partial, int splits, int total, float* __restrict__ dw) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= total) return;
  float s = 0.f;
  for (int k = 0; k < splits; ++k) s += partial[(size_t)k * total + i];
  dw[i] = s;
}

// out[grp][i] = sum (fixed order) of in[r][i] over the rows r of group grp (groups of `group` consecutive rows)
__global__ void reduce_rows_kernel(const float* __restrict__ in, int rows, int total, int group, float* __restrict__ out) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x, grp = blockIdx.y;
  if (i >= total) return;
  const int r0 = grp * group, r1 = min(rows, r0 + group);
  float s = 0.f;
  for (int r = r0; r < r1; ++r) s += in[(size_t)r * total + i];
  out[(size_t)grp * total + i] = s;
}

// db[c] = sum_v g[v][c], two fixed-order passes
__global__ void __launch_bounds__(256) bias_partial_kernel(const float* __restrict__ g, long long nvox, int c, int splits, float* __restrict__ partial) {
  __shared__ float s_acc[256];
  const int split = blockIdx.x;
  const long long v0 = nvox * split / splits, v1 = nvox * (split + 1) / splits;
  const int ch = threadIdx.x % c, lane_v = threadIdx.x / c, per = 256 / c;          // c <= 64 divides 256 for the model's widths (1..64 powers of 2)
  float acc = 0.f;
  if (lane_v < per)
    for (long long v = v0 + lane_v; v < v1; v += per) acc += __ldg(g + (size_t)v * c + ch);
  s_acc[threadIdx.x] = lane_v < per ? acc : 0.f;
  __syncthreads();
  if (threadIdx.x < c) {
    float s = 0.f;
    for (int j = 0; j < per; ++j) s += s_acc[j * c + threadIdx.x];
    partial[(size_t)split * c + threadIdx.x] = s;
  }
}

// ---------------------------------------------------------------------------------------------- element-wise pieces
__global__ void relu_backward_kernel(const float* __restrict__ g, const float* __restrict__ y, size_t n, float* __restrict__ out) {
  for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (size_t)gridDim.x * blockDim.x) out[i] = y[i] > 0.f ? g[i] : 0.f;
}
// _VoxceptionResNet merge (model_voxception.py:64-67): out = relu(x + concat[t12, t23]); x, out [nvox, c]; t12, t23 [nvox, c/2]
__global__ void vrn_merge_kernel(const float* __restrict__ x, const float* __restrict__ t12, const float* __restrict__ t23, size_t nvox, int c,
                                 float* __restrict__ out) {
  const int h = c / 2;
  for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < nvox * c; i += (size_t)gridDim.x * blockDim.x) {
    const size_t v = i / c; const int ch = (int)(i % c);
    const float t = ch < h ? t12[v * h + ch] : t23[v * h + ch - h];
    out[i] = fmaxf(x[i] + t, 0.f);
  }
}
__global__ void vrn_merge_backward_kernel(const float* __restrict__ g, const float* __restrict__ out, size_t nvox, int c, float* __restrict__ gx,
                                          float* __restrict__ g12, float* __restrict__ g23) {
  const int h = c / 2;
  for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < nvox * c; i += (size_t)gridDim.x * blockDim.x) {
    const size_t v = i / c; const int ch = (int)(i % c);
    const float gv = out[i] > 0.f ? g[i] : 0.f;
    gx[i] = gv;
    if (ch < h) g12[v * h + ch] = gv; else g23[v * h + ch - h] = gv;
  }
}
// scale = max(|s|, floor) (model_voxception.py:308 + train_hyper.py:191) and its gradient
__global__ void abs_floor_kernel(const float* __restrict__ s, size_t n, float fl, float* __restrict__ out) {
  for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (size_t)gridDim.x * blockDim.x) out[i] = fmaxf(fabsf(s[i]), fl);
}
__global__ void abs_floor_backward_kernel(const float* __restrict__ g, const float* __restrict__ s, size_t n, float fl, float* __restrict__ out) {
  for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (size_t)gridDim.x * blockDim.x) {
    const float a = fabsf(s[i]);
    out[i] = a >= fl ? (s[i] > 0.f ? g[i] : (s[i] < 0.f ? -g[i] : 0.f)) : 0.f;     // tf.maximum passes the gradient to x where x >= y
  }
}

// ---------------------------------------------------------------------------------------------- Laplace model, backward
// p = max(|c(u') - c(l')|, bound) as det_laplace_likelihood; loss term = coef * sum(log p) (coef = delta / (-ln 2 * num_points)).
// Adds nothing to the upstream gradient of y_t: the caller (the tape) sums the synthesis path's gradient with gy.
__global__ void laplace_backward_kernel(const float* __restrict__ yt, const float* __restrict__ loc, const float* __restrict__ scale, size_t n,
                                        float bound, float coef, float* __restrict__ gy, float* __restrict__ gloc, float* __restrict__ gscale) {
  for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (size_t)gridDim.x * blockDim.x) {
    const float x = yt[i], mu = loc[i], b = scale[i];
    const float u = x + 0.5f, l = x - 0.5f;
    const float sg = det_signf(u + l - mu);
    const float up = -sg * (u - mu) + mu, lp = -sg * (l - mu) + mu;
    const float cu = det_laplace_cdf(up, mu, b), cl = det_laplace_cdf(lp, mu, b);
    const float diff = cu - cl, p = fabsf(diff);
    float dy = 0.f, dm = 0.f, db = 0.f;
    if (p >= bound) {
      const float sp = det_signf(diff);
      const float fu = 0.5f / b * det_expf(-fabsf(up - mu) / b), fl = 0.5f / b * det_expf(-fabsf(lp - mu) / b);   // density at u', l'
      const float w = coef / p * sp;                       // d loss / d (c(u') - c(l'))
      dy = w * (-sg) * (fu - fl);
      dm = w * sg * (fu - fl);
      db = w * (-(fu * (up - mu)) + fl * (lp - mu)) / b;
    }
    gy[i] = dy; gloc[i] = dm; gscale[i] = db;
  }
}

// ---------------------------------------------------------------------------------------------- factorized model, train forward / backward
// Raw variables of entropy_model.py:42-68 per channel c (the pcgc_load_bottleneck order): matrices [C*3 | C*9 | C*9 | C*3],
// biases [C*3 | C*3 | C*3 | C], factors likewise.  Forward per element: z_t = z + noise, p = max(|sig(s*U) - sig(s*L)|, bound).
struct BnRaw { const float* m; const float* b; const float* f; int C; };

__device__ __forceinline__ float softplusf_(float x) { return x > 20.f ? x : (x < -20.f ? expf(x) : log1pf(expf(x))); }
__device__ __forceinline__ float sigm_(float x) { return 1.f / (1.f + expf(-x)); }

// logits of one value through the 1-3-3-3-1 network of channel c with activations kept for the backward pass
struct BnAct { float t0[3], h0[3], t1[3], h1[3], t2[3], h2[3], t3; };
struct BnPar { float m0[3], b0[3], f0[3], m1[9], b1[3], f1[3], m2[9], b2[3], f2[3], m3[3], b3, f3; };   // transformed: softplus(m), tanh(f)

__device__ __forceinline__ void bn_load(const BnRaw& r, int c, BnPar& p) {
  const int C = r.C;
  for (int j = 0; j < 3; ++j) { p.m0[j] = softplusf_(r.m[c * 3 + j]); p.b0[j] = r.b[c * 3 + j]; p.f0[j] = tanhf(r.f[c * 3 + j]); }
  for (int j = 0; j < 9; ++j) { p.m1[j] = softplusf_(r.m[3 * C + c * 9 + j]); p.m2[j] = softplusf_(r.m[12 * C + c * 9 + j]); }
  for (int j = 0; j < 3; ++j) {
    p.b1[j] = r.b[3 * C + c * 3 + j]; p.f1[j] = tanhf(r.f[3 * C + c * 3 + j]);
    p.b2[j] = r.b[6 * C + c * 3 + j]; p.f2[j] = tanhf(r.f[6 * C + c * 3 + j]);
    p.m3[j] = softplusf_(r.m[21 * C + c * 3 + j]);
  }
  p.b3 = r.b[9 * C + c]; p.f3 = tanhf(r.f[9 * C + c]);
}
__device__ __forceinline__ float bn_fwd(float x, const BnPar& p, BnAct& a) {
  for (int j = 0; j < 3; ++j) { a.t0[j] = p.m0[j] * x + p.b0[j]; a.h0[j] = a.t0[j] + p.f0[j] * tanhf(a.t0[j]); }
  for (int j = 0; j < 3; ++j) { a.t1[j] = p.m1[3 * j] * a.h0[0] + p.m1[3 * j + 1] * a.h0[1] + p.m1[3 * j + 2] * a.h0[2] + p.b1[j]; a.h1[j] = a.t1[j] + p.f1[j] * tanhf(a.t1[j]); }
  for (int j = 0; j < 3; ++j) { a.t2[j] = p.m2[3 * j] * a.h1[0] + p.m2[3 * j + 1] * a.h1[1] + p.m2[3 * j + 2] * a.h1[2] + p.b2[j]; a.h2[j] = a.t2[j] + p.f2[j] * tanhf(a.t2[j]); }
  a.t3 = p.m3[0] * a.h2[0] + p.m3[1] * a.h2[1] + p.m3[2] * a.h2[2] + p.b3;
  return a.t3 + p.f3 * tanhf(a.t3);
}
// backward of bn_fwd: d = d loss / d logit; accumulates gradients w.r.t. the TRANSFORMED parameters into gp, returns d loss / d x
__device__ __forceinline__ float bn_bwd(float x, float d, const BnPar& p, const BnAct& a, BnPar& gp) {
  float th = tanhf(a.t3);
  gp.f3 += d * th;
  float dt3 = d * (1.f + p.f3 * (1.f - th * th));
  gp.b3 += dt3;
  float dh2[3], dh1[3] = {0.f, 0.f, 0.f}, dh0[3] = {0.f, 0.f, 0.f};
  for (int k = 0; k < 3; ++k) { gp.m3[k] += dt3 * a.h2[k]; dh2[k] = dt3 * p.m3[k]; }
  for (int j = 0; j < 3; ++j) {
    th = tanhf(a.t2[j]);
    gp.f2[j] += dh2[j] * th;
    const float dt = dh2[j] * (1.f + p.f2[j] * (1.f - th * th));
    gp.b2[j] += dt;
    for (int k = 0; k < 3; ++k) { gp.m2[3 * j + k] += dt * a.h1[k]; dh1[k] += dt * p.m2[3 * j + k]; }
  }
  for (int j = 0; j < 3; ++j) {
    th = tanhf(a.t1[j]);
    gp.f1[j] += dh1[j] * th;
    const float dt = dh1[j] * (1.f + p.f1[j] * (1.f - th * th));
    gp.b1[j] += dt;
    for (int k = 0; k < 3; ++k) { gp.m1[3 * j + k] += dt * a.h0[k]; dh0[k] += dt * p.m1[3 * j + k]; }
  }
  float dx = 0.f;
  for (int j = 0; j < 3; ++j) {
    th = tanhf(a.t0[j]);
    gp.f0[j] += dh0[j] * th;
    const float dt = dh0[j] * (1.f + p.f0[j] * (1.f - th * th));
    gp.b0[j] += dt;
    gp.m0[j] += dt * x;
    dx += dt * p.m0[j];
  }
  return dx;
}

// Training forward of the EntropyBottleneck (entropy_model.py:153-181 with training=True): z_t = z + U(-1/2, 1/2) (the Philox
// stream of entropy.cu: element i draws word i % 4 of block i / 4), per-block partial sums of log max(p, bound) in double.
__global__ void __launch_bounds__(256)
factorized_train_forward_kernel(BnRaw r, const float* __restrict__ z, size_t n, uint64_t seed, float bound, float* __restrict__ zt,
                                double* __restrict__ partial) {
  __shared__ double s_r[256];
  const int C = r.C;
  double acc = 0.0;
  for (size_t i = (size_t)blockIdx.x * 256 + threadIdx.x; i < n; i += (size_t)gridDim.x * 256) {
    float u[4];
    noise4(seed, (uint64_t)(i >> 2), u);
    const float x = z[i] + u[i & 3];
    zt[i] = x;
    BnPar p; bn_load(r, (int)(i % C), p);
    BnAct a;
    const float lo = bn_fwd(x - 0.5f, p, a), up = bn_fwd(x + 0.5f, p, a);
    const float s = -det_signf(lo + up);
    const float pr = fmaxf(fabsf(sigm_(s * up) - sigm_(s * lo)), bound);
    acc += (double)logf(pr);
  }
  s_r[threadIdx.x] = acc;
  __syncthreads();
  if (threadIdx.x == 0) { double t = 0; for (int k = 0; k < 256; ++k) t += s_r[k]; partial[blockIdx.x] = t; }
}
__global__ void sum_double_kernel(const double* __restrict__ partial, int n, double* __restrict__ out) {
  if (threadIdx.x == 0 && blockIdx.x == 0) { double t = 0; for (int k = 0; k < n; ++k) t += partial[k]; out[0] = t; }
}

constexpr int BN_NP = sizeof(BnPar) / sizeof(float);       // 44 transformed parameters per channel, BnPar order

// One block per channel (C blocks); threads stride over the channel's elements.  Writes gz and the per-channel gradients w.r.t. the
// RAW variables (chain through softplus / tanh applied once per channel at the end), reduced over the block in a fixed order.
__global__ void __launch_bounds__(256)
factorized_backward_kernel(BnRaw r, const float* __restrict__ zt, size_t nvox, float bound, float coef, float* __restrict__ gz,
                           float* __restrict__ gm, float* __restrict__ gb, float* __restrict__ gf) {
  __shared__ float s_red[256];
  const int c = blockIdx.x, C = r.C;
  BnPar p; bn_load(r, c, p);
  BnPar gp;
  float* gpf = reinterpret_cast<float*>(&gp);
  for (int i = 0; i < BN_NP; ++i) gpf[i] = 0.f;
  for (size_t v = threadIdx.x; v < nvox; v += 256) {
    const float x = zt[v * C + c];
    BnAct al, au;
    const float lo = bn_fwd(x - 0.5f, p, al), up = bn_fwd(x + 0.5f, p, au);
    const float s = -det_signf(lo + up);
    const float su = sigm_(s * up), sl = sigm_(s * lo);
    const float diff = su - sl, pr = fabsf(diff);
    float dx = 0.f;
    if (pr >= bound) {
      const float w = coef / pr * det_signf(diff);
      const float dup = w * su * (1.f - su) * s, dlo = -w * sl * (1.f - sl) * s;
      dx = bn_bwd(x + 0.5f, dup, p, au, gp) + bn_bwd(x - 0.5f, dlo, p, al, gp);
    }
    gz[v * C + c] = dx;
  }
  // block reduction of the 58 accumulators, fixed order; thread 0 applies the chain rule to the raw variables
  float total[BN_NP];
  for (int i = 0; i < BN_NP; ++i) {
    s_red[threadIdx.x] = gpf[i];
    __syncthreads();
    if (threadIdx.x == 0) { float s = 0.f; for (int t = 0; t < 256; ++t) s += s_red[t]; total[i] = s; }
    __syncthreads();
  }
  if (threadIdx.x == 0) {
    const BnPar& g = *reinterpret_cast<const BnPar*>(total);
    auto dsp = [](float raw) { return 1.f / (1.f + expf(-raw)); };                 // d softplus / d raw
    auto dth = [](float raw) { const float t = tanhf(raw); return 1.f - t * t; };   // d tanh / d raw
    for (int j = 0; j < 3; ++j) {
      gm[c * 3 + j] = g.m0[j] * dsp(r.m[c * 3 + j]); gb[c * 3 + j] = g.b0[j]; gf[c * 3 + j] = g.f0[j] * dth(r.f[c * 3 + j]);
      gb[3 * C + c * 3 + j] = g.b1[j]; gf[3 * C + c * 3 + j] = g.f1[j] * dth(r.f[3 * C + c * 3 + j]);
      gb[6 * C + c * 3 + j] = g.b2[j]; gf[6 * C + c * 3 + j] = g.f2[j] * dth(r.f[6 * C + c * 3 + j]);
      gm[21 * C + c * 3 + j] = g.m3[j] * dsp(r.m[21 * C + c * 3 + j]);
    }
    for (int j = 0; j < 9; ++j) {
      gm[3 * C + c * 9 + j] = g.m1[j] * dsp(r.m[3 * C + c * 9 + j]);
      gm[12 * C + c * 9 + j] = g.m2[j] * dsp(r.m[12 * C + c * 9 + j]);
    }
    gb[9 * C + c] = g.b3; gf[9 * C + c] = g.f3 * dth(r.f[9 * C + c]);
  }
}

// ---------------------------------------------------------------------------------------------- BCE occupancy loss (loss.py:8-33)
// sums[0] = sum over empty voxels of -log(1 - occ), sums[1] = sum over occupied voxels of -log(occ), sums[2] = #empty, sums[3] = #occupied
__global__ void __launch_bounds__(256) bce_partial_kernel(const float* __restrict__ logits, const uint8_t* __restrict__ label, size_t n, double* __restrict__ partial) {
  __shared__ double s_r[4][256];
  double a[4] = {0, 0, 0, 0};
  for (size_t i = (size_t)blockIdx.x * 256 + threadIdx.x; i < n; i += (size_t)gridDim.x * 256) {
    const float occ = fminf(fmaxf(sigm_(logits[i]), 1e-7f), 1.0f - 1e-7f);
    if (label[i]) { a[1] -= (double)logf(occ); a[3] += 1.0; } else { a[0] -= (double)logf(1.0f - occ); a[2] += 1.0; }
  }
  for (int k = 0; k < 4; ++k) s_r[k][threadIdx.x] = a[k];
  __syncthreads();
  if (threadIdx.x < 4) { double s = 0; for (int t = 0; t < 256; ++t) s += s_r[threadIdx.x][t]; partial[(size_t)blockIdx.x * 4 + threadIdx.x] = s; }
}
__global__ void bce_final_kernel(const double* __restrict__ partial, int blocks, double* __restrict__ sums) {
  if (threadIdx.x < 4) { double s = 0; for (int b = 0; b < blocks; ++b) s += partial[(size_t)b * 4 + threadIdx.x]; sums[threadIdx.x] = s; }
}
// g = d (w_empty * mean_empty + w_full * mean_full) / d logits, sums from bce_final_kernel (device: no host round trip)
__global__ void bce_backward_kernel(const float* __restrict__ logits, const uint8_t* __restrict__ label, size_t n, const double* __restrict__ sums,
                                    float w_empty, float w_full, float* __restrict__ g) {
  const float ce = sums[2] > 0 ? w_empty / (float)sums[2] : 0.f, cf = sums[3] > 0 ? w_full / (float)sums[3] : 0.f;
  for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (size_t)gridDim.x * blockDim.x) {
    const float sg = sigm_(logits[i]);
    const bool inside = sg >= 1e-7f && sg <= 1.0f - 1e-7f;          // tf.clip_by_value: zero gradient outside the range
    // d(-log(1 - s))/dx = s ; d(-log s)/dx = -(1 - s)
    g[i] = inside ? (label[i] ? -cf * (1.f - sg) : ce * sg) : 0.f;
  }
}

// ---------------------------------------------------------------------------------------------- focal occupancy loss (loss.py:83-93)
// get_focal_loss(y_pred, y_true, gamma, alpha) on y_pred = sigmoid(logits) (the reference's function takes probabilities; its
// synthesis transform ends without an activation, so the sigmoid of get_bce_loss is applied first):
//   pt_1 = clip(label == 1 ? p : 1, 1e-3, .999), pt_0 = clip(label == 0 ? p : 0, 1e-3, .999)
//   loss = -sum(alpha (1 - pt_1)^gamma log pt_1) - sum((1 - alpha) pt_0^gamma log(1 - pt_0))            (a SUM, not a mean)
// The "other" branch of each tf.where is a constant after the clip (pt_1 = .999 on empty voxels, pt_0 = 1e-3 on occupied ones) and
// is part of the reference's value, so it is part of this one.  sums[0] = first sum, sums[1] = second sum.
__device__ __forceinline__ void focal_terms(float p, bool occupied, float gamma, float alpha, float& t1, float& t0) {
  const float pt1 = fminf(fmaxf(occupied ? p : 1.0f, 1e-3f), 0.999f), pt0 = fminf(fmaxf(occupied ? 0.0f : p, 1e-3f), 0.999f);
  t1 = -alpha * powf(1.0f - pt1, gamma) * logf(pt1);
  t0 = -(1.0f - alpha) * powf(pt0, gamma) * logf(1.0f - pt0);
}
__global__ void __launch_bounds__(256) focal_partial_kernel(const float* __restrict__ logits, const uint8_t* __restrict__ label, size_t n, float gamma,
                                                            float alpha, double* __restrict__ partial) {
  __shared__ double s_r[2][256];
  double a0 = 0, a1 = 0;
  for (size_t i = (size_t)blockIdx.x * 256 + threadIdx.x; i < n; i += (size_t)gridDim.x * 256) {
    float t1, t0;
    focal_terms(sigm_(logits[i]), label[i] != 0, gamma, alpha, t1, t0);
    a0 += (double)t1; a1 += (double)t0;
  }
  s_r[0][threadIdx.x] = a0; s_r[1][threadIdx.x] = a1;
  __syncthreads();
  if (threadIdx.x < 2) { double s = 0; for (int t = 0; t < 256; ++t) s += s_r[threadIdx.x][t]; partial[(size_t)blockIdx.x * 2 + threadIdx.x] = s; }
}
__global__ void focal_final_kernel(const double* __restrict__ partial, int blocks, double* __restrict__ sums) {
  if (threadIdx.x < 2) { double s = 0; for (int b = 0; b < blocks; ++b) s += partial[(size_t)b * 2 + threadIdx.x]; sums[threadIdx.x] = s; }
}
// g = weight * d loss / d logits; K.clip has a zero gradient outside [1e-3, .999]
__global__ void focal_backward_kernel(const float* __restrict__ logits, const uint8_t* __restrict__ label, size_t n, float gamma, float alpha,
                                      float weight, float* __restrict__ g) {
  for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (size_t)gridDim.x * blockDim.x) {
    const float p = sigm_(logits[i]);
    float d = 0.f;                                                   // d loss / d p
    if (p >= 1e-3f && p <= 0.999f) {
      const float q = 1.0f - p;
      if (label[i]) d = alpha * (gamma * powf(q, gamma - 1.0f) * logf(p) - powf(q, gamma) / p);
      else d = (1.0f - alpha) * (powf(p, gamma) / q - gamma * powf(p, gamma - 1.0f) * logf(q));
    }
    g[i] = weight * d * p * (1.0f - p);
  }
}

// ---------------------------------------------------------------------------------------------- Adam (tf.train.AdamOptimizer)
__global__ void adam_kernel(float* __restrict__ p, const float* __restrict__ g, float* __restrict__ m, float* __restrict__ v, size_t n, float lr_t,
                            float b1, float b2, float eps) {
  for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (size_t)gridDim.x * blockDim.x) {
    const float gi = g[i];
    const float mi = b1 * m[i] + (1.f - b1) * gi, vi = b2 * v[i] + (1.f - b2) * gi * gi;
    m[i] = mi; v[i] = vi;
    p[i] -= lr_t * mi / (sqrtf(vi) + eps);
  }
}

inline int ew_blocks(size_t n) { return (int)std::min<size_t>((n + 255) / 256, 148 * 16); }

}  // namespace
}  // namespace pcgc

using namespace pcgc;

extern "C" {

int pcgc_train_conv_forward(pcgc_ctx* ctx, const float* x, int B, int n, int cin, int cout, int k, int stride, int transposed,
                            const float* w_keras, const float* bias, int relu, float* out) {
  if (!ctx || !x || !w_keras || !out || B < 1) return PCGC_ERR_BAD_ARG;
  ctx_prof_begin(ctx, "train_conv_fwd", 2.0 * B * pow((double)(transposed ? n : n / stride), 3) * k * k * k * cin * cout, 0);
  const int r = run_gather_conv(ctx, transposed ? 2 : 0, k, stride, cin, cout, x, n, w_keras, bias, relu, B, out);
  ctx_prof_end(ctx);
  return r;
}

/* dx of y = conv(x): g [B, n_out^3, cout] -> dx [B, n^3, cin]; n = the layer's INPUT grid. */
int pcgc_train_conv_dgrad(pcgc_ctx* ctx, const float* g, int B, int n, int cin, int cout, int k, int stride, int transposed,
                          const float* w_keras, float* dx) {
  if (!ctx || !g || !w_keras || !dx || B < 1) return PCGC_ERR_BAD_ARG;
  ctx_prof_begin(ctx, "train_conv_dgrad", 2.0 * B * pow((double)(transposed ? n : n / stride), 3) * k * k * k * cin * cout, 0);
  int r;
  if (transposed) r = run_gather_conv(ctx, 0, k, stride, cout, cin, g, n * stride, w_keras, nullptr, 0, B, dx);            // adjoint of convT = the s2 conv, same array
  else if (stride == 1) r = run_gather_conv(ctx, 1, k, 1, cout, cin, g, n, w_keras, nullptr, 0, B, dx);                    // flipped taps, swapped channels
  else r = run_gather_conv(ctx, 2, k, stride, cout, cin, g, n / stride, w_keras, nullptr, 0, B, dx);                       // adjoint of the s2 conv = convT, same array
  ctx_prof_end(ctx);
  return r;
}

}  // extern "C"

namespace {

// The slice form takes k in {3, 5, 9} (the model's extents) and up to 64 anchor channels (the staged A tile).
bool slice_form_supported(int k, int ca) { return (k == 3 || k == 5 || k == 9) && ca >= 1 && ca <= 64; }

// Slice count of the slice form: enough blocks for ~4 per SM, from the layer shape only (never from the batch).
int slice_count(int k, int cg, int ca, int* ychunks) {
  const int quads = (ca + 3) / 4, gmax = std::min(cg, WGL_GN);
  *ychunks = (gmax * quads * k * k + WGL_THREADS - 1) / WGL_THREADS;
  const int ys = *ychunks * ((cg + WGL_GN - 1) / WGL_GN);
  return std::max(1, std::min(WGL_MAX_SLICES, (148 * 4 + ys - 1) / ys));
}

template <int K, int S>
cudaError_t launch_slice(dim3 grid, size_t smem, cudaStream_t s, const float* T, const float* A, int B, int na, int nt, int cg, int ca,
                         int pad, int slices, int ychunks, float* partial) {
  cudaError_t e = cudaFuncSetAttribute(wgrad_slice_kernel<K, S>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
  if (e != cudaSuccess) return e;
  wgrad_slice_kernel<K, S><<<grid, WGL_THREADS, smem, s>>>(T, A, B, na, nt, cg, ca, pad, slices, ychunks, partial);
  return cudaGetLastError();
}

// dW (and db when non-null) of one layer by the given form (0 = tile kernel, 1 = slice kernel); *partial_floats (nullable) = the
// size of the partial buffer the form used.
int wgrad_run(pcgc_ctx* ctx, int form, const float* x, const float* g, int B, int n, int cin, int cout, int k, int stride, int transposed,
              float* dw, float* db, int64_t* partial_floats) {
  cudaStream_t s = ctx_stream(ctx);
  // anchor grid / tensors: conv: A = g (n/stride, cout), T = x (n, cin), dW[tap][cin][cout];  convT: A = x (n, cin), T = g (n*stride, cout), dW[tap][cout][cin]
  const int na = transposed ? n : n / stride, nt = transposed ? n * stride : n;
  const int ca = transposed ? cin : cout, cg = transposed ? cout : cin;
  const float* A = transposed ? x : g; const float* T = transposed ? g : x;
  const int taps = k * k * k, pairs = cg * ca, total = taps * pairs;
  const long long va = (long long)B * na * na * na;
  if ((stride != 1 && stride != 2) || na % 8 != 0) return ctx_fail(ctx, PCGC_ERR_BAD_ARG, "train wgrad: stride 1 or 2 and an anchor grid multiple of 8");
  if (form == 1 && !slice_form_supported(k, ca)) return ctx_fail(ctx, PCGC_ERR_BAD_ARG, "train wgrad: the slice form takes k in {3,5,9} and <= 64 anchor channels");
  int64_t rows;                                                      // partial rows the fixed-order passes sum
  if (form == 1) {
    int ychunks;
    const int slices = slice_count(k, cg, ca, &ychunks);
    float* partial = ctx_workspace(ctx, 1, (size_t)slices * total + 64);
    if (!partial) return ctx_fail(ctx, PCGC_ERR_OOM, "train: wgrad workspace");
    constexpr int NV = WGL_TZ * WGL_TY * WGL_TX;
    const size_t brick = (size_t)((WGL_TZ - 1) * stride + k) * ((WGL_TY - 1) * stride + k) * ((WGL_TX - 1) * stride + k);
    const size_t smem = ((size_t)NV * ((ca + 3) & ~3) + brick * std::min(cg, WGL_GN)) * sizeof(float);
    const dim3 grid(slices, ychunks * ((cg + WGL_GN - 1) / WGL_GN));
    const int pad = pad_before(k, stride);
    ctx_prof_begin(ctx, "train_conv_wgrad_large", 2.0 * va * taps * pairs, 0);
    cudaError_t e;
#define PCGC_SLICE(KV, SV) e = launch_slice<KV, SV>(grid, smem, s, T, A, B, na, nt, cg, ca, pad, slices, ychunks, partial)
    if (stride == 1) { if (k == 3) PCGC_SLICE(3, 1); else if (k == 5) PCGC_SLICE(5, 1); else PCGC_SLICE(9, 1); }
    else { if (k == 3) PCGC_SLICE(3, 2); else if (k == 5) PCGC_SLICE(5, 2); else PCGC_SLICE(9, 2); }
#undef PCGC_SLICE
    TCK(e);
    reduce_rows_kernel<<<dim3((total + 255) / 256, 1), 256, 0, s>>>(partial, slices, total, slices, dw);
    *ctx_launches(ctx) += 2;
    rows = slices;
  } else {
    const int tz = stride == 1 ? 4 : 2, ty = stride == 1 ? 8 : 4, tx = stride == 1 ? 8 : 4;
    const int tiles = B * (na / tz) * (na / ty) * (na / tx);
    float* partial = ctx_workspace(ctx, 1, (size_t)tiles * taps * pairs + 64);
    if (!partial) return ctx_fail(ctx, PCGC_ERR_OOM, "train: wgrad workspace");
    const size_t brick = (size_t)((tz - 1) * stride + k) * ((ty - 1) * stride + k) * ((tx - 1) * stride + k);
    const size_t smem = (brick * 16 + (size_t)tz * ty * tx * 16) * sizeof(float);
    ctx_prof_begin(ctx, "train_conv_wgrad", 2.0 * va * taps * pairs, 0);
    const dim3 grid(tiles, (cg + 15) / 16, (ca + 15) / 16);
    if (stride == 1) {
      TCK(cudaFuncSetAttribute(wgrad_tile_kernel<1>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
      wgrad_tile_kernel<1><<<grid, 256, smem, s>>>(T, A, na, nt, cg, ca, k, pad_before(k, stride), partial);
    } else {
      TCK(cudaFuncSetAttribute(wgrad_tile_kernel<2>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
      wgrad_tile_kernel<2><<<grid, 256, smem, s>>>(T, A, na, nt, cg, ca, k, pad_before(k, stride), partial);
    }
    // fixed-order two-level sum over the tiles: groups of 64 tiles, then the group sums
    const int group = 64, ngrp = (tiles + group - 1) / group;
    float* p2 = ctx_workspace(ctx, 2, (size_t)ngrp * total + (size_t)64 * 64 + 64);
    if (!p2) return ctx_fail(ctx, PCGC_ERR_OOM, "train: wgrad reduce workspace");
    reduce_rows_kernel<<<dim3((total + 255) / 256, ngrp), 256, 0, s>>>(partial, tiles, total, group, p2);
    reduce_rows_kernel<<<dim3((total + 255) / 256, 1), 256, 0, s>>>(p2, ngrp, total, ngrp, dw);
    *ctx_launches(ctx) += 3;
    rows = tiles;
  }
  if (db) {
    const int no = transposed ? n * stride : n / stride;
    const long long vo = (long long)B * no * no * no;
    if (cout > 64 || 256 % cout) return ctx_fail(ctx, PCGC_ERR_BAD_ARG, "train bias grad: cout must divide 256");
    const int bs = (int)std::max<long long>(1, std::min<long long>(592, vo / 256));
    float* bp = ctx_workspace(ctx, 2, (size_t)bs * cout + 64);
    if (!bp) return ctx_fail(ctx, PCGC_ERR_OOM, "train: bias workspace");
    bias_partial_kernel<<<bs, 256, 0, s>>>(g, vo, cout, bs, bp);
    wgrad_reduce_kernel<<<1, 64, 0, s>>>(bp, bs, cout, db);
    *ctx_launches(ctx) += 2;
  }
  ctx_prof_end(ctx);
  TCK(cudaGetLastError());
  if (partial_floats) *partial_floats = rows * total;
  return PCGC_OK;
}

}  // namespace

extern "C" {

/* dw (Keras layout of the layer) and db (nullable) from the layer input x [B,n^3,cin] and the output gradient g. */
int pcgc_train_conv_wgrad(pcgc_ctx* ctx, const float* x, const float* g, int B, int n, int cin, int cout, int k, int stride,
                          int transposed, float* dw, float* db) {
  if (!ctx || !x || !g || !dw || B < 1) return PCGC_ERR_BAD_ARG;
  // The slice kernel for k = 9 (conv_1 / deconv_3 of model_simple: 1.16 ms against 6.06 ms for the tile kernel at batch 8 on a
  // B200); every other layer keeps the tile kernel -- k <= 3 (every Voxception layer) and k = 5, where the tile kernel measured
  // faster (conv_2 / deconv_2: 0.92 ms against 3.18 ms).
  const int form = k == 9 && slice_form_supported(k, transposed ? cin : cout) ? 1 : 0;
  return wgrad_run(ctx, form, x, g, B, n, cin, cout, k, stride, transposed, dw, db, nullptr);
}

/* pcgc_train_conv_wgrad with the dW form forced (0 = tile kernel, 1 = slice kernel), for tests and benchmarks. */
int pcgc_debug_train_wgrad(pcgc_ctx* ctx, int form, const float* x, const float* g, int B, int n, int cin, int cout, int k, int stride,
                           int transposed, float* dw, float* db, int64_t* partial_floats) {
  if (!ctx || !x || !g || !dw || B < 1 || (form != 0 && form != 1)) return PCGC_ERR_BAD_ARG;
  return wgrad_run(ctx, form, x, g, B, n, cin, cout, k, stride, transposed, dw, db, partial_floats);
}

int pcgc_train_relu_backward(pcgc_ctx* ctx, const float* g, const float* y, int64_t n, float* out) {
  if (!ctx || !g || !y || !out || n < 0) return PCGC_ERR_BAD_ARG;
  if (n) { relu_backward_kernel<<<ew_blocks(n), 256, 0, ctx_stream(ctx)>>>(g, y, (size_t)n, out); ++*ctx_launches(ctx); }
  return PCGC_OK;
}

int pcgc_train_vrn_merge(pcgc_ctx* ctx, const float* x, const float* t12, const float* t23, int64_t nvox, int c, float* out) {
  if (!ctx || !x || !t12 || !t23 || !out || c < 2 || (c & 1)) return PCGC_ERR_BAD_ARG;
  if (nvox) { vrn_merge_kernel<<<ew_blocks(nvox * c), 256, 0, ctx_stream(ctx)>>>(x, t12, t23, (size_t)nvox, c, out); ++*ctx_launches(ctx); }
  return PCGC_OK;
}

int pcgc_train_vrn_merge_backward(pcgc_ctx* ctx, const float* g, const float* out, int64_t nvox, int c, float* gx, float* g12, float* g23) {
  if (!ctx || !g || !out || !gx || !g12 || !g23 || c < 2 || (c & 1)) return PCGC_ERR_BAD_ARG;
  if (nvox) { vrn_merge_backward_kernel<<<ew_blocks(nvox * c), 256, 0, ctx_stream(ctx)>>>(g, out, (size_t)nvox, c, gx, g12, g23); ++*ctx_launches(ctx); }
  return PCGC_OK;
}

int pcgc_train_abs_floor(pcgc_ctx* ctx, const float* s, int64_t n, float floor_v, float* out) {
  if (!ctx || !s || !out) return PCGC_ERR_BAD_ARG;
  if (n) { abs_floor_kernel<<<ew_blocks(n), 256, 0, ctx_stream(ctx)>>>(s, (size_t)n, floor_v, out); ++*ctx_launches(ctx); }
  return PCGC_OK;
}

int pcgc_train_abs_floor_backward(pcgc_ctx* ctx, const float* g, const float* s, int64_t n, float floor_v, float* out) {
  if (!ctx || !g || !s || !out) return PCGC_ERR_BAD_ARG;
  if (n) { abs_floor_backward_kernel<<<ew_blocks(n), 256, 0, ctx_stream(ctx)>>>(g, s, (size_t)n, floor_v, out); ++*ctx_launches(ctx); }
  return PCGC_OK;
}

int pcgc_train_laplace_backward(pcgc_ctx* ctx, const float* y_t, const float* loc, const float* scale, int64_t n, float bound, float coef,
                                float* gy, float* gloc, float* gscale) {
  if (!ctx || !y_t || !loc || !scale || !gy || !gloc || !gscale) return PCGC_ERR_BAD_ARG;
  if (n) { laplace_backward_kernel<<<ew_blocks(n), 256, 0, ctx_stream(ctx)>>>(y_t, loc, scale, (size_t)n, bound, coef, gy, gloc, gscale); ++*ctx_launches(ctx); }
  return PCGC_OK;
}

int pcgc_train_factorized_forward(pcgc_ctx* ctx, const float* matrices, const float* biases, const float* factors, int C, const float* z,
                                  int64_t nvox, uint64_t seed, float bound, float* z_t, double* logsum_dev) {
  if (!ctx || !matrices || !biases || !factors || !z || !z_t || !logsum_dev || C < 1 || nvox < 1) return PCGC_ERR_BAD_ARG;
  const size_t n = (size_t)nvox * C;
  const int blocks = (int)std::min<size_t>((n + 255) / 256, 592);
  double* partial = reinterpret_cast<double*>(ctx_workspace(ctx, 3, (size_t)blocks * 2 + 64));
  if (!partial) return ctx_fail(ctx, PCGC_ERR_OOM, "train: factorized workspace");
  BnRaw r{matrices, biases, factors, C};
  factorized_train_forward_kernel<<<blocks, 256, 0, ctx_stream(ctx)>>>(r, z, n, seed, bound, z_t, partial);
  sum_double_kernel<<<1, 32, 0, ctx_stream(ctx)>>>(partial, blocks, logsum_dev);
  *ctx_launches(ctx) += 2;
  return PCGC_OK;
}

int pcgc_train_factorized_backward(pcgc_ctx* ctx, const float* matrices, const float* biases, const float* factors, int C, const float* z_t,
                                   int64_t nvox, float bound, float coef, float* gz, float* gmatrices, float* gbiases, float* gfactors) {
  if (!ctx || !matrices || !biases || !factors || !z_t || !gz || !gmatrices || !gbiases || !gfactors || C < 1) return PCGC_ERR_BAD_ARG;
  BnRaw r{matrices, biases, factors, C};
  factorized_backward_kernel<<<C, 256, 0, ctx_stream(ctx)>>>(r, z_t, (size_t)nvox, bound, coef, gz, gmatrices, gbiases, gfactors);
  ++*ctx_launches(ctx);
  return PCGC_OK;
}

/* sums_dev double[4] = {sum_empty(-log(1-occ)), sum_full(-log occ), #empty, #full}; losses: empty = s0/s2, full = s1/s3. */
int pcgc_train_bce(pcgc_ctx* ctx, const float* logits, const uint8_t* label, int64_t n, double* sums_dev) {
  if (!ctx || !logits || !label || !sums_dev || n < 1) return PCGC_ERR_BAD_ARG;
  const int blocks = ew_blocks(n);
  double* partial = reinterpret_cast<double*>(ctx_workspace(ctx, 3, (size_t)blocks * 8 + 64));
  if (!partial) return ctx_fail(ctx, PCGC_ERR_OOM, "train: bce workspace");
  bce_partial_kernel<<<blocks, 256, 0, ctx_stream(ctx)>>>(logits, label, (size_t)n, partial);
  bce_final_kernel<<<1, 32, 0, ctx_stream(ctx)>>>(partial, blocks, sums_dev);
  *ctx_launches(ctx) += 2;
  return PCGC_OK;
}

int pcgc_train_bce_backward(pcgc_ctx* ctx, const float* logits, const uint8_t* label, int64_t n, const double* sums_dev, float w_empty,
                            float w_full, float* g) {
  if (!ctx || !logits || !label || !sums_dev || !g || n < 1) return PCGC_ERR_BAD_ARG;
  bce_backward_kernel<<<ew_blocks(n), 256, 0, ctx_stream(ctx)>>>(logits, label, (size_t)n, sums_dev, w_empty, w_full, g);
  ++*ctx_launches(ctx);
  return PCGC_OK;
}

/* get_focal_loss (loss.py:83-93) on sigmoid(logits): sums_dev double[2] = {-sum(alpha (1-pt_1)^gamma log pt_1), -sum((1-alpha) pt_0^gamma log(1-pt_0))}. */
int pcgc_train_focal(pcgc_ctx* ctx, const float* logits, const uint8_t* label, int64_t n, float gamma, float alpha, double* sums_dev) {
  if (!ctx || !logits || !label || !sums_dev || n < 1 || !(gamma >= 1.0f) || !(alpha >= 0.0f && alpha <= 1.0f)) return PCGC_ERR_BAD_ARG;
  const int blocks = ew_blocks(n);
  double* partial = reinterpret_cast<double*>(ctx_workspace(ctx, 3, (size_t)blocks * 4 + 64));
  if (!partial) return ctx_fail(ctx, PCGC_ERR_OOM, "train: focal workspace");
  focal_partial_kernel<<<blocks, 256, 0, ctx_stream(ctx)>>>(logits, label, (size_t)n, gamma, alpha, partial);
  focal_final_kernel<<<1, 32, 0, ctx_stream(ctx)>>>(partial, blocks, sums_dev);
  *ctx_launches(ctx) += 2;
  return PCGC_OK;
}

int pcgc_train_focal_backward(pcgc_ctx* ctx, const float* logits, const uint8_t* label, int64_t n, float gamma, float alpha, float weight,
                              float* g) {
  if (!ctx || !logits || !label || !g || n < 1 || !(gamma >= 1.0f) || !(alpha >= 0.0f && alpha <= 1.0f)) return PCGC_ERR_BAD_ARG;
  focal_backward_kernel<<<ew_blocks(n), 256, 0, ctx_stream(ctx)>>>(logits, label, (size_t)n, gamma, alpha, weight, g);
  ++*ctx_launches(ctx);
  return PCGC_OK;
}

int pcgc_train_adam(pcgc_ctx* ctx, float* p, const float* g, float* m, float* v, int64_t n, float lr_t, float beta1, float beta2, float eps) {
  if (!ctx || !p || !g || !m || !v || n < 0) return PCGC_ERR_BAD_ARG;
  if (n) { adam_kernel<<<ew_blocks(n), 256, 0, ctx_stream(ctx)>>>(p, g, m, v, (size_t)n, lr_t, beta1, beta2, eps); ++*ctx_launches(ctx); }
  return PCGC_OK;
}

}  // extern "C"
