// FP32 CUDA-core convolution for every Conv3D / Conv3DTranspose shape of the reference
// (models/model_voxception.py:21-54,83-122,153-192,224-297; models/model_simple.py:21-86).
//
// One kernel template covers them all: a stride-S gather convolution with a (KZ,KY,KX) tap box
// over a channels-last grid.  A CTA owns an 8x8x8 tile of outputs; the haloed input brick of CC
// input channels is staged channel-planar in shared memory, the matching weight slab
// [KY][KX][CC][KZ][CoutBlock] beside it.  A thread owns one (x,y) column: 4 consecutive z outputs
// x CT output channels in registers, sliding a (3S+KZ)-deep register window along z so every
// staged input is read from shared memory once per (ky,kx,ci).  The reduction order
// (ci-chunk, ky, kx, ci, kz) is fixed and independent of batch size and grid => bit-reproducible
// (the property README.md:111-114 / eval.py:96-100 lack).  Epilogue: +bias, ReLU, residual add+ReLU
// (the VRN block's concat/add/relu, model_voxception.py:64-67), |.| and floor (HyperDecoder scale).
//
// This is the exact-FP32 engine: used for layers the tcgen05 engine does not take (stride 2,
// transposed, 1^3, Cin=1, k=5/9) and as the on-device cross-check for the tcgen05 engine.
#include "common.cuh"
#include "pm_format.cuh"

namespace pcgc {

struct FfmaArgs {
  const float* in; float* out; const float* w; const float* bias; const float* res;
  int in_n, in_cs, in_co;
  int out_n, out_cs, out_co;
  int res_cs, res_co;
  int tn;                 // t-grid edge (multiple of 8)
  int ky, kx;             // runtime tap extents (kz is a template parameter)
  int pz, py, px;
  int ostride, oz, oy, ox;
  int cin, cout;
  int cc;                 // input channels staged per chunk
  int plane;              // padded floats per staged channel plane
  int ey, ex, exp_;       // brick extents (y, x) and padded x pitch
  int flags; float floor_v;
  const __nv_bfloat16* in_pm; __nv_bfloat16* out_pm;
  int class_mode, cls_o0a, cls_o0b;   // see ConvDesc::class_mode
};

template <int KZ, int S, int CT>
__global__ void __launch_bounds__(512) conv_ffma_kernel(const FfmaArgs a) {
  constexpr int EZ = 7 * S + KZ;
  constexpr int WIN = 3 * S + KZ;
  extern __shared__ float smem[];
  const int G = blockDim.y;
  const int CB = G * CT;                         // couts handled by this CTA
  float* s_in = smem;
  float* s_w = smem + ((a.cc * a.plane + 3) & ~3);      // 16-byte aligned for the float4 weight reads

  const int tid = threadIdx.x;
  const int tx = tid & 7, ty = (tid >> 3) & 7, tzg = tid >> 6;
  const int cg = threadIdx.y;
  const int nthreads = blockDim.x * blockDim.y;
  const int ltid = threadIdx.y * blockDim.x + tid;

  const int tiles = a.tn >> 3;
  int bid = blockIdx.x;
  const int bx = bid % tiles; bid /= tiles;
  const int by = bid % tiles; bid /= tiles;
  const int bz = bid % tiles; bid /= tiles;
  const int b = bid;
  const int co_base = blockIdx.y * CB;

  // input coordinates of the brick origin
  const int iz0 = bz * 8 * S - a.pz, iy0 = by * 8 * S - a.py, ix0 = bx * 8 * S - a.px;
  const float* in_b = a.in + (size_t)b * a.in_n * a.in_n * a.in_n * a.in_cs + a.in_co;

  float acc[4][CT];
#pragma unroll
  for (int j = 0; j < 4; ++j)
#pragma unroll
    for (int c = 0; c < CT; ++c) acc[j][c] = 0.f;

  const int brick_vox = EZ * a.ey * a.ex;
  const int kyx = a.ky * a.kx;

  for (int c0 = 0; c0 < a.cin; c0 += a.cc) {
    const int ccn = min(a.cc, a.cin - c0);
    __syncthreads();
    // ---- stage the input brick: global -> shared channel-planar ----
    if (a.in_pm) {
      // PM split-bf16 input: groups of 4 channels (half a 16-byte cell), value = hi + lo
      const size_t pe = (size_t)a.in_n * a.in_n * a.in_n * 8;
      const __nv_bfloat16* pb = a.in_pm + (size_t)b * (2 * (a.cin / 8)) * pe;
      const int g4n = a.cc >> 2;
      for (int i = ltid; i < brick_vox * g4n; i += nthreads) {
        const int g = i % g4n;
        int e = i / g4n;
        const int x = e % a.ex; e /= a.ex;
        const int y = e % a.ey; const int z = e / a.ey;
        const int gz = iz0 + z, gy = iy0 + y, gx = ix0 + x;
        const int c = c0 + 4 * g;
        float v[4] = {0.f, 0.f, 0.f, 0.f};
        if (c < a.cin && (unsigned)gz < (unsigned)a.in_n && (unsigned)gy < (unsigned)a.in_n && (unsigned)gx < (unsigned)a.in_n) {
          const size_t vox = ((size_t)(gz * a.in_n + gy) * a.in_n + gx) * 8 + (c & 7);
          load_half_cell_sum(pb + (size_t)(2 * (c >> 3)) * pe + vox, pb + (size_t)(2 * (c >> 3) + 1) * pe + vox, v);
        }
#pragma unroll
        for (int k = 0; k < 4; ++k) s_in[(4 * g + k) * a.plane + (z * a.ey + y) * a.exp_ + x] = v[k];
      }
    } else
    for (int i = ltid; i < brick_vox * a.cc; i += nthreads) {
      const int c = i % a.cc;
      int e = i / a.cc;
      const int x = e % a.ex; e /= a.ex;
      const int y = e % a.ey; const int z = e / a.ey;
      const int gz = iz0 + z, gy = iy0 + y, gx = ix0 + x;
      float v = 0.f;
      if (c < ccn && (unsigned)gz < (unsigned)a.in_n && (unsigned)gy < (unsigned)a.in_n && (unsigned)gx < (unsigned)a.in_n)
        v = __ldg(in_b + ((size_t)(gz * a.in_n + gy) * a.in_n + gx) * a.in_cs + c0 + c);
      s_in[c * a.plane + (z * a.ey + y) * a.exp_ + x] = v;
    }
    // ---- stage the weight slab: global [KY][KX][Cin][KZ][Cout] -> shared [KY*KX][CC][KZ][CB] ----
    for (int i = ltid; i < kyx * a.cc * KZ * CB; i += nthreads) {
      const int co = i % CB;
      int e = i / CB;
      const int kz = e % KZ; e /= KZ;
      const int c = e % a.cc; const int t = e / a.cc;
      float v = 0.f;
      if (c < ccn && co_base + co < a.cout)
        v = __ldg(a.w + (((size_t)t * a.cin + c0 + c) * KZ + kz) * a.cout + co_base + co);
      s_w[i] = v;
    }
    __syncthreads();

    // ---- accumulate ----
    for (int t = 0; t < kyx; ++t) {
      const int ky = t / a.kx, kx = t - ky * a.kx;
      const float* ip = s_in + ((tzg * 4 * S) * a.ey + ty * S + ky) * a.exp_ + tx * S + kx;
      const float* wp = s_w + (size_t)t * a.cc * KZ * CB + cg * CT;
      for (int c = 0; c < ccn; ++c) {
        float win[WIN];
#pragma unroll
        for (int i = 0; i < WIN; ++i) win[i] = ip[c * a.plane + i * a.ey * a.exp_];
        const float* wc = wp + c * KZ * CB;
#pragma unroll
        for (int kz = 0; kz < KZ; ++kz) {
          float wv[CT];
          if constexpr (CT % 4 == 0) {
#pragma unroll
            for (int q = 0; q < CT / 4; ++q) {
              const float4 f = *reinterpret_cast<const float4*>(wc + kz * CB + 4 * q);
              wv[4 * q] = f.x; wv[4 * q + 1] = f.y; wv[4 * q + 2] = f.z; wv[4 * q + 3] = f.w;
            }
          } else {
#pragma unroll
            for (int q = 0; q < CT; ++q) wv[q] = wc[kz * CB + q];
          }
#pragma unroll
          for (int j = 0; j < 4; ++j)
#pragma unroll
            for (int q = 0; q < CT; ++q) acc[j][q] = fmaf(win[j * S + kz], wv[q], acc[j][q]);
        }
      }
    }
  }

  // ---- epilogue ----
  const int t_y = by * 8 + ty, t_x = bx * 8 + tx;
  const int o_y = t_y * a.ostride + a.oy, o_x = t_x * a.ostride + a.ox;
#pragma unroll
  for (int j = 0; j < 4; ++j) {
    const int t_z = bz * 8 + tzg * 4 + j;
    const int o_z = t_z * a.ostride + a.oz;
    const size_t vox = (((size_t)b * a.out_n + o_z) * a.out_n + o_y) * a.out_n + o_x;
    if constexpr (CT == 8) {
      if (a.out_pm) {
        const int co0 = co_base + cg * CT;
        if (co0 < a.cout) {
          float v[8];
#pragma unroll
          for (int q = 0; q < 8; ++q) {
            float t = acc[j][q];
            if (a.bias) t += __ldg(a.bias + co0 + q);
            if (a.flags & EPI_RELU) t = fmaxf(t, 0.f);
            v[q] = t;
          }
          const size_t pe = (size_t)a.out_n * a.out_n * a.out_n * 8;
          const size_t lv = (((size_t)o_z * a.out_n + o_y) * a.out_n + o_x) * 8;
          __nv_bfloat16* ob = a.out_pm + ((size_t)b * (2 * (a.cout / 8)) + 2 * (co0 >> 3)) * pe + lv;
          split_store(ob, ob + pe, v);
        }
        continue;
      }
    }
    if (a.class_mode) {
      // the CT = 8 accumulators are the 8 output-parity classes of a single-channel transposed conv
      if constexpr (CT == 8) {
        const float bz0 = a.bias ? __ldg(a.bias) : 0.f;
#pragma unroll
        for (int q = 0; q < 8; ++q) {
          const int oz = 2 * t_z + (((q >> 2) & 1) ? a.cls_o0b : a.cls_o0a), oy = 2 * t_y + (((q >> 1) & 1) ? a.cls_o0b : a.cls_o0a),
                    ox = 2 * t_x + ((q & 1) ? a.cls_o0b : a.cls_o0a);
          float v = acc[j][q] + bz0;
          if (a.flags & EPI_RELU) v = fmaxf(v, 0.f);
          if (a.flags & EPI_ABS) v = fabsf(v);
          if (a.flags & EPI_FLOOR) v = fmaxf(v, a.floor_v);
          a.out[((((size_t)b * a.out_n + oz) * a.out_n + oy) * a.out_n + ox) * a.out_cs + a.out_co] = v;
        }
      }
      continue;
    }
    float* op = a.out + vox * a.out_cs + a.out_co;
    const float* rp = a.res ? a.res + vox * a.res_cs + a.res_co : nullptr;
#pragma unroll
    for (int q = 0; q < CT; ++q) {
      const int co = co_base + cg * CT + q;
      if (co < a.cout) {
        float v = acc[j][q];
        if (a.bias) v += __ldg(a.bias + co);
        if (a.flags & EPI_RELU) v = fmaxf(v, 0.f);
        if (rp) v = fmaxf(v + __ldg(rp + co), 0.f);
        if (a.flags & EPI_ABS) v = fabsf(v);
        if (a.flags & EPI_FLOOR) v = fmaxf(v, a.floor_v);
        op[co] = v;
      }
    }
  }
}

template <int KZ, int S>
static cudaError_t launch_kzs(const FfmaArgs& a, int B, cudaStream_t s) {
  int ct = a.cout >= 8 ? 8 : (a.cout >= 4 ? 4 : 1);
  int groups = (a.cout + ct - 1) / ct;
  int G = groups < 4 ? groups : 4;
  int gy = (groups + G - 1) / G;
  const int CB = G * ct;
  FfmaArgs b = a;
  constexpr int EZ = 7 * S + KZ;
  b.ey = 7 * S + a.ky; b.ex = 7 * S + a.kx; b.exp_ = b.ex;
  // choose the channel chunk so that brick + weights fit a ~96 KB budget (PM inputs: multiples of 4)
  int cc = a.cin < 16 ? a.cin : 16;
  const int cc_min = a.in_pm ? 4 : 1;
  size_t smem = 0;
  for (;; cc = (cc + 1) / 2) {
    int plane = EZ * b.ey * b.exp_;
    int want = cc >= 2 ? 32 / (cc > 32 ? 32 : cc) : 0;       // plane % 32 == 32/cc -> conflict-free staging
    if (cc >= 2) { while (plane % 32 != want % 32) ++plane; }
    b.plane = plane; b.cc = cc;
    smem = ((((size_t)cc * plane + 3) & ~(size_t)3) + (size_t)a.ky * a.kx * cc * KZ * CB) * sizeof(float);
    if (smem <= 96 * 1024 || cc <= cc_min) break;
  }
  if (smem > 200 * 1024) return cudaErrorInvalidConfiguration;
  const int tiles = a.tn / 8;
  dim3 grid((unsigned)((size_t)tiles * tiles * tiles * B), gy, 1), block(128, G, 1);
  cudaError_t e = cudaSuccess;
#define PCGC_LAUNCH(CTV)                                                                              \
  do {                                                                                                \
    prefer_shared_carveout(conv_ffma_kernel<KZ, S, CTV>);                                                   \
    e = cudaFuncSetAttribute(conv_ffma_kernel<KZ, S, CTV>, cudaFuncAttributeMaxDynamicSharedMemorySize, \
                             (int)smem);                                                              \
    if (e == cudaSuccess) { conv_ffma_kernel<KZ, S, CTV><<<grid, block, smem, s>>>(b); e = cudaGetLastError(); } \
  } while (0)
  if (ct == 8) PCGC_LAUNCH(8); else if (ct == 4) PCGC_LAUNCH(4); else PCGC_LAUNCH(1);
#undef PCGC_LAUNCH
  return e;
}

cudaError_t launch_conv_ffma(const ConvCall& c, cudaStream_t s, int64_t* launches) {
  FfmaArgs a;
  a.in = c.in; a.out = c.out; a.w = c.d.w; a.bias = c.bias; a.res = c.res;
  a.in_n = c.in_n; a.in_cs = c.in_cs; a.in_co = c.in_co;
  a.out_n = c.out_n; a.out_cs = c.out_cs; a.out_co = c.out_co;
  a.res_cs = c.res_cs; a.res_co = c.res_co;
  a.tn = c.tn; a.ky = c.d.ky; a.kx = c.d.kx;
  a.pz = c.d.pz; a.py = c.d.py; a.px = c.d.px;
  a.ostride = c.d.ostride; a.oz = c.d.oz; a.oy = c.d.oy; a.ox = c.d.ox;
  a.cin = c.d.cin; a.cout = c.d.cout;
  a.flags = c.flags; a.floor_v = c.floor_v;
  a.class_mode = c.d.class_mode; a.cls_o0a = c.d.cls_o0[0]; a.cls_o0b = c.d.cls_o0[1];
  if (a.class_mode && (c.out_pm || c.res || c.d.cout != 8)) return cudaErrorInvalidValue;
  a.in_pm = (const __nv_bfloat16*)c.in_pm; a.out_pm = (__nv_bfloat16*)c.out_pm;
  if (a.in_pm && (c.d.cin % 8 != 0)) return cudaErrorInvalidValue;
  if (a.out_pm && (c.d.cout % 8 != 0 || c.res)) return cudaErrorInvalidValue;
  a.cc = 0; a.plane = 0; a.ey = a.ex = a.exp_ = 0;
  if (c.tn % 8 != 0 || c.B <= 0) return cudaErrorInvalidValue;
  if (launches) ++*launches;
  const int key = c.d.kz * 10 + c.d.stride;
  switch (key) {
    case 11: return launch_kzs<1, 1>(a, c.B, s);
    case 21: return launch_kzs<2, 1>(a, c.B, s);
    case 31: return launch_kzs<3, 1>(a, c.B, s);
    case 41: return launch_kzs<4, 1>(a, c.B, s);
    case 51: return launch_kzs<5, 1>(a, c.B, s);
    case 32: return launch_kzs<3, 2>(a, c.B, s);
    case 52: return launch_kzs<5, 2>(a, c.B, s);
    case 92: return launch_kzs<9, 2>(a, c.B, s);
    default: return cudaErrorInvalidValue;
  }
}

// ---- conv_in of the voxception analysis transform (model_voxception.py:83-88): 1 -> 16 channels on the 64^3 occupancy grid
// Reads the cube in its input dtype (uint8 / float32 / float64: no separate conversion pass), applies the 3x3x3 conv +
// bias + ReLU in FP32 and writes the PM split-bf16 tensor the tcgen05 engine consumes.  CTA tile 4(z) x 8(y) x 64(x);
// a thread owns two voxels (y and y+4) so every broadcast weight load feeds 8 FMAs; lanes run along x (conflict-free).
// The 27x16 weights + bias travel as a by-value kernel parameter: they sit in the constant bank and every FFMA takes its
// weight as a constant operand (no shared-memory weight loads; the first version was LDS.128-bound at 9 TFLOP/s).
// r02 last session: all-zero taps are skipped per warp (see the loop).
// Far-field voxels (ff_mask): a voxel with no occupied voxel within radius 1 is the empty cube's; it is stored only where the slot's
// previous cube left it different (ff_prev), and a CTA none of whose voxels is stored returns at once.
struct ConvInParams { float w[27 * 16]; float b[16]; };

template <typename T>
__global__ void __launch_bounds__(256) conv_in_pm_kernel(const T* __restrict__ in, const __grid_constant__ ConvInParams prm,
                                                         __nv_bfloat16* __restrict__ out, const uint8_t* __restrict__ ff_mask,
                                                         const uint8_t* __restrict__ ff_prev) {
  constexpr int N = 64, TZ = 4, TY = 8;
  __shared__ float s_in[TZ + 2][TY + 2][N + 2];
  const int tid = threadIdx.x;
  int bid = blockIdx.x;
  const int by = bid % (N / TY); bid /= (N / TY);
  const int bz = bid % (N / TZ); bid /= (N / TZ);
  const int b = bid;
  // mask byte of (b, z, 32-line y tile): bit = 8-voxel x tile; the CTA's 8 lines lie in one y tile
  const size_t m0 = ((size_t)b * N + bz * TZ) * 2 + (by * TY) / 32;
  if (ff_mask) {
    uint32_t any = 0;
#pragma unroll
    for (int zi = 0; zi < TZ; ++zi) any |= ff_mask[m0 + 2 * zi] | ff_prev[m0 + 2 * zi];
    if (!any) return;                                              // CTA-uniform, before the barrier
  }
  const T* ib = in + (size_t)b * N * N * N;
  for (int i = tid; i < (TZ + 2) * (TY + 2) * (N + 2); i += 256) {
    const int x = i % (N + 2), y = (i / (N + 2)) % (TY + 2), z = i / ((N + 2) * (TY + 2));
    const int gz = bz * TZ + z - 1, gy = by * TY + y - 1, gx = x - 1;
    float v = 0.f;
    if ((unsigned)gz < (unsigned)N && (unsigned)gy < (unsigned)N && (unsigned)gx < (unsigned)N) v = (float)ib[((size_t)gz * N + gy) * N + gx];
    s_in[z][y][x] = v;
  }
  __syncthreads();
  const int x = tid & 63, z = tid >> 6;
  const size_t pe = (size_t)N * N * N * 8;
  __nv_bfloat16* ob = out + (size_t)b * 4 * pe;
  const bool store = !ff_mask || (((ff_mask[m0 + 2 * z] | ff_prev[m0 + 2 * z]) >> (x >> 3)) & 1u);
  if (!__any_sync(0xFFFFFFFFu, store)) return;                    // warp-uniform; no barrier follows
#pragma unroll 1
  for (int yy = 0; yy < 4; ++yy) {
    float a0[16], a1[16];
#pragma unroll
    for (int c = 0; c < 16; ++c) { a0[c] = prm.b[c]; a1[c] = prm.b[c]; }
#pragma unroll
    for (int t = 0; t < 27; ++t) {
      const int kz = t / 9, ky = (t / 3) % 3, kx = t % 3;
      const float v0 = s_in[z + kz][yy + ky][x + kx], v1 = s_in[z + kz][yy + 4 + ky][x + kx];
      // occupancy cubes are ~98 % zeros: a tap none of the warp's 64 voxels sees occupied adds exactly nothing (0 * w + a = a), skip its
      // 32 FMAs (warp-uniform branch; the result is bit-identical)
      if (!__any_sync(0xffffffffu, v0 != 0.f || v1 != 0.f)) continue;
#pragma unroll
      for (int c = 0; c < 16; ++c) {
        a0[c] = fmaf(v0, prm.w[t * 16 + c], a0[c]);
        a1[c] = fmaf(v1, prm.w[t * 16 + c], a1[c]);
      }
    }
#pragma unroll
    for (int c = 0; c < 16; ++c) { a0[c] = fmaxf(a0[c], 0.f); a1[c] = fmaxf(a1[c], 0.f); }
    if (!store) continue;
    const int gz = bz * TZ + z, gy0 = by * TY + yy, gy1 = gy0 + 4;
    __nv_bfloat16* o0 = ob + (((size_t)gz * N + gy0) * N + x) * 8;
    __nv_bfloat16* o1 = ob + (((size_t)gz * N + gy1) * N + x) * 8;
    split_store(o0, o0 + pe, a0); split_store(o0 + 2 * pe, o0 + 3 * pe, a0 + 8);
    split_store(o1, o1 + pe, a1); split_store(o1 + 2 * pe, o1 + 3 * pe, a1 + 8);
  }
}

// w: HOST float [27][16] tap-major (the Keras [3,3,3,1,16] kernel as is), bias HOST [16] or null.
cudaError_t launch_conv_in_pm(const void* cubes, int dtype, const float* w_host, const float* bias_host, void* out_pm, int B,
                              const uint8_t* ff_mask, const uint8_t* ff_prev, cudaStream_t s, int64_t* launches) {
  if ((ff_mask != nullptr) != (ff_prev != nullptr) || (ff_mask && dtype != PCGC_DTYPE_U8)) return cudaErrorInvalidValue;
  ConvInParams prm;
  for (int i = 0; i < 27 * 16; ++i) prm.w[i] = w_host[i];
  for (int i = 0; i < 16; ++i) prm.b[i] = bias_host ? bias_host[i] : 0.f;
  const int grid = (64 / 8) * (64 / 4) * B;
  if (launches) ++*launches;
  switch (dtype) {
    case PCGC_DTYPE_U8: PCGC_CARVEOUT_ONCE(conv_in_pm_kernel<uint8_t>); conv_in_pm_kernel<uint8_t><<<grid, 256, 0, s>>>((const uint8_t*)cubes, prm, (__nv_bfloat16*)out_pm, ff_mask, ff_prev); break;
    case PCGC_DTYPE_F32: conv_in_pm_kernel<float><<<grid, 256, 0, s>>>((const float*)cubes, prm, (__nv_bfloat16*)out_pm, nullptr, nullptr); break;
    case PCGC_DTYPE_F64: conv_in_pm_kernel<double><<<grid, 256, 0, s>>>((const double*)cubes, prm, (__nv_bfloat16*)out_pm, nullptr, nullptr); break;
    default: return cudaErrorInvalidValue;
  }
  return cudaGetLastError();
}

// ---- input conversion: occupancy cubes of any host dtype -> float32 ---------------------------
template <typename T>
__global__ void to_f32_kernel(const T* __restrict__ in, float* __restrict__ out, int64_t n) {
  int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  const int64_t stride = (int64_t)gridDim.x * blockDim.x;
  for (; i < n; i += stride) out[i] = (float)in[i];
}

cudaError_t launch_u8_to_f32(const void* in, int dtype, float* out, int64_t n, cudaStream_t s, int64_t* launches) {
  const int threads = 256;
  int64_t blocks = (n + threads - 1) / threads;
  if (blocks > 148 * 32) blocks = 148 * 32;
  if (launches) ++*launches;
  switch (dtype) {
    case PCGC_DTYPE_U8: to_f32_kernel<uint8_t><<<(unsigned)blocks, threads, 0, s>>>((const uint8_t*)in, out, n); break;
    case PCGC_DTYPE_F32: to_f32_kernel<float><<<(unsigned)blocks, threads, 0, s>>>((const float*)in, out, n); break;
    case PCGC_DTYPE_F64: to_f32_kernel<double><<<(unsigned)blocks, threads, 0, s>>>((const double*)in, out, n); break;
    default: return cudaErrorInvalidValue;
  }
  return cudaGetLastError();
}

}  // namespace pcgc
