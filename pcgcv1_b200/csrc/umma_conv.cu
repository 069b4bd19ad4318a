// tcgen05 / TMEM / TMA implicit-GEMM engine for the 3x3x3 stride-1 SAME convolutions -- the Voxception
// blocks and the convs around them (models/model_voxception.py:21-68,83-88,118-122,153-158,188-192),
// ~87 % of the path's MACs (SURVEY.md appendix A).
//
// GEMM view per CTA: M = 128 output voxels (8 along x  x 16 along y, one z slice), N = output channels,
// K = 27 taps x Cin.  Nothing is im2col'ed:
//   * activations live in HBM in the "PM" split-bf16 plane-major format (umma_conv.cuh).  ONE 5-D TMA box
//     {10 x-cells, 18 y, zt+2 z, 4 planes} with out-of-bounds zero fill (= TF SAME padding) lands the
//     haloed brick of 16 input channels (hi and lo planes) in shared memory, already in the UMMA
//     no-swizzle K-major core-matrix layout: 8 consecutive x voxels x 8 channels = 128 contiguous bytes.
//   * every tap is then just a different START ADDRESS of the A descriptor into the same brick
//     (kx: +16 B, ky: +160 B, kz: +2880 B; SBO = 160 B steps the 16 y-lines of the M tile, LBO steps the
//     two 8-channel halves of K = 16), so a brick is read from L2 once and re-used by all 27 taps.
//   * FP32-grade accuracy from BF16 tensor cores: x = x_hi + x_lo, w = w_hi + w_lo and
//     D = x_hi*[w_hi | w_lo] + x_lo*w_hi: two tcgen05.mma per tap (N = 2*NP, then N = NP into the same
//     TMEM columns), FP32 accumulation in TMEM, the dropped x_lo*w_lo term is ~2^-18 relative.
//     This is what keeps >= 99.9 % of the quantised latents bit-identical to the FP32 reference.
//   * zt z-slices keep zt accumulators (zt * 2NP columns) in TMEM; one elected thread issues all MMAs.
//   * the epilogue reads TMEM (tcgen05.ld 32x32b), adds hi/lo halves + bias, applies ReLU / the whole
//     Voxception tail (1x1x1 conv2_3, concat, residual add, ReLU: model_voxception.py:62-67) and writes
//     PM (or float32 NDHWC for external tensors).
// Deterministic: fixed K order, no atomics, no split-K; the tile shape never depends on the batch.
//
// Three kernels share the operand formats, the epilogues and the weight packing below; launch_conv_umma_pm picks per layer shape:
//   conv_umma_kernel         tile kernel (this description): persistent CTAs, 2-3 per SM, one haloed brick per tile.  Serves the
//                            multi-chunk layers (Cin >= 32 at 16^3), the stride-2 / transposed forms and K_b16.
//   conv_umma_stream_kernel  z-streaming: one CTA per SM walks a column of z slices through a ring of shared-memory slots, with
//                            the TMA producer, three MMA issuers and the epilogue split over warps.  Serves K_b32, deconv_in.
//   conv_umma_zband_kernel   z-banded streaming: input-slice stationary, the three kz taps are column blocks of one MMA, so an
//                            A tile is fetched once for the three output slices it feeds.  Serves the 16-column layers (K_a16,
//                            K_a32, deconv_out), which were bound by exactly that fetch.
// PCGC_UMMA_STREAM / PCGC_UMMA_ZBAND select among them for experiments; tests/test_gpu_umma_modes.py runs every setting.
#include <cuda.h>
#include <stdio.h>
#include <stdlib.h>

#include <algorithm>
#include <map>
#include <mutex>
#include <tuple>
#include <vector>

#include "pm_format.cuh"
#include "umma_conv.cuh"
#include "umma_dev.cuh"

namespace pcgc {

namespace {

constexpr int EXC = 10;                 // brick cells along x (8 + halo)
constexpr int EYC = 18;                 // brick lines along y (16 + halo)
constexpr int CELL = 16;                // bytes per cell (8 bf16)
constexpr int TILE_X = 8, TILE_Y = 16;

struct UmmaArgs {
  int n, zt, ez;
  int cin8;                  // Cin == 8: K = 16 spans two taps
  int kchunks, ppc;          // 16-channel chunks, planes per chunk (4, or 2 when cin8)
  int n_mma;                 // MMA pairs per z-slice per chunk
  int plane_bytes;           // shared-memory bytes of one brick plane
  int a_bytes, b_bytes;      // per-chunk bytes of the A brick / B tiles
  int tmem_cols;
  const __nv_bfloat16* wpacked;
  const float* bias;
  int n_real, flags; float floor_v;
  float* out_f32; int out_cs, out_co;
  float* out2_f32; int split, flags2;      // UEPI_F32: columns >= split go to out2_f32 (stride n_real - split) with flags2
  __nv_bfloat16* out_pm; int out_planes;
  const __nv_bfloat16* res_pm; int res_planes;
  const float* w23; const float* b23; int c4, c2;
  int* err;
  int nsets;                 // TMEM accumulator sets (2: ping-pong between tiles, 1 when the columns do not allow it)
  int batch;                 // cubes in this launch (tiles = per-cube tiles * batch; the grid is persistent)
  int origin;                // brick origin relative to the tile: -1 (SAME 3x3x3, transposed) or 0 (stride-2 conv on a space-to-depth input)
  uint32_t tap_mask[16];     // per 16-channel chunk: taps with non-zero weights (others are skipped)
  int out_s2d;               // UEPI_VRN: write the output space-to-depth (grid n/2, 8*C channels) for a following stride-2 conv
  int up_ncls, up_cls0, up_cout;   // UEPI_UP: classes in this launch, first class, channels per class
  int dbg;                   // PCGC_UMMA_DBG bit mask (timing experiments only): 1 skip MMAs, 2 skip the A TMA, 4 skip epilogue
  // far-field tiles of the analysis 64^3 stage: ff_mask[(b*n + z)*ty_n + by] bit bx = 1 when some occupied voxel lies inside the receptive
  // field of that (z, y tile, x tile) of the output layer; ff_prev is the same mask of the cube the output slot held before (the slot
  // holds the empty cube's values wherever that bit is clear), or nullptr when the slot holds nothing known.
  //   tile kernel (UEPI_VRN): a tile whose zt slices are all clear in ff_mask is not computed.  It is COPIED from ff_src, the same
  //     layer's output for the all-zero cube (one cube, same layout as out_pm), unless it is clear in ff_prev too: then nothing is written.
  //   z-banded kernel (UEPI_PM): the segments (ZS slices) clear in both masks are left out of ff_list; every listed segment is computed whole.
  // ff_list = {count, unit indices in the kernel's tile / segment numbering} (launch_ff_list): the tiles or segments the persistent CTAs
  // share; nullptr: all of them.  Bit-identical to computing every tile.  ff_mask nullptr: every tile is computed.
  const uint8_t* ff_mask; const uint8_t* ff_prev; const __nv_bfloat16* ff_src;
  const int* ff_list;
  // z-streaming kernel (conv_umma_stream_kernel)
  int ring, zs, nacc;        // input-slice ring slots, output slices per segment, accumulator slots
  int slot_bytes;            // bytes of one ring slot = planes * slice_plane
  int slice_plane;           // bytes of one plane of one z-slice: EY * EXC * CELL
};

// N consecutive accumulator columns of this lane in ONE tcgen05.ld (one TMEM round trip instead of N/16).
template <int N>
__device__ __forceinline__ void tmem_ld(uint32_t taddr, float* v) {
  static_assert(N == 32 || N == 64, "supported widths");
  uint32_t r[N];
  if (N == 32) {
    asm volatile(
        "tcgen05.ld.sync.aligned.32x32b.x32.b32 {%0,%1,%2,%3,%4,%5,%6,%7,%8,%9,%10,%11,%12,%13,%14,%15,%16,%17,%18,%19,%20,%21,%22,%23,%24,%25,%26,%27,%28,%29,%30,%31}, [%32];"
        : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]), "=r"(r[8]), "=r"(r[9]),
          "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15]), "=r"(r[16]), "=r"(r[17]), "=r"(r[18]), "=r"(r[19]),
          "=r"(r[20]), "=r"(r[21]), "=r"(r[22]), "=r"(r[23]), "=r"(r[24]), "=r"(r[25]), "=r"(r[26]), "=r"(r[27]), "=r"(r[28]), "=r"(r[29]),
          "=r"(r[30]), "=r"(r[31])
        : "r"(taddr));
  } else {
    asm volatile(
        "tcgen05.ld.sync.aligned.32x32b.x64.b32 {%0,%1,%2,%3,%4,%5,%6,%7,%8,%9,%10,%11,%12,%13,%14,%15,%16,%17,%18,%19,%20,%21,%22,%23,%24,%25,%26,%27,%28,%29,%30,%31,"
        "%32,%33,%34,%35,%36,%37,%38,%39,%40,%41,%42,%43,%44,%45,%46,%47,%48,%49,%50,%51,%52,%53,%54,%55,%56,%57,%58,%59,%60,%61,%62,%63}, [%64];"
        : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]), "=r"(r[8]), "=r"(r[9]),
          "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15]), "=r"(r[16]), "=r"(r[17]), "=r"(r[18]), "=r"(r[19]),
          "=r"(r[20]), "=r"(r[21]), "=r"(r[22]), "=r"(r[23]), "=r"(r[24]), "=r"(r[25]), "=r"(r[26]), "=r"(r[27]), "=r"(r[28]), "=r"(r[29]),
          "=r"(r[30]), "=r"(r[31]), "=r"(r[32]), "=r"(r[33]), "=r"(r[34]), "=r"(r[35]), "=r"(r[36]), "=r"(r[37]), "=r"(r[38]), "=r"(r[39]),
          "=r"(r[40]), "=r"(r[41]), "=r"(r[42]), "=r"(r[43]), "=r"(r[44]), "=r"(r[45]), "=r"(r[46]), "=r"(r[47]), "=r"(r[48]), "=r"(r[49]),
          "=r"(r[50]), "=r"(r[51]), "=r"(r[52]), "=r"(r[53]), "=r"(r[54]), "=r"(r[55]), "=r"(r[56]), "=r"(r[57]), "=r"(r[58]), "=r"(r[59]),
          "=r"(r[60]), "=r"(r[61]), "=r"(r[62]), "=r"(r[63])
        : "r"(taddr));
  }
  asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory");
#pragma unroll
  for (int i = 0; i < N; ++i) v[i] = __uint_as_float(r[i]);
}

enum TapMode : int { TAPS_27 = 0, TAPS_27_PAIRED = 1, TAPS_8 = 2 };

// Brick y extent.  WT > 1 is the Y-BANDED form: M row (g, x) stands for WT consecutive output lines y = WT*g + j, the
// output columns are (j, channel) and the A tiles are indexed by the input line offset d in [0, WT+2) instead of ky
// (weights W[kz][d - j][kx], zero outside the band).  The same brick then needs 9*(WT+2) A tiles for 128*WT outputs
// instead of 27*WT -- and the kernels are bound by exactly that: every MMA waits for its 4 KiB A tile from shared
// memory (ncu r01: sm__pipe_tc_cycles_active 95 %, tensor math 27 %).
__host__ __device__ constexpr int brick_ey(int wt) { return 16 * wt + 2; }

// Issues every MMA of one z-slice for one 16-channel chunk.  Fully unrolled: tile offsets are compile-time
// constants, so each MMA costs two 64-bit adds on the descriptors -- the single issuing thread must not be the
// bottleneck (the first version recomputed descriptors with integer divisions and ran at ~125 cycles per MMA).
template <int NP, int TAPS, int WT>
__device__ __forceinline__ void issue_slice(uint32_t d, uint64_t a_hi, uint64_t a_lo, uint64_t bdesc, bool first, uint32_t mask) {
  constexpr uint32_t idesc_full = make_idesc(128, 2 * NP), idesc_half = make_idesc(128, NP);
  constexpr int EY = brick_ey(WT);
  constexpr int NT = 9 * (WT + 2);                               // A tiles (kz, d, kx) of the 3x3x3 modes
  constexpr int NM = TAPS == TAPS_27 ? NT : (TAPS == TAPS_27_PAIRED ? (NT + 1) / 2 : 8);
  constexpr uint64_t b_step = (uint64_t)((2 * NP * 32) >> 4);
  auto tile_off = [](int t) { return ((((t / (3 * (WT + 2))) * EY + (t / 3) % (WT + 2)) * EXC + t % 3) * CELL); };
#pragma unroll
  for (int m = 0; m < NM; ++m) {
    uint64_t add;
    if (TAPS == TAPS_27) {
      add = (uint64_t)(tile_off(m) >> 4);
    } else if (TAPS == TAPS_8) {
      const int kz = m >> 2, ky = (m >> 1) & 1, kx = m & 1;      // brick index 0 = input t-1, 1 = input t
      add = (uint64_t)((((kz * EY + ky) * EXC + kx) * CELL) >> 4);
    } else {
      // Cin == 8: K = 16 spans two tiles (LBO = their address difference).  Odd tile count: tile 0 goes alone
      // (its partner carries zero weights).
      const int ta = (NT & 1) ? (m == 0 ? 0 : 2 * m - 1) : 2 * m, tb = (NT & 1) ? (m == 0 ? 1 : 2 * m) : 2 * m + 1;
      const int oa = tile_off(ta), ob = tile_off(tb);
      add = (uint64_t)(oa >> 4) | ((uint64_t)((ob - oa) >> 4) << 16);      // start offset | LBO (second tile)
    }
    if (TAPS == TAPS_8 && !((mask >> m) & 1u) && !(first && m == 0)) continue;   // all-zero weight tile (the first MMA still initialises D)
    const uint64_t bd = bdesc + (uint64_t)m * b_step;
    umma_f16(d, a_hi + add, bd, idesc_full, (first && m == 0) ? 0u : 1u);   // x_hi * [w_hi | w_lo]
    umma_f16(d, a_lo + add, bd, idesc_half, 1u);                             // x_lo * w_hi
  }
}

constexpr int EPI_WARPS = 8;                       // warps 0..7: epilogue; warp 8: TMA producer + MMA issuer
constexpr int UMMA_THREADS = 32 * (EPI_WARPS + 1);
constexpr int MAX_ZT = 8;

// Epilogue of ONE output voxel whose NPJ accumulator columns (+bias) are in v[].
// Residual cells (8 channels each, hi and lo plane) of one voxel of the Voxception block input.
template <int RC>
__device__ __forceinline__ void vrn_load_residual(const UmmaArgs& a, int b, int vz, int vy, int vx, size_t plane_elems, uint4* rhi, uint4* rlo) {
  const size_t vox = ((size_t)vz * a.n + vy) * a.n + vx;
  const __nv_bfloat16* rb = a.res_pm + (size_t)b * a.res_planes * plane_elems + vox * 8;
#pragma unroll
  for (int c8 = 0; c8 < RC; ++c8) {
    rhi[c8] = __ldg(reinterpret_cast<const uint4*>(rb + (size_t)(2 * c8) * plane_elems));
    rlo[c8] = __ldg(reinterpret_cast<const uint4*>(rb + (size_t)(2 * c8 + 1) * plane_elems));
  }
}
template <int NPJ> struct VrnRc { static constexpr int value = NPJ == 16 ? 2 : (NPJ == 24 || NPJ == 32 ? 4 : 8); };

template <int NPJ, int EPI>
__device__ __forceinline__ void epilogue_voxel(const UmmaArgs& a, float* v, const float* s_w23, int b, int vz, int vy, int vx,
                                               size_t plane_elems, const uint4* pre_hi = nullptr, const uint4* pre_lo = nullptr) {
  const size_t vox = ((size_t)vz * a.n + vy) * a.n + vx;
  if (EPI == UEPI_F32) {
    const size_t gv = (size_t)b * a.n * a.n * a.n + vox;
    float* op = a.out_f32 + gv * a.out_cs + a.out_co;
    float* op2 = a.out2_f32 ? a.out2_f32 + gv * (a.n_real - a.split) : nullptr;
#pragma unroll
    for (int i = 0; i < NPJ; ++i) {
      if (i < a.n_real) {
        float t = v[i];
        const int fl = i < a.split ? a.flags : a.flags2;
        if (fl & EPI_RELU) t = fmaxf(t, 0.f);
        if (fl & EPI_ABS) t = fabsf(t);
        if (fl & EPI_FLOOR) t = fmaxf(t, a.floor_v);
        if (i < a.split) op[i] = t; else op2[i - a.split] = t;
      }
    }
  } else if (EPI == UEPI_PM) {
    __nv_bfloat16* ob = a.out_pm + (size_t)b * a.out_planes * plane_elems + vox * 8;
#pragma unroll
    for (int c8 = 0; c8 < NPJ / 8; ++c8) {
      if (c8 * 8 < a.n_real) {
        float t[8];
#pragma unroll
        for (int i = 0; i < 8; ++i) t[i] = (a.flags & EPI_RELU) ? fmaxf(v[c8 * 8 + i], 0.f) : v[c8 * 8 + i];
        split_store(ob + (size_t)(2 * c8) * plane_elems, ob + (size_t)(2 * c8 + 1) * plane_elems, t);
      }
    }
  } else if (EPI == UEPI_VRN) {
    // Voxception tail.  columns [0,c2) = conv1_2, [c2,c2+c4) = conv2_2 (both ReLU'd), then conv2_3 (1x1x1),
    // concat, residual add and ReLU (model_voxception.py:62-67).
    constexpr int RC = NPJ == 16 ? 2 : (NPJ == 24 || NPJ == 32 ? 4 : 8);       // residual cells (8 channels each)
    const int c2 = a.c2, c4 = a.c4;
    const __nv_bfloat16* rb = a.res_pm + (size_t)b * a.res_planes * plane_elems + vox * 8;
    // normal: plane stride = n^3 cells.  space-to-depth: voxel (z,y,x) channel c -> voxel (z/2,y/2,x/2) of the n/2 grid,
    // channel p*C + c with p = parity(z,y,x); the tensor then has 8x the planes of 1/8 the size.
    size_t ops = plane_elems;                         // elements between consecutive output planes
    __nv_bfloat16* ob = a.out_pm + (size_t)b * a.out_planes * plane_elems + vox * 8;
    if (a.out_s2d) {
      const int h = a.n >> 1;
      ops = plane_elems >> 3;
      const int par = ((vz & 1) << 2) | ((vy & 1) << 1) | (vx & 1);
      ob = a.out_pm + ((size_t)b * a.out_planes * 8 + (size_t)par * a.out_planes) * ops + ((((size_t)(vz >> 1) * h + (vy >> 1)) * h + (vx >> 1)) * 8);
    }
    // all residual cells first (independent loads in flight together), then the math, then the stores
    uint4 rhi[RC], rlo[RC];
#pragma unroll
    for (int c8 = 0; c8 < RC; ++c8) {
      if (pre_hi) { rhi[c8] = pre_hi[c8]; rlo[c8] = pre_lo[c8]; }                  // fetched before the accumulator wait (stream kernel)
      else {
        rhi[c8] = __ldg(reinterpret_cast<const uint4*>(rb + (size_t)(2 * c8) * plane_elems));
        rlo[c8] = __ldg(reinterpret_cast<const uint4*>(rb + (size_t)(2 * c8 + 1) * plane_elems));
      }
    }
#pragma unroll
    for (int i = 0; i < NPJ; ++i) v[i] = fmaxf(v[i], 0.f);
#pragma unroll
    for (int c8 = 0; c8 < RC / 2; ++c8) {            // first half of the output channels: relu(x + t12)
      float x[8], t[8];
      cell_sum(rhi[c8], rlo[c8], x);
#pragma unroll
      for (int i = 0; i < 8; ++i) t[i] = fmaxf(x[i] + v[c8 * 8 + i], 0.f);
      split_store(ob + (size_t)(2 * c8) * ops, ob + (size_t)(2 * c8 + 1) * ops, t);
    }
#pragma unroll
    for (int j8 = 0; j8 < RC / 2; ++j8) {            // second half: t23 = relu(b23 + t22 . W23), relu(x + t23)
      float t23[8];
      const float4* bp = reinterpret_cast<const float4*>(s_w23 + c4 * c2 + j8 * 8);
      { const float4 b0v = bp[0], b1v = bp[1]; t23[0] = b0v.x; t23[1] = b0v.y; t23[2] = b0v.z; t23[3] = b0v.w; t23[4] = b1v.x; t23[5] = b1v.y; t23[6] = b1v.z; t23[7] = b1v.w; }
#pragma unroll
      for (int q = RC * 4; q < NPJ; ++q) {           // q in [c2, c2 + c4): c2 = RC*4 channels
        if (q < c2 + c4) {
          const float tq = v[q];
          const float4* wr = reinterpret_cast<const float4*>(s_w23 + (q - c2) * c2 + j8 * 8);
          const float4 w0 = wr[0], w1 = wr[1];
          t23[0] = fmaf(tq, w0.x, t23[0]); t23[1] = fmaf(tq, w0.y, t23[1]); t23[2] = fmaf(tq, w0.z, t23[2]); t23[3] = fmaf(tq, w0.w, t23[3]);
          t23[4] = fmaf(tq, w1.x, t23[4]); t23[5] = fmaf(tq, w1.y, t23[5]); t23[6] = fmaf(tq, w1.z, t23[6]); t23[7] = fmaf(tq, w1.w, t23[7]);
        }
      }
      float x[8], t[8];
      const int c8 = RC / 2 + j8;
      cell_sum(rhi[c8], rlo[c8], x);
#pragma unroll
      for (int i = 0; i < 8; ++i) t[i] = fmaxf(x[i] + fmaxf(t23[i], 0.f), 0.f);
      split_store(ob + (size_t)(2 * c8) * ops, ob + (size_t)(2 * c8 + 1) * ops, t);
    }
  }
}

// Far-field tiles: is tile (b, by, bx, z0 .. z0 + zt) free of occupied voxels inside its receptive field?  Both roles of the kernel
// evaluate this on the same read-only mask, so they agree on which tiles exist for the barrier protocol.
// (__noinline__, scalar arguments: inlined into the single-thread producer branch this loop crashes nvcc 12.9's optimiser.)
__device__ __noinline__ bool ff_tile_clear(const uint8_t* mask, int n, int zt, int b, int by, int bx, int z0, int ty_n) {
  const uint8_t* m = mask + ((size_t)b * n + z0) * ty_n + by;
  uint32_t need = 0;
  for (int zi = 0; zi < zt; ++zi) need |= m[zi * ty_n];
  return !((need >> bx) & 1u);
}
// WT output voxels (the lines vy .. vy + WT - 1) of a far-field tile: the cells of the empty cube's output at the same positions
// (addressing as epilogue_voxel's).  All loads are issued before the first store: the copy is latency-bound (L2 hits), not bandwidth-bound.
template <int NPJ, int WT>
__device__ __forceinline__ void ff_copy_voxels(const UmmaArgs& a, int b, int vz, int vy, int vx, size_t plane_elems) {
  constexpr int RC = VrnRc<NPJ>::value;
  uint4 t[WT][2 * RC];
  size_t ops = plane_elems, offs[WT], cube = (size_t)a.out_planes * plane_elems;
#pragma unroll
  for (int j = 0; j < WT; ++j) {
    offs[j] = (((size_t)vz * a.n + (vy + j)) * a.n + vx) * 8;
    if (a.out_s2d) {
      const int h = a.n >> 1;
      ops = plane_elems >> 3;
      const int par = ((vz & 1) << 2) | (((vy + j) & 1) << 1) | (vx & 1);
      offs[j] = ((size_t)par * a.out_planes) * ops + ((((size_t)(vz >> 1) * h + ((vy + j) >> 1)) * h + (vx >> 1)) * 8);
      cube = (size_t)a.out_planes * 8 * ops;
    }
  }
#pragma unroll
  for (int j = 0; j < WT; ++j)
#pragma unroll
    for (int p = 0; p < 2 * RC; ++p) t[j][p] = __ldg(reinterpret_cast<const uint4*>(a.ff_src + offs[j] + (size_t)p * ops));
  __nv_bfloat16* dst = a.out_pm + (size_t)b * cube;
#pragma unroll
  for (int j = 0; j < WT; ++j)
#pragma unroll
    for (int p = 0; p < 2 * RC; ++p) *reinterpret_cast<uint4*>(dst + offs[j] + (size_t)p * ops) = t[j][p];
}

// PERSISTENT kernel: a CTA allocates TMEM, initialises its mbarriers, stages bias / 1x1x1 weights and (single-chunk
// layers) the B tiles ONCE, then walks tiles t = blockIdx.x, blockIdx.x + gridDim.x, ...  The r01 timing experiments showed
// that per-CTA set-up + the 27 KB weight reload was ~40 % of the non-persistent kernel (0.23 of 0.58 ms for K_a16).
// Two TMEM accumulator sets alternate between tiles, so the MMAs of tile i+1 overlap the epilogue of tile i; the A brick
// is single-buffered (its TMA is issued as soon as the previous tile's MMAs retire) and 2-3 co-resident CTAs per SM cover
// each other's load latency.
//   barriers: full (TMA landed), mma (all MMAs of the tile/chunk retired: brick reusable), z[set][slice] (accumulator
//   slice final), tmem_free[set] (8 epilogue warps done with the set).
// min-blocks: the unrolled issue loop otherwise inflates the register count (88 vs 55) and costs the third CTA per SM
template <int NP, int EPI, int TAPS, int WT>
__global__ void __launch_bounds__(UMMA_THREADS, (NP <= 16 ? 3 : (NP <= 32 ? 2 : 1))) conv_umma_kernel(const __grid_constant__ CUtensorMap tmap, const UmmaArgs a) {
  extern __shared__ __align__(128) uint8_t smem[];
  uint8_t* s_a = smem;
  uint8_t* s_b = smem + a.a_bytes;
  uint64_t* s_bar = reinterpret_cast<uint64_t*>(s_b + a.b_bytes);          // full, mma, tmem_free[2], z[2][8]
  uint32_t* s_tmem = reinterpret_cast<uint32_t*>(s_bar + 4 + 2 * MAX_ZT);
  float* s_bias = reinterpret_cast<float*>(s_bar + 6 + 2 * MAX_ZT);        // 16-byte aligned (float4 reads)
  float* s_w23 = s_bias + NP;                                              // [c4][c2] then b23[c2] (UEPI_VRN only)
  const uint32_t bar_full = smem_u32(s_bar), bar_mma = smem_u32(s_bar + 1), bar_free = smem_u32(s_bar + 2), bar_z = smem_u32(s_bar + 4);

  constexpr bool CIN8 = TAPS == TAPS_27_PAIRED;
  constexpr int EY = brick_ey(WT);
  constexpr int NPJ = NP / WT;                       // accumulator columns per output line j
  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  const int tx_n = a.n / TILE_X, ty_n = a.n / (TILE_Y * WT), tz_n = a.n / a.zt;
  constexpr bool FFL = EPI == UEPI_VRN && WT == 2;             // the only form launched with a far-field list (K_b16)
  const int total_tiles = (FFL && a.ff_list) ? a.ff_list[0] : tx_n * ty_n * tz_n * a.batch;   // far-field tiles: the listed ones only
  const uint32_t set_cols = (uint32_t)(a.zt * 2 * NP);

  for (int i = tid; i < NP; i += UMMA_THREADS) s_bias[i] = a.bias ? a.bias[i] : 0.f;
  if (EPI == UEPI_VRN) for (int i = tid; i < a.c4 * a.c2 + a.c2; i += UMMA_THREADS) s_w23[i] = i < a.c4 * a.c2 ? a.w23[i] : a.b23[i - a.c4 * a.c2];
  if (tid == 0) {
    mbar_init(bar_full, 1); mbar_init(bar_mma, 1);
    mbar_init(bar_free, EPI_WARPS); mbar_init(bar_free + 8, EPI_WARPS);
    for (int i = 0; i < 2 * MAX_ZT; ++i) mbar_init(bar_z + 8 * i, 1);
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  }
  if (warp == EPI_WARPS) {
    asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(s_tmem)), "r"(a.tmem_cols) : "memory");
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
  }
  asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
  __syncthreads();
  asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
  const uint32_t tmem_base = *s_tmem;

  if (warp == EPI_WARPS) {
    if (elect_one()) {
      // ------------------------------ TMA producer + MMA issuer (one thread) ------------------------------
      const uint32_t brick = smem_u32(s_a), bsm = smem_u32(s_b);
      const uint32_t PL = (uint32_t)a.plane_bytes;
      const uint32_t b_lbo = 2 * NP * 16;
      const uint64_t z_step = (uint64_t)((EY * EXC * CELL) >> 4);
      // cin >= 16: K halves are the two 8-channel planes (LBO = 2 planes); cin == 8: LBO is set per tile pair.
      // SBO steps the 16 row groups: WT brick lines apart.
      const uint64_t a_hi0 = make_desc(brick, CIN8 ? 0u : 2 * PL, WT * EXC * CELL);
      const uint64_t a_lo0 = make_desc(brick + PL, CIN8 ? 0u : 2 * PL, WT * EXC * CELL);
      const uint64_t b0 = make_desc(bsm, b_lbo, 128);
      const bool b_resident = a.kchunks == 1;          // weights loaded once per CTA
      bool alive = true;
      uint32_t n_full = 0, n_mma = 0;                  // completed phases of bar_full / bar_mma
      int it = 0;
      for (int tile = blockIdx.x; tile < total_tiles && alive; tile += gridDim.x) {
        int r = (FFL && a.ff_list) ? a.ff_list[1 + tile] : tile;
        const int bx = r % tx_n; r /= tx_n;
        const int by = r % ty_n; r /= ty_n;
        const int bz = r % tz_n; r /= tz_n;
        const int b = r;
        const int x0 = bx * TILE_X, y0 = by * TILE_Y * WT, z0 = bz * a.zt;
        bool computed = true;                                      // far-field tiles are copied by the epilogue warps instead
        if constexpr (EPI == UEPI_VRN) computed = !(a.ff_mask && ff_tile_clear(a.ff_mask, a.n, a.zt, b, by, bx, z0, ty_n));
        const int set = it % a.nsets, use = it / a.nsets;          // use-th time this accumulator set is filled (it counts COMPUTED tiles)
        for (int ch = 0; ch < a.kchunks && alive && computed; ++ch) {
          const bool load_b = !b_resident || it == 0;
          if (it > 0 || ch > 0) { alive = mbar_wait(bar_mma, (n_mma - 1) & 1, a.err, -102); if (!alive) break; }   // brick (and B) free
          mbar_expect_tx(bar_full, (uint32_t)(((a.dbg & 2) ? 0 : a.a_bytes) + (load_b ? a.b_bytes : 0)));
          if (!(a.dbg & 2)) tma_load_5d(brick, &tmap, bar_full, (x0 + a.origin) * 8, y0 + a.origin, z0 + a.origin, ch * a.ppc, b);
          if (load_b) bulk_load(bsm, reinterpret_cast<const uint8_t*>(a.wpacked) + (size_t)ch * a.b_bytes, (uint32_t)a.b_bytes, bar_full);
          if (ch == 0 && use >= 1) { alive = mbar_wait(bar_free + 8 * set, (use - 1) & 1, a.err, -104); if (!alive) break; }   // epilogue of the set's previous tile done
          alive = mbar_wait(bar_full, n_full & 1, a.err, -101);
          ++n_full;
          if (!alive) break;
          asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
          const bool last = ch + 1 == a.kchunks;
          for (int zi = 0; zi < a.zt; ++zi) {
            if (!(a.dbg & 1))
              issue_slice<NP, TAPS, WT>(tmem_base + set * set_cols + (uint32_t)(zi * 2 * NP), a_hi0 + zi * z_step, a_lo0 + zi * z_step, b0, ch == 0,
                                        a.tap_mask[ch & 15]);
            if (last) umma_commit(bar_z + 8 * (set * MAX_ZT + zi));      // slice final: its epilogue overlaps the following MMAs
          }
          umma_commit(bar_mma);                       // brick reusable once these MMAs retire
          ++n_mma;
        }
        it += computed ? 1 : 0;
      }
    }
    __syncwarp();
  } else {
    // ------------------------------ epilogue: 8 warps; warp w reads TMEM lanes 32*(w&3).., z-slices of parity w>>2 ------------------------------
    const int row = (warp & 3) * 32 + lane;          // M row = TMEM lane = (y group, x) of the tile
    const size_t plane_elems = (size_t)a.n * a.n * a.n * 8;
    int it = 0;
    for (int tile = blockIdx.x; tile < total_tiles; tile += gridDim.x) {
      int r = (FFL && a.ff_list) ? a.ff_list[1 + tile] : tile;
      const int bx = r % tx_n; r /= tx_n;
      const int by = r % ty_n; r /= ty_n;
      const int bz = r % tz_n; r /= tz_n;
      const int b = r;
      const int x0 = bx * TILE_X, y0 = by * TILE_Y * WT, z0 = bz * a.zt;
      const int vx = x0 + (row & 7), vyb = y0 + WT * (row >> 3);
      if constexpr (EPI == UEPI_VRN) {
        if (a.ff_mask && ff_tile_clear(a.ff_mask, a.n, a.zt, b, by, bx, z0, ty_n)) {
          // far-field tile: no MMA, no barrier -- every voxel is the empty cube's at the same position, which the slot already holds
          // where the tile was far for its previous cube as well
          if (!a.ff_prev || !ff_tile_clear(a.ff_prev, a.n, a.zt, b, by, bx, z0, ty_n))
            for (int zi = (warp >> 2); zi < a.zt; zi += 2) ff_copy_voxels<NPJ, WT>(a, b, z0 + zi, vyb, vx, plane_elems);
          continue;
        }
      }
      const int set = it % a.nsets, use = it / a.nsets;
      const uint32_t lane_base = tmem_base + set * set_cols + ((uint32_t)((warp & 3) * 32) << 16);
      for (int zi = (warp >> 2); zi < ((a.dbg & 4) ? 0 : a.zt); zi += 2) {
        const int vz = z0 + zi;
        // Voxception tail: the block input does not depend on the accumulator -- fetch it before waiting for the MMAs
        constexpr int RCP = EPI == UEPI_VRN ? VrnRc<NPJ>::value : 1;
        constexpr bool PREF = EPI == UEPI_VRN && WT * RCP <= 4;             // register budget: up to 4 cells (32 registers)
        uint4 rhi[PREF ? WT : 1][RCP], rlo[PREF ? WT : 1][RCP];
        if (PREF) {
#pragma unroll
          for (int j = 0; j < WT; ++j) vrn_load_residual<RCP>(a, b, vz, vyb + j, vx, plane_elems, rhi[j], rlo[j]);
        }
        if (!mbar_wait(bar_z + 8 * (set * MAX_ZT + zi), use & 1, a.err, -103)) break;
        asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
        if (EPI == UEPI_UP) {
          // stride-2 transposed conv: column block [cls*cout, (cls+1)*cout) is output voxel 2t + r(cls) (gather form, no atomics)
          const int on = 2 * a.n;
          const size_t out_plane = (size_t)on * on * on * 8;
          __nv_bfloat16* ob = a.out_pm + (size_t)b * a.out_planes * out_plane;
#pragma unroll 1
          for (int cls = 0; cls < a.up_ncls; ++cls) {
            const int gc = a.up_cls0 + cls;
            const int oz = 2 * vz + ((gc >> 2) & 1), oy = 2 * vyb + ((gc >> 1) & 1), ox = 2 * vx + (gc & 1);
            __nv_bfloat16* oc = ob + (((size_t)oz * on + oy) * on + ox) * 8;
            for (int j = 0; j < a.up_cout / 16; ++j) {
              const int col = cls * a.up_cout + j * 16;
              float d1[16], d2[16], t[16];
              tmem_ld16(lane_base + (uint32_t)(zi * 2 * NP + col), d1);
              tmem_ld16(lane_base + (uint32_t)(zi * 2 * NP + NP + col), d2);
#pragma unroll
              for (int i = 0; i < 16; ++i) t[i] = fmaxf((d1[i] + d2[i]) + s_bias[col + i], 0.f);
              split_store(oc + (size_t)(4 * j) * out_plane, oc + (size_t)(4 * j + 1) * out_plane, t);
              split_store(oc + (size_t)(4 * j + 2) * out_plane, oc + (size_t)(4 * j + 3) * out_plane, t + 8);
            }
          }
          continue;
        }
        float v[EPI == UEPI_UP ? 16 : NP];
#pragma unroll
        for (int j = 0; j < (EPI == UEPI_UP ? 0 : NP / 16); ++j) {
          float d1[16], d2[16];
          tmem_ld16(lane_base + (uint32_t)(zi * 2 * NP + j * 16), d1);
          tmem_ld16(lane_base + (uint32_t)(zi * 2 * NP + NP + j * 16), d2);
#pragma unroll
          for (int i4 = 0; i4 < 4; ++i4) {                     // bias as 16-byte shared loads (4x fewer LSU wavefronts than scalar reads)
            const float4 bq = reinterpret_cast<const float4*>(s_bias)[j * 4 + i4];
            v[j * 16 + 4 * i4 + 0] = (d1[4 * i4 + 0] + d2[4 * i4 + 0]) + bq.x;
            v[j * 16 + 4 * i4 + 1] = (d1[4 * i4 + 1] + d2[4 * i4 + 1]) + bq.y;
            v[j * 16 + 4 * i4 + 2] = (d1[4 * i4 + 2] + d2[4 * i4 + 2]) + bq.z;
            v[j * 16 + 4 * i4 + 3] = (d1[4 * i4 + 3] + d2[4 * i4 + 3]) + bq.w;
          }
        }
#pragma unroll
        for (int j = 0; j < WT; ++j)
          epilogue_voxel<NPJ, (EPI == UEPI_UP ? UEPI_F32 : EPI)>(a, v + (EPI == UEPI_UP ? 0 : j * NPJ), s_w23, b, vz, vyb + j, vx, plane_elems,
                                                                  PREF ? rhi[j] : nullptr, PREF ? rlo[j] : nullptr);
      }
      // A warp without a slice of its own (zt == 1: warps 4..7) must not run ahead of the MMAs: its arrival for a LATER use
      // of the set would otherwise complete the current phase early.  Pace it on the tile's last slice.
      if ((warp >> 2) >= a.zt) mbar_wait(bar_z + 8 * (set * MAX_ZT + a.zt - 1), use & 1, a.err, -105);
      // this warp is done reading the accumulator set of tile `it`: hand it back to the MMA issuer
      asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
      __syncwarp();
      if (lane == 0) asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(bar_free + 8 * set) : "memory");
      ++it;
    }
  }
  asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
  __syncthreads();
  if (warp == EPI_WARPS) {
    asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem_base), "r"(a.tmem_cols) : "memory");
  }
}

// Z-STREAMING kernel (r01, third form).  The tile kernel above re-reads every input z-slice (zt+2)/zt times from L2 and holds
// one single-buffered brick per CTA, so it needs 2-3 co-resident CTAs to hide the brick load and the serial work of its one
// producer/issuer thread -- which the y-banded forms (larger bricks, more B tiles) cannot afford.  Here ONE CTA per SM walks
// column segments (b, x tile, y tile, zs output slices) along z with the roles split over warps:
//   * warp 8 (one lane): TMA producer.  Input z-slices stream through a ring of 8 shared-memory slots, one 5-D TMA box of ONE
//     slice per slot, as far ahead as the ring allows; every slice is fetched (zs+2)/zs times instead of (zt+2)/zt.
//   * warps 9-11 (one lane each): MMA issuers.  Output slice O belongs to issuer O % 3, which multiplies the slots of input
//     slices O, O+1, O+2 (kz = 0, 1, 2: three descriptor bases instead of an address offset) into accumulator slot
//     O % NACC.  Three issuers keep three independent accumulation chains in the tensor pipe and hide each other's barrier
//     waits; one output is issued by ONE thread in the tile kernel's tap order, so results are bit-identical to it.
//   * warps 0-7: epilogue, even / odd outputs; the accumulator slot is released as soon as it is in registers.
//   * barriers, one phase per use: full[slot] (TMA landed; up to three issuers wait on it), sfree[slot] (count 3: one
//     tcgen05.commit per reading issuer; the producer supplies the missing arrivals of the halo slices that have fewer than
//     three readers), afull[acc] (commit after the output's 3 x NTZ tiles), afree[acc] (4 epilogue warps), b (weights, once).
// Loads and outputs are flat sequences across the CTA's segments, so the ring never drains at a segment boundary.
constexpr int RING_MAX = 8;                              // ring slots: 8, or 4 where 8 do not fit (power of two: slot = load & (R-1))
constexpr int STREAM_ISSUERS = 3;
constexpr int STREAM_THREADS = 32 * (EPI_WARPS + 1 + STREAM_ISSUERS);

// The taps of ONE kz of one output slice: NTZ (d, kx) tiles, two MMAs each.
template <int NP, bool PAIRED, int WT>
__device__ __forceinline__ void issue_kz(uint32_t d, uint64_t a_hi, uint64_t a_lo, uint64_t bdesc, bool first) {
  constexpr uint32_t idesc_full = make_idesc(128, 2 * NP), idesc_half = make_idesc(128, NP);
  constexpr int NTZ = 3 * (WT + 2);                              // A tiles (d, kx) per kz
  constexpr uint64_t b_step = (uint64_t)((2 * NP * 32) >> 4);
  static_assert(!PAIRED || NTZ % 2 == 0, "paired taps must not straddle two z-slices");
#pragma unroll
  for (int t = 0; t < (PAIRED ? NTZ / 2 : NTZ); ++t) {
    uint64_t add;
    if (!PAIRED) {
      add = (uint64_t)(((((t / 3) * EXC) + t % 3) * CELL) >> 4);
    } else {
      const int ta = 2 * t, tb = 2 * t + 1;
      const int oa = ((ta / 3) * EXC + ta % 3) * CELL, ob = ((tb / 3) * EXC + tb % 3) * CELL;
      add = (uint64_t)(oa >> 4) | ((uint64_t)((ob - oa) >> 4) << 16);
    }
    const uint64_t bd = bdesc + (uint64_t)t * b_step;
    umma_f16(d, a_hi + add, bd, idesc_full, (t == 0 && first) ? 0u : 1u);      // x_hi * [w_hi | w_lo]
    umma_f16(d, a_lo + add, bd, idesc_half, 1u);                               // x_lo * w_hi
  }
}

template <int NP, int EPI, bool PAIRED, int WT>
__global__ void __launch_bounds__(STREAM_THREADS, 1) conv_umma_stream_kernel(const __grid_constant__ CUtensorMap tmap, const UmmaArgs a) {
  extern __shared__ __align__(128) uint8_t smem[];
  uint8_t* s_a = smem;
  uint8_t* s_b = smem + (size_t)a.ring * a.slot_bytes;
  uint64_t* s_bar = reinterpret_cast<uint64_t*>(s_b + a.b_bytes);          // full[8], sfree[8], afull[8], afree[8], b
  uint32_t* s_tmem = reinterpret_cast<uint32_t*>(s_bar + 4 * 8 + 1);
  float* s_bias = reinterpret_cast<float*>(s_bar + 4 * 8 + 2);             // 16-byte aligned
  float* s_w23 = s_bias + NP;
  const uint32_t bar_full = smem_u32(s_bar), bar_sfree = smem_u32(s_bar + 8), bar_afull = smem_u32(s_bar + 16),
                 bar_afree = smem_u32(s_bar + 24), bar_b = smem_u32(s_bar + 32);
  constexpr int NACC = NP <= 32 ? 8 : 4;                         // accumulator slots of 2*NP columns (power of two)
  constexpr int NACC_SH = NP <= 32 ? 3 : 2;
  constexpr int NPJ = NP / WT;
  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  const int ZS = a.zs;
  const int RMASK = a.ring - 1, RSH = a.ring == 8 ? 3 : 2;
  const int tx_n = a.n / TILE_X, ty_n = a.n / (TILE_Y * WT), tz_n = a.n / ZS;
  const int total_segs = tx_n * ty_n * tz_n * a.batch;
  const int n_my = ((int)blockIdx.x < total_segs) ? (total_segs - (int)blockIdx.x + (int)gridDim.x - 1) / (int)gridDim.x : 0;
  const int total_outs = n_my * ZS;

  for (int i = tid; i < NP; i += STREAM_THREADS) s_bias[i] = a.bias ? a.bias[i] : 0.f;
  if (EPI == UEPI_VRN) for (int i = tid; i < a.c4 * a.c2 + a.c2; i += STREAM_THREADS) s_w23[i] = i < a.c4 * a.c2 ? a.w23[i] : a.b23[i - a.c4 * a.c2];
  if (tid == 0) {
    for (int i = 0; i < 8; ++i) {
      mbar_init(bar_full + 8 * i, 1); mbar_init(bar_sfree + 8 * i, 3);
      mbar_init(bar_afull + 8 * i, 1); mbar_init(bar_afree + 8 * i, EPI_WARPS / 2);
    }
    mbar_init(bar_b, 1);
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  }
  if (warp == EPI_WARPS) {
    asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(s_tmem)), "r"(a.tmem_cols) : "memory");
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
  }
  asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
  __syncthreads();
  asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
  const uint32_t tmem_base = *s_tmem;
  const uint32_t ring0 = smem_u32(s_a);
  const uint32_t SP = (uint32_t)a.slice_plane, SB = (uint32_t)a.slot_bytes;

  if (warp == EPI_WARPS) {
    if (elect_one() && n_my > 0) {
      // ------------------------------ TMA producer ------------------------------
      mbar_expect_tx(bar_b, (uint32_t)a.b_bytes);
      bulk_load(smem_u32(s_b), a.wpacked, (uint32_t)a.b_bytes, bar_b);
      int l = 0;
      bool alive = true;
      for (int sk = 0; sk < n_my && alive; ++sk) {
        int r = (int)blockIdx.x + sk * (int)gridDim.x;
        const int bx = r % tx_n; r /= tx_n;
        const int by = r % ty_n; r /= ty_n;
        const int bz = r % tz_n; r /= tz_n;
        const int cx = (bx * TILE_X + a.origin) * 8, cy = by * TILE_Y * WT + a.origin, cz = bz * ZS + a.origin;
        for (int k = 0; k < ZS + 2; ++k, ++l) {
          const int slot = l & RMASK, use = l >> RSH;
          if (use >= 1 && !mbar_wait(bar_sfree + 8 * slot, (use - 1) & 1, a.err, -112)) { alive = false; break; }
          mbar_expect_tx(bar_full + 8 * slot, SB);
          tma_load_5d(ring0 + slot * SB, &tmap, bar_full + 8 * slot, cx, cy, cz + k, 0, r);
          // halo slices have fewer than three reading outputs: supply the missing releases now
          const int readers = min(k, ZS - 1) - max(k - 2, 0) + 1;
          for (int e = readers; e < 3; ++e) asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(bar_sfree + 8 * slot) : "memory");
        }
      }
    }
    __syncwarp();
  } else if (warp > EPI_WARPS) {
    if (elect_one() && n_my > 0) {
      // ------------------------------ MMA issuer `me`: outputs O = me, me + 3, ... ------------------------------
      const int me = warp - EPI_WARPS - 1;
      constexpr int NTK = PAIRED ? 3 * (WT + 2) / 2 : 3 * (WT + 2);  // B tiles per kz
      constexpr uint64_t b_step = (uint64_t)((2 * NP * 32) >> 4);
      const uint64_t b0 = make_desc(smem_u32(s_b), 2 * NP * 16, 128);
      bool alive = mbar_wait(bar_b, 0, a.err, -110);
      int sk = 0, o = me;
      while (o >= ZS) { o -= ZS; ++sk; }
      for (int O = me; O < total_outs && alive; O += STREAM_ISSUERS) {
        const int l0 = O + 2 * sk;                              // = sk * (ZS + 2) + o: the slice read with kz = 0
        const int acc = O & (NACC - 1), ause = O >> NACC_SH;
        if (ause >= 1) { alive = mbar_wait(bar_afree + 8 * acc, (ause - 1) & 1, a.err, -114); if (!alive) break; }
        const uint32_t d = tmem_base + (uint32_t)(acc * 2 * NP);
#pragma unroll
        for (int kz = 0; kz < 3; ++kz) {
          const int l = l0 + kz, slot = l & RMASK;
          alive = mbar_wait(bar_full + 8 * slot, (l >> RSH) & 1, a.err, -111);
          if (!alive) break;
          asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
          const uint32_t base = ring0 + (uint32_t)slot * SB;
          // cin >= 16: K halves are the two 8-channel planes (LBO = 2 planes); cin == 8: LBO is set per tile pair
          const uint64_t dh = make_desc(base, PAIRED ? 0u : 2 * SP, WT * EXC * CELL), dl = make_desc(base + SP, PAIRED ? 0u : 2 * SP, WT * EXC * CELL);
          if (!(a.dbg & 1)) issue_kz<NP, PAIRED, WT>(d, dh, dl, b0 + (uint64_t)(kz * NTK) * b_step, kz == 0);
          umma_commit(bar_sfree + 8 * slot);                    // this reader is done with the slice once its MMAs retire
        }
        if (!alive) break;
        umma_commit(bar_afull + 8 * acc);
        o += STREAM_ISSUERS;
        while (o >= ZS) { o -= ZS; ++sk; }
      }
    }
    __syncwarp();
  } else {
    // ------------------------------ epilogue: warps 0-3 take even outputs, 4-7 odd ones ------------------------------
    const int row = (warp & 3) * 32 + lane;
    const size_t plane_elems = (size_t)a.n * a.n * a.n * 8;
    int sk = 0, o = warp >> 2, cur = -1, bx = 0, by = 0, bz = 0, b = 0;
    while (o >= ZS) { o -= ZS; ++sk; }
    for (int O = (warp >> 2); O < ((a.dbg & 4) ? 0 : total_outs); O += 2) {
      if (sk != cur) {
        int r = (int)blockIdx.x + sk * (int)gridDim.x;
        bx = r % tx_n; r /= tx_n;
        by = r % ty_n; r /= ty_n;
        bz = r % tz_n; r /= tz_n;
        b = r; cur = sk;
      }
      const int vx = bx * TILE_X + (row & 7), vyb = by * TILE_Y * WT + WT * (row >> 3), vz = bz * ZS + o;
      const int acc = O & (NACC - 1), ause = O >> NACC_SH;
      // Voxception tail: the block input does not depend on the accumulator -- fetch it while the MMAs still run
      constexpr int RC = EPI == UEPI_VRN ? VrnRc<NPJ>::value : 1;
      uint4 rhi[WT][RC], rlo[WT][RC];
      if (EPI == UEPI_VRN) {
#pragma unroll
        for (int j = 0; j < WT; ++j) vrn_load_residual<RC>(a, b, vz, vyb + j, vx, plane_elems, rhi[j], rlo[j]);
      }
      if (!mbar_wait(bar_afull + 8 * acc, ause & 1, a.err, -113)) break;
      asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
      const uint32_t lane_base = tmem_base + (uint32_t)(acc * 2 * NP) + ((uint32_t)((warp & 3) * 32) << 16);
      float v[NP];
      if (NP == 16 || NP == 32) {
        float dd[2 * NP];                                        // [x_hi*w_hi + x_lo*w_hi | x_hi*w_lo] in one TMEM round trip
        tmem_ld<(NP == 16 || NP == 32) ? 2 * NP : 32>(lane_base, dd);
#pragma unroll
        for (int i4 = 0; i4 < NP / 4; ++i4) {
          const float4 bq = reinterpret_cast<const float4*>(s_bias)[i4];
          v[4 * i4 + 0] = (dd[4 * i4 + 0] + dd[NP + 4 * i4 + 0]) + bq.x;
          v[4 * i4 + 1] = (dd[4 * i4 + 1] + dd[NP + 4 * i4 + 1]) + bq.y;
          v[4 * i4 + 2] = (dd[4 * i4 + 2] + dd[NP + 4 * i4 + 2]) + bq.z;
          v[4 * i4 + 3] = (dd[4 * i4 + 3] + dd[NP + 4 * i4 + 3]) + bq.w;
        }
      } else {
#pragma unroll
        for (int j = 0; j < NP / 16; ++j) {
          float d1[16], d2[16];
          tmem_ld16(lane_base + (uint32_t)(j * 16), d1);
          tmem_ld16(lane_base + (uint32_t)(NP + j * 16), d2);
#pragma unroll
          for (int i4 = 0; i4 < 4; ++i4) {                     // bias as 16-byte shared loads (4x fewer LSU wavefronts than scalar reads)
            const float4 bq = reinterpret_cast<const float4*>(s_bias)[j * 4 + i4];
            v[j * 16 + 4 * i4 + 0] = (d1[4 * i4 + 0] + d2[4 * i4 + 0]) + bq.x;
            v[j * 16 + 4 * i4 + 1] = (d1[4 * i4 + 1] + d2[4 * i4 + 1]) + bq.y;
            v[j * 16 + 4 * i4 + 2] = (d1[4 * i4 + 2] + d2[4 * i4 + 2]) + bq.z;
            v[j * 16 + 4 * i4 + 3] = (d1[4 * i4 + 3] + d2[4 * i4 + 3]) + bq.w;
          }
        }
      }
      // the accumulator slot is in registers now: hand it back before the (long) epilogue math and stores
      asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
      __syncwarp();
      if (lane == 0) asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(bar_afree + 8 * acc) : "memory");
#pragma unroll
      for (int j = 0; j < WT; ++j)
        epilogue_voxel<NPJ, EPI>(a, v + j * NPJ, s_w23, b, vz, vyb + j, vx, plane_elems, EPI == UEPI_VRN ? rhi[j] : nullptr, EPI == UEPI_VRN ? rlo[j] : nullptr);
      o += 2;
      while (o >= ZS) { o -= ZS; ++sk; }
    }
  }
  asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
  __syncthreads();
  if (warp == EPI_WARPS) {
    asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem_base), "r"(a.tmem_cols) : "memory");
  }
}

// Z-BANDED streaming kernel (r01, fourth form) for the thin-N layers at 64^3 (K_a16: 8 real columns; deconv_out: 1).  Same roles
// and ring as conv_umma_stream_kernel, but the MMA is INPUT-slice stationary: one MMA per (d, kx) tile of input slice i carries
// the three kz taps as column blocks [kz=0 | kz=1 | kz=2] (N = 2*48 then 48), so the 4 KiB A tile -- the operand fetch that
// bounds these layers -- is read once for the three output slices it feeds instead of three times.  The accumulator slot of
// input slice i then holds the partial sums P_i[kz] of outputs i, i-1, i-2; the epilogue of output O adds P_O[0] + P_{O+1}[1] +
// P_{O+2}[2] (+ bias) in registers.  FP32 partial sums are added in a different order than in the tile kernel, so results agree
// with it to FP32 rounding (not bit for bit); the order is fixed, so the kernel is deterministic.
//   barriers: full[slot] / sfree[slot] (count 1: one issuer reads a slice), pfull[ts] (partial sums of an input slice complete),
//   pfree[ts] (count 12 = 3 reading outputs x 4 epilogue warps; the issuer supplies the arrivals of the missing readers of halo
//   slices), b.  5 TMEM slots of 96 columns.
constexpr int ZB_SLOTS = 5;                          // TMEM slots of 96 columns (one per input slice in flight)

// EG epilogue groups of 4 warps (output O belongs to group O % EG), NI issuer warps (input slice l belongs to issuer l % NI).
// The Voxception-tail form (K_b16) is bound by its epilogue: it runs 3 groups and 1 issuer; the plain forms 2 and 3.
// NPT = accumulator columns per kz block: 16 (hi and lo products in separate column halves, two MMAs per tile) or 32 (SPLIT3:
// x_hi*w_hi, x_lo*w_hi and x_hi*w_lo are three MMAs into the SAME 96 columns, so that 5 slots still fit the 512 TMEM columns).
template <int NPT, int EPI, int WT, bool PAIRED, int EG, int NI>
__global__ void __launch_bounds__(32 * (4 * EG + 1 + NI), 1) conv_umma_zband_kernel(const __grid_constant__ CUtensorMap tmap, const UmmaArgs a) {
  extern __shared__ __align__(128) uint8_t smem[];
  uint8_t* s_a = smem;
  uint8_t* s_b = smem + (size_t)a.ring * a.slot_bytes;
  uint64_t* s_bar = reinterpret_cast<uint64_t*>(s_b + a.b_bytes);          // full[8], sfree[8], pfull[8], pfree[8], b
  uint32_t* s_tmem = reinterpret_cast<uint32_t*>(s_bar + 4 * 8 + 1);
  float* s_bias = reinterpret_cast<float*>(s_bar + 4 * 8 + 2);
  const uint32_t bar_full = smem_u32(s_bar), bar_sfree = smem_u32(s_bar + 8), bar_pfull = smem_u32(s_bar + 16),
                 bar_pfree = smem_u32(s_bar + 24), bar_b = smem_u32(s_bar + 32);
  constexpr int NP = NPT, NB = 3 * NP, NPJ = NP / WT;
  constexpr bool SPLIT3 = NP == 32;
  constexpr int SLOT_COLS = SPLIT3 ? NB : 2 * NB;
  constexpr int NTZ = 3 * (WT + 2);
  constexpr int EW = 4 * EG, THREADS = 32 * (EW + 1 + NI);
  float* s_w23 = s_bias + NP;                                              // [c4][c2] then b23[c2] (UEPI_VRN only)
  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  const int ZS = a.zs, LPS = ZS + 2;
  const int RMASK = a.ring - 1, RSH = a.ring == 8 ? 3 : 2;
  const int tx_n = a.n / TILE_X, ty_n = a.n / (TILE_Y * WT), tz_n = a.n / ZS;
  const int total_segs = tx_n * ty_n * tz_n * a.batch;
  // far-field segments (UmmaArgs::ff_list): the CTAs share the list of the segments to compute, so that the work is balanced however the
  // occupied voxels lie; loads, outputs and barrier phases count listed segments only
  const int n_units = a.ff_list ? a.ff_list[0] : total_segs;
  const int n_my = ((int)blockIdx.x < n_units) ? (n_units - (int)blockIdx.x + (int)gridDim.x - 1) / (int)gridDim.x : 0;
  auto seg_of = [&](int sk) -> int { const int u = (int)blockIdx.x + sk * (int)gridDim.x; return a.ff_list ? a.ff_list[1 + u] : u; };
  const int total_outs = n_my * ZS, total_loads = n_my * LPS;

  for (int i = tid; i < NP; i += THREADS) s_bias[i] = a.bias ? a.bias[i] : 0.f;
  if (EPI == UEPI_VRN) for (int i = tid; i < a.c4 * a.c2 + a.c2; i += THREADS) s_w23[i] = i < a.c4 * a.c2 ? a.w23[i] : a.b23[i - a.c4 * a.c2];
  if (tid == 0) {
    for (int i = 0; i < 8; ++i) {
      mbar_init(bar_full + 8 * i, 1); mbar_init(bar_sfree + 8 * i, 1);
      mbar_init(bar_pfull + 8 * i, 1); mbar_init(bar_pfree + 8 * i, 12);            // 3 reading outputs x 4 warps
    }
    mbar_init(bar_b, 1);
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  }
  if (warp == EW) {
    asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(s_tmem)), "r"(a.tmem_cols) : "memory");
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
  }
  asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
  __syncthreads();
  asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
  const uint32_t tmem_base = *s_tmem;
  const uint32_t ring0 = smem_u32(s_a);
  const uint32_t SP = (uint32_t)a.slice_plane, SB = (uint32_t)a.slot_bytes;

  if (warp == EW) {
    if (elect_one() && n_my > 0) {
      // ------------------------------ TMA producer ------------------------------
      mbar_expect_tx(bar_b, (uint32_t)a.b_bytes);
      bulk_load(smem_u32(s_b), a.wpacked, (uint32_t)a.b_bytes, bar_b);
      int l = 0;
      bool alive = true;
      for (int sk = 0; sk < n_my && alive; ++sk) {
        int r = seg_of(sk);
        const int bx = r % tx_n; r /= tx_n;
        const int by = r % ty_n; r /= ty_n;
        const int bz = r % tz_n; r /= tz_n;
        const int cx = (bx * TILE_X + a.origin) * 8, cy = by * TILE_Y * WT + a.origin, cz = bz * ZS + a.origin;
        for (int k = 0; k < LPS; ++k, ++l) {
          const int slot = l & RMASK, use = l >> RSH;
          if (use >= 1 && !mbar_wait(bar_sfree + 8 * slot, (use - 1) & 1, a.err, -122)) { alive = false; break; }
          mbar_expect_tx(bar_full + 8 * slot, SB);
          tma_load_5d(ring0 + slot * SB, &tmap, bar_full + 8 * slot, cx, cy, cz + k, 0, r);
        }
      }
    }
    __syncwarp();
  } else if (warp > EW) {
    if (elect_one() && n_my > 0) {
      // ------------------------------ MMA issuer `me`: input slices l = me, me + NI, ... ------------------------------
      const int me = warp - EW - 1;
      constexpr uint32_t idesc_full = make_idesc(128, SPLIT3 ? NB : 2 * NB), idesc_half = make_idesc(128, NB);
      constexpr uint64_t b_step = (uint64_t)((2 * NB * 32) >> 4);
      const uint64_t b0 = make_desc(smem_u32(s_b), 2 * NB * 16, 128);
      bool alive = mbar_wait(bar_b, 0, a.err, -120);
      int k = me;                                               // position of slice l inside its segment
      while (k >= LPS) k -= LPS;
      for (int l = me; l < total_loads && alive; l += NI) {
        const int slot = l & RMASK, ts = l % ZB_SLOTS, tuse = l / ZB_SLOTS;
        if (tuse >= 1) { alive = mbar_wait(bar_pfree + 8 * ts, (tuse - 1) & 1, a.err, -124); if (!alive) break; }
        alive = mbar_wait(bar_full + 8 * slot, (l >> RSH) & 1, a.err, -121);
        if (!alive) break;
        asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
        const uint32_t d = tmem_base + (uint32_t)(ts * SLOT_COLS);
        if (PAIRED) {
          // cin == 8: K = 16 spans a PAIR of (d, kx) tiles (LBO = their address difference); odd tile count: tile 0 goes alone
          const uint32_t base = ring0 + (uint32_t)slot * SB;
          const uint64_t dh = make_desc(base, 0u, WT * EXC * CELL), dl = make_desc(base + SP, 0u, WT * EXC * CELL);
          constexpr int NTP = (NTZ + 1) / 2;
#pragma unroll
          for (int m = 0; m < NTP && !(a.dbg & 1); ++m) {
            const int ta = (NTZ & 1) ? (m == 0 ? 0 : 2 * m - 1) : 2 * m, tb = (NTZ & 1) ? (m == 0 ? 1 : 2 * m) : 2 * m + 1;
            const int oa = ((ta / 3) * EXC + ta % 3) * CELL, ob = ((tb / 3) * EXC + tb % 3) * CELL;
            const uint64_t add = (uint64_t)(oa >> 4) | ((uint64_t)((ob - oa) >> 4) << 16);
            const uint64_t bd = b0 + (uint64_t)m * b_step;
            umma_f16(d, dh + add, bd, idesc_full, m == 0 ? 0u : 1u);
            umma_f16(d, dl + add, bd, idesc_half, 1u);
            if (SPLIT3) umma_f16(d, dh + add, bd + (uint64_t)NB, idesc_half, 1u);      // x_hi * w_lo (rows NB.. of the B tile)
          }
        } else {
          for (int ch = 0; ch < a.kchunks && !(a.dbg & 1); ++ch) {          // 16 input channels (4 planes) per chunk
            const uint32_t base = ring0 + (uint32_t)slot * SB + (uint32_t)ch * 4u * SP;
            const uint64_t dh = make_desc(base, 2 * SP, WT * EXC * CELL), dl = make_desc(base + SP, 2 * SP, WT * EXC * CELL);
            const uint64_t bc = b0 + (uint64_t)(ch * NTZ) * b_step;
#pragma unroll
            for (int t = 0; t < NTZ; ++t) {
              const uint64_t add = (uint64_t)(((((t / 3) * EXC) + t % 3) * CELL) >> 4);
              const uint64_t bd = bc + (uint64_t)t * b_step;
              umma_f16(d, dh + add, bd, idesc_full, (ch == 0 && t == 0) ? 0u : 1u);   // x_hi * [w_hi(kz 0,1,2) | w_lo(kz 0,1,2)]  (SPLIT3: w_hi only)
              umma_f16(d, dl + add, bd, idesc_half, 1u);                               // x_lo * w_hi(kz 0,1,2)
              if (SPLIT3) umma_f16(d, dh + add, bd + (uint64_t)NB, idesc_half, 1u);    // x_hi * w_lo(kz 0,1,2) into the same columns
            }
          }
        }
        umma_commit(bar_sfree + 8 * slot);
        umma_commit(bar_pfull + 8 * ts);
        // halo slices feed fewer than three outputs: supply the epilogue arrivals of the missing readers
        const int readers = min(k, ZS - 1) - max(k - 2, 0) + 1;
        for (int e = readers * 4; e < 12; ++e)
          asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(bar_pfree + 8 * ts) : "memory");
        k += NI;
        while (k >= LPS) k -= LPS;
      }
    }
    __syncwarp();
  } else {
    // ------------------------------ epilogue: group g = warp / 4 takes outputs O = g, g + EG, ... ------------------------------
    const int row = (warp & 3) * 32 + lane;
    const size_t plane_elems = (size_t)a.n * a.n * a.n * 8;
    int sk = 0, o = warp >> 2, cur = -1, bx = 0, by = 0, bz = 0, b = 0;
    while (o >= ZS) { o -= ZS; ++sk; }
    for (int O = (warp >> 2); O < ((a.dbg & 4) ? 0 : total_outs); O += EG) {
      if (sk != cur) {
        int r = seg_of(sk);
        bx = r % tx_n; r /= tx_n;
        by = r % ty_n; r /= ty_n;
        bz = r % tz_n; r /= tz_n;
        b = r; cur = sk;
      }
      const int vx = bx * TILE_X + (row & 7), vyb = by * TILE_Y * WT + WT * (row >> 3), vz = bz * ZS + o;
      const int l0 = O + 2 * sk;                                // input slice read with kz = 0
      // Voxception tail: the block input does not depend on the accumulators -- fetch it while the MMAs still run
      constexpr int RC = EPI == UEPI_VRN ? VrnRc<NPJ>::value : 1;
      uint4 rhi[WT][RC], rlo[WT][RC];
      if (EPI == UEPI_VRN) {
#pragma unroll
        for (int j = 0; j < WT; ++j) vrn_load_residual<RC>(a, b, vz, vyb + j, vx, plane_elems, rhi[j], rlo[j]);
      }
      float v[NP];
      bool ok = true;
#pragma unroll
      for (int kz = 0; kz < 3; ++kz) {
        const int l = l0 + kz, ts = l % ZB_SLOTS;
        if (!mbar_wait(bar_pfull + 8 * ts, (l / ZB_SLOTS) & 1, a.err, -123)) { ok = false; break; }
        asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
        const uint32_t lane_base = tmem_base + (uint32_t)(ts * SLOT_COLS + kz * NP) + ((uint32_t)((warp & 3) * 32) << 16);
#pragma unroll
        for (int q = 0; q < NP / 16; ++q) {
          float d1[16], d2[16];
          tmem_ld16(lane_base + (uint32_t)(q * 16), d1);
          if (!SPLIT3) tmem_ld16(lane_base + (uint32_t)(NB + q * 16), d2);
#pragma unroll
          for (int i = 0; i < 16; ++i) {
            const float p = SPLIT3 ? d1[i] : (d1[i] + d2[i]);
            v[q * 16 + i] = kz == 0 ? p : v[q * 16 + i] + p;
          }
        }
        asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
        __syncwarp();
        if (lane == 0) asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(bar_pfree + 8 * ts) : "memory");
      }
      if (!ok) break;
#pragma unroll
      for (int i = 0; i < NP; ++i) v[i] += s_bias[i];
#pragma unroll
      for (int j = 0; j < WT; ++j)
        epilogue_voxel<NPJ, EPI>(a, v + j * NPJ, s_w23, b, vz, vyb + j, vx, plane_elems, EPI == UEPI_VRN ? rhi[j] : nullptr, EPI == UEPI_VRN ? rlo[j] : nullptr);
      o += EG;
      while (o >= ZS) { o -= ZS; ++sk; }
    }
  }
  asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
  __syncthreads();
  if (warp == EW) {
    asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem_base), "r"(a.tmem_cols) : "memory");
  }
}

// ---------------------------------------------------------------------------------------------- host
typedef CUresult (*EncodeTiledFn)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*, const cuuint64_t*,
                                  const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave, CUtensorMapSwizzle,
                                  CUtensorMapL2promotion, CUtensorMapFloatOOBfill);

EncodeTiledFn get_encode_fn() {
  static EncodeTiledFn fn = nullptr;
  static std::once_flag once;
  std::call_once(once, [] {
    void* p = nullptr;
    cudaDriverEntryPointQueryResult q;
    if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &p, cudaEnableDefault, &q) == cudaSuccess &&
        q == cudaDriverEntryPointSuccess)
      fn = (EncodeTiledFn)p;
  });
  return fn;
}

cudaError_t make_tmap(const PmTensor& t, int ey, int ez, int ppc, CUtensorMap* out) {
  EncodeTiledFn fn = get_encode_fn();
  if (!fn) return cudaErrorNotSupported;
  const cuuint64_t n = (cuuint64_t)t.n, planes = (cuuint64_t)(2 * t.c / 8);
  cuuint64_t gdim[5] = {n * 8, n, n, planes, (cuuint64_t)t.B};
  cuuint64_t gstride[4] = {n * 16, n * n * 16, n * n * n * 16, planes * n * n * n * 16};
  cuuint32_t box[5] = {(cuuint32_t)(EXC * 8), (cuuint32_t)ey, (cuuint32_t)ez, (cuuint32_t)ppc, 1};
  cuuint32_t estr[5] = {1, 1, 1, 1, 1};
  CUresult r = fn(out, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 5, (void*)t.p, gdim, gstride, box, estr, CU_TENSOR_MAP_INTERLEAVE_NONE,
                  CU_TENSOR_MAP_SWIZZLE_NONE, CU_TENSOR_MAP_L2_PROMOTION_L2_128B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  return r == CUDA_SUCCESS ? cudaSuccess : cudaErrorInvalidValue;
}

int pick_zt(int n, int np, int cin, int epi, int wt, int n_mma, int kchunks) {
  // zt accumulators of 2*np columns must fit 512 TMEM columns (256 so two CTAs can share an SM) and the
  // brick + weights should leave room for two CTAs per SM where possible.
  int zt = 8;
  while (zt > 1 && (zt * 2 * np > 256 || zt > n)) zt /= 2;          // one accumulator set within 256 TMEM columns
  const int ppc = cin == 8 ? 2 : 4;
  const int nm = n_mma;
  auto smem = [&](int z) { return ppc * (z + 2) * brick_ey(wt) * EXC * CELL + nm * 2 * np * 32; };
  static const int smem_kb = getenv("PCGC_UMMA_SMEM_KB") ? atoi(getenv("PCGC_UMMA_SMEM_KB")) : 100;      // tuning experiments
  while (zt > 1 && smem(zt) > smem_kb * 1024) zt /= 2;
  // MMA-bound kernels (light epilogue) overlap load / MMA / epilogue better with three CTAs per SM (measured on B200:
  // K_a16 0.676 -> 0.582 ms); the VRN-tail kernels are epilogue/HBM bound and prefer deep z tiles (less halo re-read).
  static const int three = getenv("PCGC_UMMA_3CTA") ? atoi(getenv("PCGC_UMMA_3CTA")) : 1;          // tuning experiments
  // (multi-chunk kernels re-load a brick per chunk and are L2-bound on the halo: they keep the deeper z tile)
  if (epi != UEPI_VRN && three && kchunks == 1) while (zt > 2 && smem(zt) > 75 * 1024) zt /= 2;
  static const int force = getenv("PCGC_UMMA_ZT") ? atoi(getenv("PCGC_UMMA_ZT")) : 0;      // tuning experiments
  if (force > 0 && force < zt) zt = force;
  return zt;
}

template <int NP, int E, int TAPS, int WT>
cudaError_t launch_one(const CUtensorMap& tm, const UmmaArgs& a, int grid, size_t smem, cudaStream_t s) {
  PCGC_CARVEOUT_ONCE((conv_umma_kernel<NP, E, TAPS, WT>));
  cudaError_t e = cudaFuncSetAttribute(conv_umma_kernel<NP, E, TAPS, WT>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
  if (e != cudaSuccess) return e;
  conv_umma_kernel<NP, E, TAPS, WT><<<grid, UMMA_THREADS, smem, s>>>(tm, a);
  return cudaGetLastError();
}

template <int NP, int TAPS>
cudaError_t launch_np(const CUtensorMap& tm, const UmmaArgs& a, int epi, int grid, size_t smem, cudaStream_t s) {
  if (epi == UEPI_F32) return launch_one<NP, UEPI_F32, TAPS, 1>(tm, a, grid, smem, s);
  if (epi == UEPI_PM) return launch_one<NP, UEPI_PM, TAPS, 1>(tm, a, grid, smem, s);
  if (epi == UEPI_VRN) return launch_one<NP, UEPI_VRN, TAPS, 1>(tm, a, grid, smem, s);
  return cudaErrorNotSupported;
}

// y-banded instantiations (only the shapes the layer programs use + their float32 test forms)
cudaError_t launch_banded(const CUtensorMap& tm, const UmmaArgs& a, int np, int epi, bool paired, int wt, int grid, size_t smem, cudaStream_t s) {
  if (wt == 2 && !paired) {
    if (np == 16 && epi == UEPI_PM) return launch_one<16, UEPI_PM, TAPS_27, 2>(tm, a, grid, smem, s);        // K_a16
    if (np == 16 && epi == UEPI_F32) return launch_one<16, UEPI_F32, TAPS_27, 2>(tm, a, grid, smem, s);
    if (np == 32 && epi == UEPI_PM) return launch_one<32, UEPI_PM, TAPS_27, 2>(tm, a, grid, smem, s);        // K_a32
    if (np == 32 && epi == UEPI_F32) return launch_one<32, UEPI_F32, TAPS_27, 2>(tm, a, grid, smem, s);
    if (np == 48 && epi == UEPI_VRN) return launch_one<48, UEPI_VRN, TAPS_27, 2>(tm, a, grid, smem, s);      // K_b32
    if (np == 48 && epi == UEPI_F32) return launch_one<48, UEPI_F32, TAPS_27, 2>(tm, a, grid, smem, s);
  }
  if (wt == 2 && paired) {
    if (np == 32 && epi == UEPI_VRN) return launch_one<32, UEPI_VRN, TAPS_27_PAIRED, 2>(tm, a, grid, smem, s);   // K_b16
    if (np == 32 && epi == UEPI_F32) return launch_one<32, UEPI_F32, TAPS_27_PAIRED, 2>(tm, a, grid, smem, s);
  }
  if (wt == 4 && !paired && np == 16 && epi == UEPI_F32) return launch_one<16, UEPI_F32, TAPS_27, 4>(tm, a, grid, smem, s);   // deconv_out
  return cudaErrorNotSupported;
}

template <int NP, int E, bool PAIRED, int WT>
cudaError_t launch_stream_one(const CUtensorMap& tm, const UmmaArgs& a, int grid, size_t smem, cudaStream_t s) {
  PCGC_CARVEOUT_ONCE((conv_umma_stream_kernel<NP, E, PAIRED, WT>));
  cudaError_t e = cudaFuncSetAttribute(conv_umma_stream_kernel<NP, E, PAIRED, WT>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
  if (e != cudaSuccess) return e;
  conv_umma_stream_kernel<NP, E, PAIRED, WT><<<grid, STREAM_THREADS, smem, s>>>(tm, a);
  return cudaGetLastError();
}

// the shapes the layer programs stream (+ their float32 test forms); anything else falls back to the tile kernel
cudaError_t launch_stream(const CUtensorMap& tm, const UmmaArgs& a, int np, int epi, bool paired, int wt, int grid, size_t smem, cudaStream_t s) {
  if (!paired && wt == 1) {
    if (np == 16 && epi == UEPI_PM) return launch_stream_one<16, UEPI_PM, false, 1>(tm, a, grid, smem, s);
    if (np == 16 && epi == UEPI_F32) return launch_stream_one<16, UEPI_F32, false, 1>(tm, a, grid, smem, s);
    if (np == 32 && epi == UEPI_VRN) return launch_stream_one<32, UEPI_VRN, false, 1>(tm, a, grid, smem, s);      // K_b32
    if (np == 32 && epi == UEPI_F32) return launch_stream_one<32, UEPI_F32, false, 1>(tm, a, grid, smem, s);
    if (np == 64 && epi == UEPI_PM) return launch_stream_one<64, UEPI_PM, false, 1>(tm, a, grid, smem, s);        // deconv_in
    if (np == 64 && epi == UEPI_F32) return launch_stream_one<64, UEPI_F32, false, 1>(tm, a, grid, smem, s);
  }
  if (!paired && wt == 2) {
    if (np == 16 && epi == UEPI_PM) return launch_stream_one<16, UEPI_PM, false, 2>(tm, a, grid, smem, s);        // K_a16
    if (np == 16 && epi == UEPI_F32) return launch_stream_one<16, UEPI_F32, false, 2>(tm, a, grid, smem, s);
  }
  if (paired && wt == 2) {
    if (np == 32 && epi == UEPI_VRN) return launch_stream_one<32, UEPI_VRN, true, 2>(tm, a, grid, smem, s);       // K_b16
    if (np == 32 && epi == UEPI_F32) return launch_stream_one<32, UEPI_F32, true, 2>(tm, a, grid, smem, s);
  }
  return cudaErrorNotSupported;
}

bool stream_shape_ok(int np, int epi, bool paired, int wt) {
  if (!paired && wt == 1) return ((np == 16 || np == 64) && (epi == UEPI_PM || epi == UEPI_F32)) || (np == 32 && (epi == UEPI_VRN || epi == UEPI_F32));
  if (!paired && wt == 2) return np == 16 && (epi == UEPI_PM || epi == UEPI_F32);
  // K_b16 (Cin = 8, Voxception tail): bound by its epilogue, which 2-3 co-resident CTAs of the tile kernel serve better than the
  // 8 epilogue warps of one streaming CTA (measured r01: 0.34-0.36 ms tiled vs 0.38-0.39 ms streamed) -> only with PCGC_UMMA_STREAM=2
  if (paired && wt == 2) return umma_stream_mode() >= 2 && np == 32 && (epi == UEPI_VRN || epi == UEPI_F32);
  return false;
}

}  // namespace

int umma_stream_mode() {
  static const int m = getenv("PCGC_UMMA_STREAM") ? atoi(getenv("PCGC_UMMA_STREAM")) : 1;
  return m;
}
int umma_zband_mode() {
  static const int m = getenv("PCGC_UMMA_ZBAND") ? atoi(getenv("PCGC_UMMA_ZBAND")) : 1;
  return m && umma_stream_mode();
}

cudaError_t pack_umma_weights_dense(const float* dense, const float* bias, int cin, int n_real, UmmaWeights& out, int ntaps, int wt) {
  free_umma_weights(out);
  if (!(cin == 8 || cin == 16 || cin == 32 || cin == 64 || cin == 128 || cin == 256) || n_real < 1 || n_real > 128) return cudaErrorNotSupported;
  if (!(ntaps == 27 || (ntaps == 8 && cin >= 16))) return cudaErrorNotSupported;
  if (!(wt == 1 || ((wt == 2 || wt == 4) && ntaps == 27))) return cudaErrorNotSupported;
  // columns: n = j * npj + co  (j = output line within the band, co < n_real <= npj); np = wt * npj is a multiple of 16
  const int unit = 16 / wt;
  const int npj = (n_real + unit - 1) / unit * unit;
  const int np = wt * npj;
  if (np > 128) return cudaErrorNotSupported;
  const int kchunks = cin == 8 ? 1 : cin / 16;
  const int nt = ntaps == 8 ? 8 : 9 * (wt + 2);                 // A tiles per chunk: (kz, d, kx), d = input line offset
  const int n_mma = (ntaps == 27 && cin == 8) ? (nt + 1) / 2 : nt;
  const size_t tile = (size_t)2 * np * 16;                    // bf16 elements per B tile
  std::vector<__nv_bfloat16> p((size_t)kchunks * n_mma * tile, __float2bfloat16(0.f));
  std::vector<uint8_t> nz((size_t)kchunks * n_mma, 0);
  auto put = [&](size_t tile_idx, int n, int k, float w) {
    if (w == 0.f) return;
    const __nv_bfloat16 hi = __float2bfloat16_rn(w);
    const __nv_bfloat16 lo = __float2bfloat16_rn(w - __bfloat162float(hi));
    auto at = [&](int row) { return tile_idx * tile + (size_t)(k / 8) * (2 * np * 8) + (size_t)(row / 8) * 64 + (row % 8) * 8 + (k % 8); };
    p[at(n)] = hi;
    p[at(np + n)] = lo;
    nz[tile_idx] = 1;
  };
  // value of A tile t, input channel ci -> column (j, co)
  auto weight = [&](int t, int ci, int j, int co) -> float {
    if (ntaps == 8) return j == 0 ? dense[((size_t)t * cin + ci) * n_real + co] : 0.f;
    const int kz = t / (3 * (wt + 2)), d = (t / 3) % (wt + 2), kx = t % 3, ky = d - j;
    if (ky < 0 || ky > 2) return 0.f;
    return dense[((size_t)((kz * 3 + ky) * 3 + kx) * cin + ci) * n_real + co];
  };
  for (int ch = 0; ch < kchunks; ++ch)
    for (int m = 0; m < n_mma; ++m)
      for (int k = 0; k < 16; ++k) {
        int t, ci;
        if (ntaps == 27 && cin == 8) {
          const int ta = (nt & 1) ? (m == 0 ? 0 : 2 * m - 1) : 2 * m, tb = (nt & 1) ? (m == 0 ? -1 : 2 * m) : 2 * m + 1;
          t = k < 8 ? ta : tb; ci = k % 8;
        } else { t = m; ci = ch * 16 + k; }
        if (t < 0) continue;
        for (int j = 0; j < wt; ++j)
          for (int co = 0; co < n_real; ++co) put((size_t)ch * n_mma + m, j * npj + co, k, weight(t, ci, j, co));
      }
  cudaError_t e = cudaMalloc(&out.packed, p.size() * sizeof(__nv_bfloat16));
  if (e != cudaSuccess) return e;
  e = cudaMemcpy(out.packed, p.data(), p.size() * sizeof(__nv_bfloat16), cudaMemcpyHostToDevice);
  if (e != cudaSuccess) return e;
  if (ntaps == 27 && (cin == 8 || cin == 16 || cin == 32) && (wt == 1 || wt == 2) && (np == 16 || (np == 32 && cin != 32))) {
    // z-banded form (conv_umma_zband_kernel): ONE MMA per (d, kx) tile carries the three kz taps as column blocks, so the A tile
    // of an input slice is fetched once for the three output slices it feeds.  Rows: hi = kz*np + n, lo = 3*np + kz*np + n.
    const int nb = 3 * np, ntz = 3 * (wt + 2);
    const size_t tile3 = (size_t)2 * nb * 16;
    const int ntile = cin == 8 ? (ntz + 1) / 2 : ntz;            // cin == 8: K = 16 is a pair of tiles (tile 0 alone when odd)
    std::vector<__nv_bfloat16> pz((size_t)kchunks * ntile * tile3, __float2bfloat16(0.f));
    for (int ch = 0; ch < kchunks; ++ch)
     for (int t = 0; t < ntile; ++t)
      for (int kz = 0; kz < 3; ++kz)
        for (int k = 0; k < 16; ++k)
          for (int j = 0; j < wt; ++j)
            for (int co = 0; co < n_real; ++co) {
              int tt = t, ci = ch * 16 + k;
              if (cin == 8) {
                const int ta = (ntz & 1) ? (t == 0 ? 0 : 2 * t - 1) : 2 * t, tb = (ntz & 1) ? (t == 0 ? -1 : 2 * t) : 2 * t + 1;
                tt = k < 8 ? ta : tb; ci = k % 8;
                if (tt < 0) continue;
              }
              const float w = weight(kz * ntz + tt, ci, j, co);
              if (w == 0.f) continue;
              const __nv_bfloat16 hi = __float2bfloat16_rn(w);
              const __nv_bfloat16 lo = __float2bfloat16_rn(w - __bfloat162float(hi));
              auto at3 = [&](int row) { return (size_t)(ch * ntile + t) * tile3 + (size_t)(k / 8) * (2 * nb * 8) + (size_t)(row / 8) * 64 + (row % 8) * 8 + (k % 8); };
              pz[at3(kz * np + j * npj + co)] = hi;
              pz[at3(nb + kz * np + j * npj + co)] = lo;
            }
    cudaError_t ez = cudaMalloc(&out.packed_zb, pz.size() * sizeof(__nv_bfloat16));
    if (ez != cudaSuccess) return ez;
    ez = cudaMemcpy(out.packed_zb, pz.data(), pz.size() * sizeof(__nv_bfloat16), cudaMemcpyHostToDevice);
    if (ez != cudaSuccess) return ez;
    out.zb_bytes = (int)(pz.size() * sizeof(__nv_bfloat16));
  }
  std::vector<float> bz(np, 0.f);
  if (bias) for (int j = 0; j < wt; ++j) for (int i = 0; i < n_real; ++i) bz[j * npj + i] = bias[i];
  e = cudaMalloc((void**)&out.bias, np * sizeof(float));
  if (e != cudaSuccess) return e;
  e = cudaMemcpy(out.bias, bz.data(), np * sizeof(float), cudaMemcpyHostToDevice);
  if (e != cudaSuccess) return e;
  for (int ch = 0; ch < 16; ++ch) {
    uint32_t mask = 0;
    if (ch < kchunks && ntaps == 8)
      for (int m = 0; m < n_mma; ++m) if (nz[(size_t)ch * n_mma + m]) mask |= 1u << m;
    out.tap_mask[ch] = ntaps == 8 ? mask : 0xFFFFFFFFu;
  }
  out.cin = cin; out.n_real = n_real; out.np = np; out.npj = npj; out.wt = wt; out.n_mma = n_mma; out.kchunks = kchunks; out.ntaps = ntaps; out.ok = true;
  return cudaSuccess;
}

cudaError_t pack_umma_weights(const float* kernel, int cin, int cout, UmmaWeights& out) {
  // Keras [3,3,3,Cin,Cout] is already tap-major dense [27][cin][cout]
  return pack_umma_weights_dense(kernel, nullptr, cin, cout, out, 27, 1);
}

void free_umma_weights(UmmaWeights& w) {
  if (w.packed) cudaFree(w.packed);
  if (w.packed_zb) cudaFree(w.packed_zb);
  if (w.bias) cudaFree(w.bias);
  if (w.w23) cudaFree(w.w23);
  if (w.b23) cudaFree(w.b23);
  w = UmmaWeights();
}

cudaError_t launch_conv_umma_pm(const UmmaCall& c, const UmmaWeights& w, cudaStream_t s, int64_t* launches) {
  if (!w.ok || c.in.c != w.cin || c.in.n % (TILE_Y * w.wt) != 0) return cudaErrorNotSupported;
  const int n = c.in.n;
  UmmaArgs a;
  a.n = n; a.zt = pick_zt(n, w.np, w.cin, c.epi, w.wt, w.n_mma, w.kchunks); a.ez = a.zt + 2;
  a.cin8 = w.cin == 8; a.kchunks = w.kchunks; a.ppc = a.cin8 ? 2 : 4; a.n_mma = w.n_mma;
  a.plane_bytes = a.ez * brick_ey(w.wt) * EXC * CELL;
  a.a_bytes = a.ppc * a.plane_bytes;
  a.b_bytes = w.n_mma * 2 * w.np * 32;
  a.wpacked = (const __nv_bfloat16*)w.packed; a.bias = w.bias;
  a.n_real = w.n_real; a.flags = c.flags; a.floor_v = c.floor_v;
  a.out_f32 = c.out_f32; a.out_cs = c.out_cs; a.out_co = c.out_co;
  a.out2_f32 = c.out2_f32; a.split = c.out2_f32 ? c.split : w.n_real; a.flags2 = c.flags2;
  a.out_pm = c.out.p; a.out_planes = 2 * (c.out_s2d ? c.out.c / 8 : c.out.c) / 8;
  a.res_pm = c.res.p; a.res_planes = 2 * c.res.c / 8;
  a.w23 = w.w23; a.b23 = w.b23; a.c4 = w.c4; a.c2 = w.c2;
  a.up_ncls = w.up_ncls; a.up_cls0 = w.up_cls0; a.up_cout = w.up_cout;
  a.origin = w.origin; a.out_s2d = c.out_s2d;
  a.ff_mask = nullptr; a.ff_prev = nullptr; a.ff_src = nullptr; a.ff_list = nullptr;   // set below, on the paths that read them
  for (int i = 0; i < 16; ++i) a.tap_mask[i] = w.tap_mask[i];
  a.err = c.err;
  { static const int dbg = getenv("PCGC_UMMA_DBG") ? atoi(getenv("PCGC_UMMA_DBG")) : 0; a.dbg = dbg; }
  if (c.epi == UEPI_VRN && (!w.w23 || w.c2 + w.c4 != w.n_real || c.res.c != 2 * w.c2 || c.out.c != (c.out_s2d ? 16 : 2) * w.c2)) return cudaErrorInvalidValue;
  if (c.epi == UEPI_PM && (w.n_real % 8 != 0 || c.out.c != w.n_real || w.npj % 8 != 0)) return cudaErrorInvalidValue;
  if (c.epi == UEPI_UP && (w.up_ncls * w.up_cout != w.n_real || w.up_cout % 16 != 0 || c.out.c != w.up_cout || c.out.n != 2 * n)) return cudaErrorInvalidValue;
  const int vrn_floats = c.epi == UEPI_VRN ? w.c4 * w.c2 + w.c2 : 0;
  const int sm_count = conv_sm_count();
  const int zband = umma_zband_mode();
  // 32-column z-banded forms (K_b16, K_b32): correct (tests run them with PCGC_KB_ZBAND=1) but no faster than the tile / streaming
  // kernels they would replace (r01: K_b16 0.647 vs 0.640 ms, K_b32 0.189 vs 0.166 ms per 64 cubes) -- those layers are bound by
  // their Voxception-tail epilogue and HBM traffic, not by the MMA count -> opt-in
  static const bool kb_zband = getenv("PCGC_KB_ZBAND") && atoi(getenv("PCGC_KB_ZBAND")) != 0;
  const bool zb16 = w.np == 16 && (c.epi == UEPI_PM || c.epi == UEPI_F32 || (c.epi == UEPI_VRN && a.cin8));
  const bool zb32 = w.np == 32 && kb_zband && (c.epi == UEPI_VRN || c.epi == UEPI_F32) && ((a.cin8 && w.wt == 2) || (!a.cin8 && w.wt == 1 && w.kchunks == 1));
  if (!c.pin_tile && zband && umma_stream_mode() && w.packed_zb && n >= 32 && (zb16 || zb32)) {
    // z-banded streaming kernel (thin-N layers): the three kz taps are column blocks of one MMA
    const int z_slice_plane = brick_ey(w.wt) * EXC * CELL, z_slot = a.ppc * w.kchunks * z_slice_plane;
    const size_t fixed = (size_t)w.zb_bytes + 34 * 8 + (w.np + vrn_floats) * sizeof(float) + 16;
    const size_t budget = (size_t)220 * 1024;
    const int z_ring = (size_t)8 * z_slot + fixed <= budget ? 8 : ((size_t)4 * z_slot + fixed <= budget ? 4 : 0);
    if (z_ring) {
      a.zs = umma_zband_zs(n);                                 // enough segments per launch to balance 148 persistent CTAs
      a.slice_plane = z_slice_plane; a.slot_bytes = z_slot; a.ring = z_ring;
      a.b_bytes = w.zb_bytes;
      a.wpacked = (const __nv_bfloat16*)w.packed_zb;
      a.nacc = ZB_SLOTS; a.tmem_cols = 512; a.batch = c.in.B;
      if (c.ff_list && c.ff_list_zs == a.zs && c.epi == UEPI_PM && w.wt == 2 && n == 64) a.ff_list = c.ff_list;   // K_a16
      CUtensorMap tmz;
      cudaError_t ez = make_tmap(c.in, brick_ey(w.wt), 1, a.ppc * w.kchunks, &tmz);
      if (ez != cudaSuccess) return ez;
      const size_t smem_z = (size_t)a.ring * a.slot_bytes + fixed;
      const int segs = (n / TILE_X) * (n / (TILE_Y * w.wt)) * (n / a.zs) * c.in.B;
      const int grid_z = std::min(segs, sm_count);
      if (launches) ++*launches;
      auto go = [&](auto kern, int threads) -> cudaError_t {
        prefer_shared_carveout(kern);
        cudaError_t e2 = cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem_z);
        if (e2 != cudaSuccess) return e2;
        kern<<<grid_z, threads, smem_z, s>>>(tmz, a);
        return cudaGetLastError();
      };
      constexpr int T23 = 32 * (4 * 2 + 1 + 3), T31 = 32 * (4 * 3 + 1 + 1), T41 = 32 * (4 * 4 + 1 + 1), T21 = 32 * (4 * 2 + 1 + 1);
      if (zb32) {
        if (a.cin8)                                            // K_b16: paired taps, y-band 2, Voxception tail: 4 epilogue groups + 1 issuer
          return c.epi == UEPI_VRN ? go(conv_umma_zband_kernel<32, UEPI_VRN, 2, true, 4, 1>, T41) : go(conv_umma_zband_kernel<32, UEPI_F32, 2, true, 4, 1>, T41);
        return c.epi == UEPI_VRN ? go(conv_umma_zband_kernel<32, UEPI_VRN, 1, false, 2, 1>, T21) : go(conv_umma_zband_kernel<32, UEPI_F32, 1, false, 2, 1>, T21);   // K_b32
      }
      if (a.cin8) {                                            // Cin = 8, 16 columns: paired taps, 3 epilogue groups + 1 issuer
        if (w.wt != 1) return cudaErrorNotSupported;
        return c.epi == UEPI_VRN ? go(conv_umma_zband_kernel<16, UEPI_VRN, 1, true, 3, 1>, T31) : go(conv_umma_zband_kernel<16, UEPI_F32, 1, true, 3, 1>, T31);
      }
      if (w.wt == 2) return c.epi == UEPI_PM ? go(conv_umma_zband_kernel<16, UEPI_PM, 2, false, 2, 3>, T23) : go(conv_umma_zband_kernel<16, UEPI_F32, 2, false, 2, 3>, T23);
      return c.epi == UEPI_PM ? go(conv_umma_zband_kernel<16, UEPI_PM, 1, false, 2, 3>, T23) : go(conv_umma_zband_kernel<16, UEPI_F32, 1, false, 2, 3>, T23);
    }
  }
  if (!c.pin_tile && umma_stream_mode() && w.ntaps == 27 && w.kchunks == 1 && n >= 16 && stream_shape_ok(w.np, c.epi, a.cin8 != 0, w.wt)) {
    // z-streaming kernel: one CTA per SM, ring of input slices, rotating accumulators
    static const int zs_env = getenv("PCGC_STREAM_ZS") ? atoi(getenv("PCGC_STREAM_ZS")) : 16;
    static const int ring_env = getenv("PCGC_STREAM_RING") ? atoi(getenv("PCGC_STREAM_RING")) : 0;
    static const int ctas_env = getenv("PCGC_STREAM_CTAS") ? atoi(getenv("PCGC_STREAM_CTAS")) : 1;
    a.zs = std::min(n, std::max(1, zs_env));
    while (n % a.zs) --a.zs;
    // small grids (16^3: deconv_in, the hyper nets): a 16-slice segment leaves 2 segments per cube -- fewer than the 148 persistent
    // CTAs at 64 cubes per launch.  Shorter segments re-read two halo slices each but fill the machine (r02: deconv_in ran at
    // 16 TFLOP/s where the same kernel reaches 100+ on the larger grids).
    if (!getenv("PCGC_STREAM_ZS"))
      while (a.zs > 4 && (n / TILE_X) * (n / (TILE_Y * w.wt)) * (n / a.zs) * c.in.B < 2 * sm_count && n % (a.zs / 2) == 0) a.zs /= 2;
    a.slice_plane = brick_ey(w.wt) * EXC * CELL;
    a.slot_bytes = a.ppc * a.slice_plane;
    const int per_sm = 1;
    (void)ctas_env;
    const size_t fixed = (size_t)a.b_bytes + 34 * 8 + (w.np + vrn_floats) * sizeof(float) + 16;
    const size_t budget = (size_t)220 * 1024;
    int ring = (size_t)8 * a.slot_bytes + fixed <= budget ? 8 : ((size_t)4 * a.slot_bytes + fixed <= budget ? 4 : 0);
    if (ring_env == 4 && ring == 8) ring = 4;
    const int nacc = w.np <= 32 ? 8 : 4;
    if (ring >= 4 && nacc >= 2) {
      a.ring = ring; a.nacc = nacc;
      int cols = 32; while (cols < nacc * 2 * w.np) cols *= 2;
      a.tmem_cols = cols;
      a.batch = c.in.B;
      CUtensorMap tms;
      cudaError_t es = make_tmap(c.in, brick_ey(w.wt), 1, a.ppc, &tms);
      if (es != cudaSuccess) return es;
      const size_t smem_s = (size_t)ring * a.slot_bytes + fixed;
      const int segs = (n / TILE_X) * (n / (TILE_Y * w.wt)) * (n / a.zs) * c.in.B;
      if (launches) ++*launches;
      return launch_stream(tms, a, w.np, c.epi, a.cin8 != 0, w.wt, std::min(segs, sm_count * per_sm), smem_s, s);
    }
  }
  CUtensorMap tm;
  cudaError_t e = make_tmap(c.in, brick_ey(w.wt), a.ez, a.ppc, &tm);
  if (e != cudaSuccess) return e;
  const size_t smem = (size_t)a.a_bytes + a.b_bytes + (6 + 2 * MAX_ZT) * 8 + (w.np + vrn_floats) * sizeof(float) + 16;
  const int tiles = (n / TILE_X) * (n / (TILE_Y * w.wt)) * (n / a.zt) * c.in.B;
  a.batch = c.in.B;
  // persistent grid: as many CTAs as fit (shared memory / TMEM columns), each walks tiles with stride gridDim.x.
  // Two accumulator sets (MMAs of tile i+1 overlap the epilogue of tile i) when the 512 TMEM columns allow it.
  int per_sm = std::max(1, std::min((int)(227 * 1024 / (smem + 1024)), 3));
  auto pow2 = [](int v) { int c = 32; while (c < v) c *= 2; return c; };
  a.nsets = pow2(2 * a.zt * 2 * w.np) * per_sm <= 512 ? 2 : 1;
  const int cols = pow2(a.nsets * a.zt * 2 * w.np);
  a.tmem_cols = cols;
  per_sm = std::max(1, std::min(per_sm, 512 / cols));
  const int sms = conv_sm_count();
  static const int persist = getenv("PCGC_UMMA_PERSIST") ? atoi(getenv("PCGC_UMMA_PERSIST")) : 1;  // 0: one tile per CTA
  const int grid = persist ? std::min(tiles, sms * per_sm) : tiles;
  if (launches) ++*launches;
  if (c.ff_mask && c.ff_src && c.epi == UEPI_VRN && w.wt == 2 && n == 64) {
    a.ff_mask = c.ff_mask; a.ff_prev = c.ff_prev; a.ff_src = c.ff_src;
    if (c.ff_list && c.ff_list_zs == a.zt) a.ff_list = c.ff_list;
  }
  if (w.wt > 1) return launch_banded(tm, a, w.np, c.epi, a.cin8 != 0, w.wt, grid, smem, s);
  if (c.epi == UEPI_UP) {
    if (w.ntaps != 8 || w.np != 128) return cudaErrorNotSupported;
    return launch_one<128, UEPI_UP, TAPS_8, 1>(tm, a, grid, smem, s);
  }
  if (w.ntaps == 8) {                                   // stride-2 conv on a space-to-depth input
    if (c.epi != UEPI_PM) return cudaErrorNotSupported;
    if (w.np == 32) return launch_one<32, UEPI_PM, TAPS_8, 1>(tm, a, grid, smem, s);
    if (w.np == 64) return launch_one<64, UEPI_PM, TAPS_8, 1>(tm, a, grid, smem, s);
    return cudaErrorNotSupported;
  }
  if (w.ntaps != 27) return cudaErrorNotSupported;
  if (a.cin8) {
    if (w.np != 16) return cudaErrorNotSupported;
    return launch_np<16, TAPS_27_PAIRED>(tm, a, c.epi, grid, smem, s);
  }
  switch (w.np) {
    case 16: return launch_np<16, TAPS_27>(tm, a, c.epi, grid, smem, s);
    case 32: return launch_np<32, TAPS_27>(tm, a, c.epi, grid, smem, s);
    case 48: return launch_np<48, TAPS_27>(tm, a, c.epi, grid, smem, s);
    case 64: return launch_np<64, TAPS_27>(tm, a, c.epi, grid, smem, s);
  }
  return cudaErrorNotSupported;
}

// ---------------------------------------------------------------------------------------------- far-field classification
// Kernel 1: one thread per row (b, z, y): the 64 occupancy bytes -> a 64-bit mask, dilated along x by r = 1 .. FF_LAYERS (shifts drop what
// leaves the cube, like the zero padding) and collapsed to one bit per 8-voxel x tile.
__global__ void __launch_bounds__(256) ff_row_mask_kernel(const uint8_t* __restrict__ cubes, int rows, uint8_t* __restrict__ row_mask) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= rows) return;
  const uint4* src = reinterpret_cast<const uint4*>(cubes + (size_t)i * 64);
  uint64_t m = 0;
#pragma unroll
  for (int q = 0; q < 4; ++q) {
    const uint4 v = __ldg(src + q);
    const uint32_t w[4] = {v.x, v.y, v.z, v.w};
#pragma unroll
    for (int k = 0; k < 4; ++k)
#pragma unroll
      for (int bb = 0; bb < 4; ++bb)
        if ((w[k] >> (8 * bb)) & 0xFFu) m |= 1ull << (q * 16 + k * 4 + bb);
  }
  uint64_t d = m;
#pragma unroll
  for (int k = 0; k < FF_LAYERS; ++k) {
    d |= (d << 1) | (d >> 1);                                      // one more voxel of dilation per layer
    uint32_t t = 0;
#pragma unroll
    for (int bx = 0; bx < 8; ++bx) t |= ((d >> (8 * bx)) & 0xFFull) ? (1u << bx) : 0u;
    row_mask[(size_t)k * rows + i] = (uint8_t)t;
  }
}
// Kernel 2: one thread per (k, b, z, by): OR of the row masks over z +- r and the tile's 32 lines +- r.
__global__ void __launch_bounds__(128) ff_tile_mask_kernel(const uint8_t* __restrict__ row_mask, int nb, size_t layer_stride, uint8_t* __restrict__ ff_mask) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  const int per = nb * 128;
  if (i >= FF_LAYERS * per) return;
  const int k = i / per, j = i - k * per;
  const int by = j & 1, z = (j >> 1) & 63, b = j >> 7;
  const int r = k + 1;
  const uint8_t* rm = row_mask + (size_t)k * nb * 4096 + (size_t)b * 4096;
  const int z0 = max(z - r, 0), z1 = min(z + r, 63), y0 = max(32 * by - r, 0), y1 = min(32 * by + 31 + r, 63);
  uint32_t t = 0;
  for (int zz = z0; zz <= z1; ++zz)
    for (int yy = y0; yy <= y1; ++yy) t |= rm[zz * 64 + yy];
  ff_mask[(size_t)k * layer_stride + j] = (uint8_t)t;
}

cudaError_t launch_ff_classify(const uint8_t* cubes, int nb, uint8_t* row_mask, uint8_t* ff_mask, size_t layer_stride, cudaStream_t s, int64_t* launches) {
  if (nb <= 0) return cudaSuccess;
  PCGC_CARVEOUT_ONCE(ff_row_mask_kernel); PCGC_CARVEOUT_ONCE(ff_tile_mask_kernel);
  const int rows = nb * 4096;
  ff_row_mask_kernel<<<(rows + 255) / 256, 256, 0, s>>>(cubes, rows, row_mask);
  ff_tile_mask_kernel<<<(FF_LAYERS * nb * 128 + 127) / 128, 128, 0, s>>>(row_mask, nb, layer_stride, ff_mask);
  if (launches) *launches += 2;
  return cudaGetLastError();
}

// Kernel 3 (launch_ff_list): one CTA per list.  Unit u = ((b*(64/zs) + bz)*2 + by)*8 + bx (zs slices of an 8 x 32-voxel tile, the kernels'
// tile / segment numbering) is listed when any of its slices is set in mask | prev; ordered compaction, list[0] = count.
__global__ void __launch_bounds__(1024) ff_list_kernel(FfListJob jobs, int nb) {
  const FfListJob::One& j = jobs.l[blockIdx.x];
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const int tz_n = 64 / j.zs, units = nb * tz_n * 16;
  __shared__ int s_warp[32];
  __shared__ int s_base;
  if (tid == 0) s_base = 0;
  __syncthreads();
  for (int c0 = 0; c0 < units; c0 += 1024) {
    const int u = c0 + tid;
    bool act = false;
    if (u < units) {
      const int bx = u & 7, by = (u >> 3) & 1, bz = (u >> 4) % tz_n, b = (u >> 4) / tz_n;
      const size_t o = ((size_t)b * 64 + bz * j.zs) * 2 + by;
      uint32_t t = 0;
      for (int zi = 0; zi < j.zs; ++zi) t |= j.mask[o + 2 * zi] | j.prev[o + 2 * zi];
      act = (t >> bx) & 1u;
    }
    const uint32_t bal = __ballot_sync(0xFFFFFFFFu, act);
    if (lane == 0) s_warp[warp] = __popc(bal);
    __syncthreads();
    if (warp == 0) {
      const int v = s_warp[lane];
      int inc = v;
#pragma unroll
      for (int d = 1; d < 32; d <<= 1) { const int t2 = __shfl_up_sync(0xFFFFFFFFu, inc, d); if (lane >= d) inc += t2; }
      s_warp[lane] = inc - v;                                      // exclusive prefix of the warp counts
    }
    __syncthreads();
    if (act) j.list[1 + s_base + s_warp[warp] + __popc(bal & ((1u << lane) - 1u))] = u;
    __syncthreads();
    if (tid == 1023) s_base += s_warp[31] + __popc(bal);           // the last warp's prefix + its count
    __syncthreads();
  }
  if (tid == 0) j.list[0] = s_base;
}

cudaError_t launch_ff_list(const FfListJob& jobs, int n_jobs, int nb, cudaStream_t s, int64_t* launches) {
  if (nb <= 0 || n_jobs <= 0) return cudaSuccess;
  if (n_jobs > FfListJob::MAX) return cudaErrorInvalidValue;
  for (int i = 0; i < n_jobs; ++i) if (jobs.l[i].zs < 1 || 64 % jobs.l[i].zs) return cudaErrorInvalidValue;
  PCGC_CARVEOUT_ONCE(ff_list_kernel);
  ff_list_kernel<<<n_jobs, 1024, 0, s>>>(jobs, nb);
  if (launches) ++*launches;
  return cudaGetLastError();
}

int umma_tile_zt(const UmmaWeights& w, int n, int epi) { return pick_zt(n, w.np, w.cin, epi, w.wt, w.n_mma, w.kchunks); }
int umma_zband_zs(int n) { return n >= 64 ? 16 : 8; }

// ---------------------------------------------------------------------------------------------- format converters
__global__ void f32_to_pm_kernel(const float* __restrict__ in, int in_cs, int in_co, __nv_bfloat16* __restrict__ out,
                                 int c8n, size_t vox_per_cube, size_t total) {
  for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (size_t)gridDim.x * blockDim.x) {
    const size_t vox = i % vox_per_cube;
    const size_t r = i / vox_per_cube;
    const int c8 = (int)(r % c8n);
    const size_t b = r / c8n;
    const float* ip = in + (b * vox_per_cube + vox) * in_cs + in_co + c8 * 8;
    float v[8];
#pragma unroll
    for (int k = 0; k < 8; ++k) v[k] = __ldg(ip + k);
    __nv_bfloat16* ob = out + ((b * (2 * c8n) + 2 * c8) * vox_per_cube + vox) * 8;
    split_store(ob, ob + vox_per_cube * 8, v);
  }
}

__global__ void pm_to_f32_kernel(const __nv_bfloat16* __restrict__ in, int c8n, float* __restrict__ out, int out_cs,
                                 int out_co, size_t vox_per_cube, size_t total) {
  for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (size_t)gridDim.x * blockDim.x) {
    const size_t vox = i % vox_per_cube;
    const size_t r = i / vox_per_cube;
    const int c8 = (int)(r % c8n);
    const size_t b = r / c8n;
    const __nv_bfloat16* ib = in + ((b * (2 * c8n) + 2 * c8) * vox_per_cube + vox) * 8;
    float v[8];
    load_cell_sum(ib, ib + vox_per_cube * 8, v);
    float* op = out + (b * vox_per_cube + vox) * out_cs + out_co + c8 * 8;
#pragma unroll
    for (int k = 0; k < 8; ++k) op[k] = v[k];
  }
}

cudaError_t launch_f32_to_pm(const float* in, int in_cs, int in_co, const PmTensor& out, cudaStream_t s, int64_t* launches) {
  const size_t vox = (size_t)out.n * out.n * out.n;
  const size_t total = vox * (out.c / 8) * out.B;
  const int blocks = (int)std::min<size_t>((total + 255) / 256, 148 * 16);
  PCGC_CARVEOUT_ONCE(f32_to_pm_kernel);
  f32_to_pm_kernel<<<blocks, 256, 0, s>>>(in, in_cs, in_co, out.p, out.c / 8, vox, total);
  if (launches) ++*launches;
  return cudaGetLastError();
}

cudaError_t launch_pm_to_f32(const PmTensor& in, float* out, int out_cs, int out_co, cudaStream_t s, int64_t* launches) {
  const size_t vox = (size_t)in.n * in.n * in.n;
  const size_t total = vox * (in.c / 8) * in.B;
  const int blocks = (int)std::min<size_t>((total + 255) / 256, 148 * 16);
  PCGC_CARVEOUT_ONCE(pm_to_f32_kernel);
  pm_to_f32_kernel<<<blocks, 256, 0, s>>>(in.p, in.c / 8, out, out_cs, out_co, vox, total);
  if (launches) ++*launches;
  return cudaGetLastError();
}

cudaError_t launch_conv_umma(const ConvCall&, const UmmaWeights&, cudaStream_t, int64_t*) { return cudaErrorNotSupported; }

}  // namespace pcgc
