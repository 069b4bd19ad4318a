// tcgen05 (UMMA) implicit-GEMM convolution engine: interface.  See umma_conv.cu for the design.
#pragma once
#include <cuda_bf16.h>

#include "common.cuh"

namespace pcgc {

// Activation format of the tcgen05 engine ("PM": plane-major split-bf16):
//   bf16 [B][P = 2*C/8][n][n][n][8]   plane p = (c/8)*2 + hl,  hl = 0: hi = bf16(v), 1: lo = bf16(v - hi)
// Every 16-byte cell holds 8 consecutive channels of one voxel; the x-run of a plane is contiguous,
// so a TMA box lands in shared memory exactly in the no-swizzle K-major core-matrix layout.
struct PmTensor {
  __nv_bfloat16* p = nullptr;
  int n = 0, c = 0, B = 0;       // grid edge, channels (multiple of 8), batch
  size_t plane_elems() const { return (size_t)n * n * n * 8; }
  size_t cube_elems() const { return plane_elems() * (size_t)(2 * c / 8); }
};

enum UmmaEpilogue : int {
  UEPI_F32 = 0,     // +bias, [relu|abs|floor] -> float32 NDHWC (external outputs: y, logits)
  UEPI_PM = 1,      // +bias, relu -> PM
  UEPI_VRN = 2,     // VRN tail: t12 | t22 -> t23 = relu(W23^T t22 + b23); out = relu(x + [t12|t23]) -> PM
  UEPI_UP = 3       // stride-2 Conv3DTranspose: 8 output-parity classes as column blocks, +bias, relu -> PM on the 2n grid
};

struct UmmaWeights {
  bool ok = false;
  int cin = 0;              // K per tap as the kernel sees it (8, 16, 32, 64)
  int n_real = 0;           // real output columns
  int np = 0;               // accumulator columns per pass: wt * npj, a multiple of 16
  int wt = 1;               // y-band width: each M row produces wt consecutive output lines (columns (j, channel))
  int npj = 0;              // columns per output line (n_real padded so that wt*npj % 16 == 0)
  int n_mma = 0;            // MMA pairs per z-slice per 16-channel chunk (27, 14 for cin == 8, 8 for transposed conv)
  int ntaps = 27;           // 27 (3x3x3) or 8 ({t-1,t}^3 window of a stride-2 transposed conv)
  int up_ncls = 0, up_cls0 = 0, up_cout = 0;   // UEPI_UP column layout
  int origin = -1;          // brick origin vs tile origin: -1 (taps reach t-1) or 0 (stride-2 conv on a space-to-depth input)
  uint32_t tap_mask[16] = {0};   // per K chunk: taps whose weight tile is non-zero
  int kchunks = 0;
  void* packed = nullptr;   // device bf16: [kchunk][n_mma][2*np x 16] canonical no-swizzle K-major tiles
  float* bias = nullptr;    // device [np] (zero padded)
  void* packed_zb = nullptr;   // device bf16, z-banded form (cin 16, wt 2, np 16 only): [12 (d,kx) tiles][2*48 x 16], columns (kz, j, channel)
  int zb_bytes = 0;
  // VRN tail (UEPI_VRN): conv2_3 1x1x1 weights [c4][c2] and bias [c2]
  float* w23 = nullptr; float* b23 = nullptr; int c4 = 0, c2 = 0;
};

// dense: HOST float32 [27][cin][n_real] (tap-major, any zero structure already applied), bias [n_real] or null.
cudaError_t pack_umma_weights_dense(const float* dense, const float* bias, int cin, int n_real, UmmaWeights& out, int ntaps = 27, int wt = 1);
// Compatibility shim used by pcgc_load_conv (single plain layer, Keras [3,3,3,Cin,Cout]).
cudaError_t pack_umma_weights(const float* kernel, int cin, int cout, UmmaWeights& out);
void free_umma_weights(UmmaWeights& w);

struct UmmaCall {
  PmTensor in;                 // input activations
  int epi = UEPI_F32;
  int flags = 0; float floor_v = 0.f;
  float* out_f32 = nullptr; int out_cs = 0, out_co = 0;     // UEPI_F32
  float* out2_f32 = nullptr; int split = 0, flags2 = 0;     // UEPI_F32: second output for columns >= split (two-headed layers)
  PmTensor out;                // UEPI_PM / UEPI_VRN
  PmTensor res;                // UEPI_VRN: the block input x
  int out_s2d = 0;             // UEPI_VRN: write `out` space-to-depth (out = the n/2-grid, 8*C-channel tensor)
  int* err = nullptr;          // device int, set on device-side timeouts
  // far-field tiles of the analysis 64^3 stage (y-band 2): masks from launch_ff_classify for the output layer's radius, of the current
  // cubes (ff_mask) and of the cubes the output slots held before (ff_prev); the layer's output for the all-zero cube (ff_src).  Read by
  // the tile kernel's UEPI_VRN form (K_b16); the z-banded kernel's UEPI_PM form (K_a16) reads only ff_list.  See UmmaArgs::ff_mask.
  // Ignored (every tile computed) by the other kernel forms.
  const uint8_t* ff_mask = nullptr; const uint8_t* ff_prev = nullptr; const __nv_bfloat16* ff_src = nullptr;
  // the units to compute or restore (launch_ff_list, built with zs = ff_list_zs slices per unit); used only where ff_list_zs is the
  // kernel's own z extent (umma_tile_zt / umma_zband_zs), otherwise every unit is visited
  const int* ff_list = nullptr; int ff_list_zs = 0;
  bool pin_tile = false;       // always the tile kernel, whatever PCGC_UMMA_STREAM / PCGC_UMMA_ZBAND / PCGC_KB_ZBAND say: the hyper
                               // decoder's loc / scale must have the same bits in the encoding and the decoding process
};

cudaError_t launch_conv_umma_pm(const UmmaCall& c, const UmmaWeights& w, cudaStream_t s, int64_t* launches);
// PCGC_UMMA_STREAM: 0 = tile kernel everywhere, 1 = z-streaming kernel for the shapes it covers (umma_conv.cu)
int umma_stream_mode();
// PCGC_UMMA_ZBAND (default 1, needs streaming): z-banded kernel for the NP = 16 layers (K_a16, K_a32, K_b16, deconv_out)
int umma_zband_mode();
// Far-field classification of a batch of uint8 occupancy cubes [nb][64][64][64] for the seven layers of the analysis 64^3 stage (conv_in
// output, then K_a and K_b of the three VRN-16 blocks: receptive-field radii 1 .. 7 voxels): ff_mask[k * layer_stride + (b*64 + z)*2 + by]
// bit bx = 1 when an occupied voxel lies within radius k + 1 of the 8 (x) x 32 (y) voxels of tile (by, bx) in slice z.
// row_mask: scratch [FF_LAYERS][nb*4096] bytes; layer_stride >= nb*128.
constexpr int FF_LAYERS = 7;
cudaError_t launch_ff_classify(const uint8_t* cubes, int nb, uint8_t* row_mask, uint8_t* ff_mask, size_t layer_stride, cudaStream_t s, int64_t* launches);
// Work lists of the far-field kernels, one per job: the units (zs slices of an 8 x 32-voxel tile, numbered ((b*(64/zs) + bz)*2 + by)*8 + bx)
// with a bit set in mask | prev, in increasing order: list = {count, units...}, room for nb*(64/zs)*16 + 1 ints.  One launch for all jobs.
struct FfListJob {
  static constexpr int MAX = 8;
  struct One { const uint8_t* mask; const uint8_t* prev; int* list; int zs; } l[MAX];
};
cudaError_t launch_ff_list(const FfListJob& jobs, int n_jobs, int nb, cudaStream_t s, int64_t* launches);
// z extent of a launch: slices per tile of the tile kernel, per segment of the z-banded kernel
int umma_tile_zt(const UmmaWeights& w, int n, int epi);
int umma_zband_zs(int n);
// float32 NDHWC (channel stride/offset) <-> PM
cudaError_t launch_f32_to_pm(const float* in, int in_cs, int in_co, const PmTensor& out, cudaStream_t s, int64_t* launches);
cudaError_t launch_pm_to_f32(const PmTensor& in, float* out, int out_cs, int out_co, cudaStream_t s, int64_t* launches);

// legacy hook kept for api.cu's generic path
cudaError_t launch_conv_umma(const ConvCall& c, const UmmaWeights& w, cudaStream_t s, int64_t* launches);

}  // namespace pcgc
