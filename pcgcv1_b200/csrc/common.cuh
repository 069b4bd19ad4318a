// Internal definitions shared by the translation units of libpcgc_b200.so (sm_100a only).
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>
#include <stdlib.h>
#include <string>
#include <vector>
#include <map>

#include "../../include/pcgc_b200.h"

namespace pcgc {

// Every kernel of the library asks for the SAME shared-memory / L1 carveout (all shared).  The carveout is per-SM state: a CTA
// whose kernel prefers another split cannot be placed on an SM until the CTAs resident there have drained, so the coder-stream
// kernels (tiny, latency-bound) would serialise with the persistent conv kernels of the main stream instead of running beside
// them (measured r02: the 0.05 ms first kernel of the hyper decoder waited 2-3 ms behind the range encoder).
template <typename K>
inline void prefer_shared_carveout(K kernel) {
  cudaFuncSetAttribute(kernel, cudaFuncAttributePreferredSharedMemoryCarveout, cudaSharedmemCarveoutMaxShared);
}
#define PCGC_CARVEOUT_ONCE(kernel)                                            \
  do {                                                                        \
    static const bool once_ = (::pcgc::prefer_shared_carveout(kernel), true); \
    (void)once_;                                                              \
  } while (0)

// SMs the persistent conv kernels size their grids for: the device's SM count.
inline int conv_sm_count() {
  static const int n = [] {
    int d = 0, v = 148;
    cudaGetDevice(&d);
    cudaDeviceGetAttribute(&v, cudaDevAttrMultiProcessorCount, d);
    return v;
  }();
  return n;
}

// One convolution as the kernels see it: a stride-S "gather" convolution over an input grid with
// a (KZ,KY,KX) tap box.  Forward Conv3D layers map 1:1; a stride-2 Conv3DTranspose is split into
// 8 output-parity classes, each of which is such a convolution over the INPUT grid whose outputs
// interleave (out index = t*ostride + ooff).  No atomics, fixed summation order => deterministic.
struct ConvDesc {
  int kz, ky, kx;        // tap box
  int stride;            // input step per output step (1 or 2)
  int pz, py, px;        // pad-before per axis: in = t*stride - p + tap
  int ostride;           // output interleave (1; 2 for transposed-conv parity classes)
  int oz, oy, ox;        // output offset per axis (parity class)
  int cin, cout;
  const float* w = nullptr;   // device, [KY][KX][Cin][KZ][Cout] fp32
  // class_mode: the 8 "output channels" are the 8 output-parity classes of a single-channel stride-2 transposed conv sharing one
  // union tap box; class q = (rz<<2)|(ry<<1)|rx writes output voxel 2t + cls_o0[r] per axis (channel 0, bias[0]).
  int class_mode = 0;
  int cls_o0[2] = {0, 0};
};

enum EpilogueFlags : int { EPI_RELU = 1, EPI_ABS = 2, EPI_RES = 4, EPI_FLOOR = 8 };

struct ConvCall {
  ConvDesc d;
  const float* in;  int in_n;  int in_cs;  int in_co;     // input grid edge, channel stride/offset
  float* out;       int out_n; int out_cs; int out_co;    // full output grid edge, channel stride/offset
  int tn;                                                 // extent of the t grid (outputs per axis per class)
  const float* bias;                                      // [Cout] or null
  const float* res; int res_cs; int res_co;               // residual (same grid as out) or null
  int flags; float floor_v;
  int B;
  // optional "PM" split-bf16 plane-major tensors (umma_conv.cuh) instead of the float32 NDHWC in/out
  const void* in_pm = nullptr;    // bf16 [B][2*cin/8][in_n^3][8]
  void* out_pm = nullptr;         // bf16 [B][2*cout/8][out_n^3][8]
};

cudaError_t launch_conv_ffma(const ConvCall& c, cudaStream_t s, int64_t* launches);
// ff_mask / ff_prev (uint8 cubes only, or both nullptr): far-field masks of radius 1 (umma_conv.cuh launch_ff_classify) of these cubes
// and of the cubes the output slots held before; voxels clear in both keep the empty cube's values already in out_pm and are not stored.
cudaError_t launch_conv_in_pm(const void* cubes, int dtype, const float* w_host, const float* bias_host, void* out_pm, int B,
                              const uint8_t* ff_mask, const uint8_t* ff_prev, cudaStream_t s, int64_t* launches);
cudaError_t launch_u8_to_f32(const void* in, int dtype, float* out, int64_t n, cudaStream_t s, int64_t* launches);

// entropy.cu
struct BottleneckDev {
  int channels = 0;
  float* params = nullptr;   // device: per channel 58 floats, see entropy.cu
};
cudaError_t launch_factorized(const BottleneckDev& bn, const float* x, int64_t n_vox, int C, float bound,
                              float* x_hat, float* p, double* bits, int32_t* minmax, double* scratch,
                              cudaStream_t s, int64_t* launches, int noise = 0, uint64_t seed = 0);
cudaError_t launch_factorized_pmf(const BottleneckDev& bn, int min_v, int max_v, float bound, float* pmf,
                                  cudaStream_t s, int64_t* launches);
cudaError_t launch_laplace(const float* y, const float* loc, const float* scale, int B, int64_t E, float bound,
                           float* y_hat, float* p, double* bits, int32_t* minmax, double* scratch,
                           cudaStream_t s, int64_t* launches, int noise = 0, uint64_t seed = 0);
cudaError_t launch_widen_minmax(int32_t* minmax, int n_pairs, cudaStream_t s, int64_t* launches);
cudaError_t launch_laplace_intervals(const float* y_hat, const float* loc, const float* scale, int B, int64_t E,
                                     const int32_t* minmax, float bound, int precision, uint32_t* intervals,
                                     int* err_flag, cudaStream_t s, int64_t* launches);
cudaError_t launch_laplace_cdf(const float* loc, const float* scale, int B, int64_t E, const int32_t* minmax_dev,
                               const int64_t* row_offset_dev, float bound, int precision, uint16_t* cdf,
                               int* err_flag, cudaStream_t s, int64_t* launches);
cudaError_t launch_debug_quantize_pmf(const float* pmf, int64_t rows, const int32_t* minmax_dev, int precision,
                                      int32_t* cdf32, int* err_flag, cudaStream_t s, int64_t* launches);
// api.cu: what train.cu may touch of a ctx
cudaStream_t ctx_stream(pcgc_ctx* c);
int64_t* ctx_launches(pcgc_ctx* c);
int ctx_device(pcgc_ctx* c);
int* ctx_err_flag(pcgc_ctx* c);
int ctx_fail(pcgc_ctx* c, int code, const char* msg);
float* ctx_workspace(pcgc_ctx* c, int slot, size_t floats);
void ctx_prof_begin(pcgc_ctx* c, const char* tag, double flops, double bytes);
void ctx_prof_end(pcgc_ctx* c);

// gpu_coder.cu
cudaError_t launch_range_encode_intervals(const uint32_t* iv, int B, int64_t E, int precision, uint8_t* scratch, int64_t stride,
                                          int64_t* lens, uint8_t* packed, int64_t cap, int64_t* offsets, int* err,
                                          cudaStream_t s, int64_t* launches);
cudaError_t launch_range_decode_rows(const uint8_t* packed, const int64_t* offsets, int B, int64_t E, const uint16_t* rows,
                                     const int64_t* row_offset, const int32_t* minmax, int max_n, int precision, float* y_hat, int* err,
                                     cudaStream_t s, int64_t* launches);
// topk.cu
cudaError_t launch_topk(const float* logits, int B, int64_t V, const int32_t* ks, uint8_t* mask, float* thres,
                        int32_t* count, int* err_flag, cudaStream_t s, int64_t* launches);
cudaError_t launch_threshold(const float* logits, int B, int64_t V, float thres, uint8_t* mask, int32_t* count,
                             cudaStream_t s, int64_t* launches);

// voxelize.cu
cudaError_t launch_voxelize(const int16_t* local, const int64_t* offsets, int B, int S, int64_t n, uint8_t* cubes, int* err,
                            cudaStream_t s, int64_t* launches);
cudaError_t launch_extract_points(const uint8_t* mask, int B, int S, int64_t* chunk_ws, int32_t* counts, int16_t* points, int64_t cap,
                                  int64_t* total, cudaStream_t s, int64_t* launches);

// metrics.cu: nearest-neighbour geometry sums with a per-ctx workspace (grown on demand, freed with the ctx)
struct GeoWorkspace;
// the grids of A and B (sized for na / nb points; the workspace is reused by the next launch_geometry_queries) ...
cudaError_t launch_geometry_grids(GeoWorkspace** ws, const double* a, int64_t na, const double* b, int64_t nb, cudaStream_t s,
                                  int64_t* launches);
// ... then both directions' nearest-neighbour queries and the sums into out double[8]
cudaError_t launch_geometry_queries(GeoWorkspace* ws, const double* a, const double* b, const double* normals_a, double* out, cudaStream_t s,
                                    int64_t* launches);
void free_geometry_workspace(GeoWorkspace* ws);
// k-nearest-neighbour PCA normals of one set, in the same workspace: its grid ...
cudaError_t launch_normals_grid(GeoWorkspace** ws, const double* p, int64_t n, cudaStream_t s, int64_t* launches);
// ... then per point the k nearest (d2, index), the covariance and its smallest eigenvector (knn may be null)
cudaError_t launch_normals_query(GeoWorkspace* ws, const double* p, int64_t n, int k, double* normals, int32_t* knn, cudaStream_t s,
                                 int64_t* launches);

// meshsample.cu: the per-ctx workspace of pcgc_mesh_sample (grown on demand, freed with the ctx)
struct MeshWorkspace;
MeshWorkspace** ctx_mesh_workspace(pcgc_ctx* c);
void free_mesh_workspace(MeshWorkspace* ws);

}  // namespace pcgc
