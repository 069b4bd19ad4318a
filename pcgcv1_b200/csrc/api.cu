// C ABI of libpcgc_b200.so: context, weights, the per-net layer programs and the entry points
// declared in include/pcgc_b200.h.  Layer tables restate models/model_voxception.py:21-54,83-122,
// 153-192,224-244,263-297 and models/model_simple.py:21-42,58-86 (names = the Keras name= args).
#include <math.h>
#include <stdarg.h>
#include <stdio.h>
#include <string.h>
#include <stdlib.h>

#include <algorithm>
#include <string>
#include <vector>

#include "common.cuh"
#include "det_math.h"
#include "umma_conv.cuh"
#include "umma_win.cuh"

using namespace pcgc;

namespace {

struct LayerSpec {
  std::string name;
  int cin, cout, k, stride;
  bool transposed, bias, relu;
};

enum Buf { BUF_IN = 0, BUF_X0, BUF_A, BUF_B, BUF_T1, BUF_T2, BUF_OUT0, BUF_OUT1, BUF_COUNT };

struct Op {
  int layer;
  int in, in_n, in_cs, in_co;
  int out, out_cs, out_co;
  int res, res_cs, res_co;      // res < 0: none
  int flags;
};

struct LayerW {
  bool loaded = false;
  int n_classes = 0;
  ConvDesc cls[8];
  float* bias = nullptr;
  UmmaWeights umma;             // (unused by the generic path)
  std::vector<float> hk, hb;    // host copies (Keras layout) used to build the fused tcgen05 weights
};

// Fused tcgen05 program of one voxception transform: per VRN block two kernels
//   K_a: [conv1_1 | conv2_1@centre tap]            C   -> C/2   (+bias, ReLU)
//   K_b: blockdiag[conv1_2, conv2_2] + VRN tail    C/2 -> C     (conv2_3 1x1x1, concat, residual, ReLU in the epilogue)
#ifndef PCGC_FARFIELD_DEFAULT
#define PCGC_FARFIELD_DEFAULT 1      // far-field tiles of the analysis transform (bit-identical, measured +2-3 % on the step); PCGC_FARFIELD=0 computes every tile
#endif

struct UmmaProgram {
  bool ready = false;
  UmmaWeights ka[9], kb[9];
  UmmaWeights first;            // synthesis: deconv_in (16 -> 64)
  UmmaWeights last;             // analysis: conv_out (64 -> 16); synthesis: deconv_out (16 -> 1)
  UmmaWeights up[2][2];         // synthesis: up_1 (two class groups), up_2 (one group) as 8-tap parity-class GEMMs
  int up_groups[2] = {0, 0};
  UmmaWeights down[2];          // analysis: down_1, down_2 as 8-tap GEMMs over the space-to-depth input
  float* conv_in_w = nullptr;   // analysis: conv_in weights [27][16] for the dedicated kernel
  // model_simple (models/model_simple.py:21-42,58-86) on the window-GEMM kernel (umma_win.cu)
  WinLayer s_conv1, s_conv2, s_conv3;   // analysis: 9^3 s2 1->32 (5^3 cells x 8 parities), 5^3 s2 32->32 (3^3 cells x 8 parities x 32) twice
  WinLayer s_deconv1[4], s_deconv2[4];  // synthesis: 5^3 s2 transposed 32->32 (8^3 -> 16^3, 16^3 -> 32^3), two output-parity classes per launch
  WinLayer s_deconv3;           // synthesis: 9^3 s2 transposed 32->1, the 8 classes as 8 columns
  WinLayer h_deconv1, h_deconv2[2];   // hyper decoder on its 8^3 grid: 3^3 conv 8->16 (paired taps), 3^3 s2 transposed 16->16 (2 x 4 classes)
};

struct Net {
  std::vector<LayerSpec> specs;
  std::vector<LayerW> w;
  std::vector<Op> ops;
  int in_n = 0, in_c = 0;       // external input grid / channels
  size_t elems[BUF_COUNT] = {0};   // floats per cube of each internal buffer
  UmmaProgram up;
  int find(const char* name) const {
    for (size_t i = 0; i < specs.size(); ++i) if (specs[i].name == name) return (int)i;
    return -1;
  }
};

void add_vrn_specs(Net& n, const std::string& p, int c) {
  n.specs.push_back({p + "_conv1_1", c, c / 4, 3, 1, false, true, true});
  n.specs.push_back({p + "_conv1_2", c / 4, c / 2, 3, 1, false, true, true});
  n.specs.push_back({p + "_conv2_1", c, c / 4, 1, 1, false, true, true});
  n.specs.push_back({p + "_conv2_2", c / 4, c / 4, 3, 1, false, true, true});
  n.specs.push_back({p + "_conv2_3", c / 4, c / 2, 1, 1, false, true, true});
}

struct Builder {
  Net& n;
  explicit Builder(Net& net) : n(net) {}
  void need(int buf, size_t e) { if (buf != BUF_IN && buf < BUF_OUT0) n.elems[buf] = std::max(n.elems[buf], e); }
  // returns the output grid edge
  int conv(const char* name, int in, int in_n, int in_cs, int in_co, int out, int out_cs, int out_co,
           int res = -1, int res_cs = 0, int res_co = 0, int extra_flags = 0) {
    const int li = n.find(name);
    const LayerSpec& s = n.specs[li];
    const int out_n = s.transposed ? in_n * s.stride : in_n / s.stride;
    Op op{li, in, in_n, in_cs, in_co, out, out_cs, out_co, res, res_cs, res_co, (s.relu ? EPI_RELU : 0) | extra_flags};
    n.ops.push_back(op);
    need(in, (size_t)in_n * in_n * in_n * in_cs);
    need(out, (size_t)out_n * out_n * out_n * out_cs);
    return out_n;
  }
  // _VoxceptionResNet.call (model_voxception.py:56-68): X -> Y, both C channels on an n^3 grid.
  void vrn(const std::string& p, int c, int nn, int X, int Y) {
    conv((p + "_conv1_1").c_str(), X, nn, c, 0, BUF_T1, c / 2, 0);
    conv((p + "_conv2_1").c_str(), X, nn, c, 0, BUF_T1, c / 2, c / 4);
    conv((p + "_conv1_2").c_str(), BUF_T1, nn, c / 2, 0, Y, c, 0, X, c, 0);           // relu(x + concat[..])
    conv((p + "_conv2_2").c_str(), BUF_T1, nn, c / 2, c / 4, BUF_T2, c / 4, 0);
    conv((p + "_conv2_3").c_str(), BUF_T2, nn, c / 4, 0, Y, c, c / 2, X, c, c / 2);
  }
};

void build_net(Net& n, int kind) {
  n.specs.clear(); n.ops.clear();
  Builder b(n);
  auto S = [&](const char* name, int cin, int cout, int k = 3, int stride = 1, bool tr = false, bool bias = true,
               bool relu = true) { n.specs.push_back({name, cin, cout, k, stride, tr, bias, relu}); };
  switch (kind) {
    case PCGC_NET_VOX_ANALYSIS: {
      S("conv_in", 1, 16);
      for (int i = 1; i <= 3; ++i) add_vrn_specs(n, "vrn1_" + std::to_string(i), 16);
      S("down_1", 16, 32, 3, 2, false, false, true);
      for (int i = 1; i <= 3; ++i) add_vrn_specs(n, "vrn2_" + std::to_string(i), 32);
      S("down_2", 32, 64, 3, 2, false, false, true);
      for (int i = 1; i <= 3; ++i) add_vrn_specs(n, "vrn3_" + std::to_string(i), 64);
      S("conv_out", 64, 16, 3, 1, false, true, false);
      n.in_n = 64; n.in_c = 1;
      b.conv("conv_in", BUF_X0, 64, 1, 0, BUF_A, 16, 0);
      b.vrn("vrn1_1", 16, 64, BUF_A, BUF_B); b.vrn("vrn1_2", 16, 64, BUF_B, BUF_A); b.vrn("vrn1_3", 16, 64, BUF_A, BUF_B);
      b.conv("down_1", BUF_B, 64, 16, 0, BUF_A, 32, 0);
      b.vrn("vrn2_1", 32, 32, BUF_A, BUF_B); b.vrn("vrn2_2", 32, 32, BUF_B, BUF_A); b.vrn("vrn2_3", 32, 32, BUF_A, BUF_B);
      b.conv("down_2", BUF_B, 32, 32, 0, BUF_A, 64, 0);
      b.vrn("vrn3_1", 64, 16, BUF_A, BUF_B); b.vrn("vrn3_2", 64, 16, BUF_B, BUF_A); b.vrn("vrn3_3", 64, 16, BUF_A, BUF_B);
      b.conv("conv_out", BUF_B, 16, 64, 0, BUF_OUT0, 16, 0);
    } break;
    case PCGC_NET_VOX_SYNTHESIS: {
      S("deconv_in", 16, 64);
      for (int i = 1; i <= 3; ++i) add_vrn_specs(n, "dvrn1_" + std::to_string(i), 64);
      S("up_1", 64, 32, 3, 2, true, true, true);
      for (int i = 1; i <= 3; ++i) add_vrn_specs(n, "dvrn2_" + std::to_string(i), 32);
      S("up_2", 32, 16, 3, 2, true, true, true);
      for (int i = 1; i <= 3; ++i) add_vrn_specs(n, "dvrn3_" + std::to_string(i), 16);
      S("deconv_out", 16, 1, 3, 1, false, true, false);
      n.in_n = 16; n.in_c = 16;
      b.conv("deconv_in", BUF_IN, 16, 16, 0, BUF_A, 64, 0);
      b.vrn("dvrn1_1", 64, 16, BUF_A, BUF_B); b.vrn("dvrn1_2", 64, 16, BUF_B, BUF_A); b.vrn("dvrn1_3", 64, 16, BUF_A, BUF_B);
      b.conv("up_1", BUF_B, 16, 64, 0, BUF_A, 32, 0);
      b.vrn("dvrn2_1", 32, 32, BUF_A, BUF_B); b.vrn("dvrn2_2", 32, 32, BUF_B, BUF_A); b.vrn("dvrn2_3", 32, 32, BUF_A, BUF_B);
      b.conv("up_2", BUF_B, 32, 32, 0, BUF_A, 16, 0);
      b.vrn("dvrn3_1", 16, 64, BUF_A, BUF_B); b.vrn("dvrn3_2", 16, 64, BUF_B, BUF_A); b.vrn("dvrn3_3", 16, 64, BUF_A, BUF_B);
      b.conv("deconv_out", BUF_B, 64, 16, 0, BUF_OUT0, 1, 0);
    } break;
    case PCGC_NET_HYPER_ENCODER: {
      S("conv1", 16, 16); S("conv2", 16, 16, 3, 2); S("conv3", 16, 8, 3, 1, false, true, false);
      n.in_n = 16; n.in_c = 16;
      b.conv("conv1", BUF_IN, 16, 16, 0, BUF_A, 16, 0);
      b.conv("conv2", BUF_A, 16, 16, 0, BUF_B, 16, 0);
      b.conv("conv3", BUF_B, 8, 16, 0, BUF_OUT0, 8, 0);
    } break;
    case PCGC_NET_HYPER_DECODER: {
      S("deconv1", 8, 16); S("deconv2", 16, 16, 3, 2, true); S("deconv3", 16, 32);
      S("deconv4_1", 32, 16, 3, 1, false, true, false); S("deconv4_2", 32, 16, 3, 1, false, true, false);
      n.in_n = 8; n.in_c = 8;
      b.conv("deconv1", BUF_IN, 8, 8, 0, BUF_A, 16, 0);
      b.conv("deconv2", BUF_A, 8, 16, 0, BUF_B, 16, 0);
      b.conv("deconv3", BUF_B, 16, 16, 0, BUF_A, 32, 0);
      b.conv("deconv4_1", BUF_A, 16, 32, 0, BUF_OUT0, 16, 0);
      b.conv("deconv4_2", BUF_A, 16, 32, 0, BUF_OUT1, 16, 0, -1, 0, 0, EPI_ABS | EPI_FLOOR);  // abs (:308) + max(.,1e-9) (transform.py:146)
    } break;
    case PCGC_NET_SIMPLE_ANALYSIS: {
      S("conv_1", 1, 32, 9, 2); S("conv_2", 32, 32, 5, 2); S("conv_3", 32, 32, 5, 2, false, false, false);
      n.in_n = 64; n.in_c = 1;
      b.conv("conv_1", BUF_X0, 64, 1, 0, BUF_A, 32, 0);
      b.conv("conv_2", BUF_A, 32, 32, 0, BUF_B, 32, 0);
      b.conv("conv_3", BUF_B, 16, 32, 0, BUF_OUT0, 32, 0);
    } break;
    case PCGC_NET_SIMPLE_SYNTHESIS: {
      S("deconv_1", 32, 32, 5, 2, true); S("deconv_2", 32, 32, 5, 2, true); S("deconv_3", 32, 1, 9, 2, true, true, false);
      n.in_n = 8; n.in_c = 32;
      b.conv("deconv_1", BUF_IN, 8, 32, 0, BUF_A, 32, 0);
      b.conv("deconv_2", BUF_A, 16, 32, 0, BUF_B, 32, 0);
      b.conv("deconv_3", BUF_B, 32, 32, 0, BUF_OUT0, 1, 0);
    } break;
  }
  n.w.assign(n.specs.size(), LayerW());
}

}  // namespace

struct pcgc_ctx {
  int device = 0;
  cudaStream_t stream = nullptr;
  int engine = PCGC_ENGINE_AUTO;
  int64_t launches = 0;
  std::string err;
  Net nets[PCGC_NET_COUNT];
  BottleneckDev bn[2];
  std::vector<float> bn_host[2];    // packed parameters (44 per channel) for the host twin of the pmf (pcgc_factorized_cdf_host)
  float* train_ws[4] = {nullptr, nullptr, nullptr, nullptr};   // train.cu: packed weights / wgrad partials / reductions
  size_t train_cap[4] = {0, 0, 0, 0};
  bool deferred_checks = false;     // pcgc_set_deferred_checks
  int quant_noise = 0;              // pcgc_set_quantize_mode: 0 = "symbols" (round), 1 = "noise" (training)
  uint64_t quant_seed = 0;
  // workspaces
  float* bufs[BUF_COUNT] = {nullptr};
  size_t buf_cap[BUF_COUNT] = {0};
  double* scratch = nullptr; size_t scratch_cap = 0;
  float* pmf_dev = nullptr;
  int* err_flag = nullptr;          // device int
  int32_t* mm_dev = nullptr; size_t mm_cap = 0;
  int64_t* off_dev = nullptr; size_t off_cap = 0;
  int64_t* chunk_dev = nullptr; size_t chunk_cap = 0;   // voxelize / extract workspace
  GeoWorkspace* geo_ws = nullptr;   // pcgc_geometry_sums (metrics.cu)
  MeshWorkspace* mesh_ws = nullptr; // pcgc_mesh_sample (meshsample.cu)
  // far-field tiles of the analysis transform (PCGC_FARFIELD; DESIGN 4.1).  The 64^3 stage keeps each layer in a buffer of its own,
  // ff_act = X0, T1a, X1, T1b, X2, T1c (one cube per sub-batch slot), so that a slot still holds a known layer between calls: every voxel
  // holds the value the slot's last cube gives, which is the empty cube's value wherever that cube's tile is far.
  uint8_t* ff_zero = nullptr; float* ff_y = nullptr;
  __nv_bfloat16* ff_e[3] = {nullptr, nullptr, nullptr};          // the empty cube's X1, X2, X3: what K_b16 copies into far tiles
  float* ff_act[6] = {nullptr}; size_t ff_act_cap[6] = {0};
  // classification masks [layer][ff_cap slots][128 tiles]: ff_masks of the current sub-batch (7 layers), ff_prev of the cube each slot
  // held before (X0 .. T1c; all ones where the slot's contents are unknown)
  uint8_t* ff_rows = nullptr; uint8_t* ff_masks = nullptr; uint8_t* ff_prev = nullptr; int ff_cap = 0;
  int* ff_lists = nullptr;         // the work lists of K_a16 (T1a, T1b, T1c) and K_b16 (X1, X2): [5][ff_cap*1024 + 1] (launch_ff_list)
  bool ff_ready = false, ff_building = false;
  bool ff_known = false;           // ff_prev describes the slots (cleared by anything that writes them without masks)
  int sub_batch = 64;     // cubes per kernel launch (measured r01: 64 beats 32 by 5 % with the persistent kernels; 96 and 128 add nothing)
  // optional per-launch CUDA-event timing (bench.py roofline): see pcgc_profile_enable
  bool profiling = false;
  struct ProfRec { std::string tag; cudaEvent_t a, b; double flops, bytes; };
  std::vector<ProfRec> prof;
  std::vector<cudaEvent_t> ev_pool;
};

namespace {

int fail(pcgc_ctx* c, int code, const char* fmt, ...) {
  char buf[512];
  va_list ap;
  va_start(ap, fmt);
  vsnprintf(buf, sizeof buf, fmt, ap);
  va_end(ap);
  if (c) c->err = buf;
  return code;
}

cudaEvent_t prof_event(pcgc_ctx* c) {
  cudaEvent_t e = nullptr;
  if (!c->ev_pool.empty()) { e = c->ev_pool.back(); c->ev_pool.pop_back(); }
  else cudaEventCreate(&e);
  return e;
}
// Brackets the launches issued between begin/end with events on the ctx stream.
void prof_begin(pcgc_ctx* c, const std::string& tag, double flops, double bytes) {
  if (!c->profiling) return;
  pcgc_ctx::ProfRec r{tag, prof_event(c), prof_event(c), flops, bytes};
  cudaEventRecord(r.a, c->stream);
  c->prof.push_back(r);
}
void prof_end(pcgc_ctx* c) {
  if (!c->profiling || c->prof.empty()) return;
  cudaEventRecord(c->prof.back().b, c->stream);
}

#define CK(call)                                                                              \
  do {                                                                                        \
    cudaError_t e_ = (call);                                                                  \
    if (e_ != cudaSuccess)                                                                    \
      return fail(ctx, e_ == cudaErrorMemoryAllocation ? PCGC_ERR_OOM : PCGC_ERR_CUDA, "%s: %s", #call, \
                  cudaGetErrorString(e_));                                                    \
  } while (0)

struct DeviceGuard {
  int prev = -1;
  explicit DeviceGuard(int dev) { cudaGetDevice(&prev); if (prev != dev) cudaSetDevice(dev); else prev = -1; }
  ~DeviceGuard() { if (prev >= 0) cudaSetDevice(prev); }
};

int ensure(pcgc_ctx* ctx, float** p, size_t* cap, size_t elems) {
  if (*cap >= elems) return PCGC_OK;
  if (*p) { CK(cudaStreamSynchronize(ctx->stream)); CK(cudaFree(*p)); *p = nullptr; *cap = 0; }
  CK(cudaMalloc((void**)p, elems * sizeof(float)));
  *cap = elems;
  return PCGC_OK;
}

int ensure_scratch(pcgc_ctx* ctx, size_t n) {
  if (ctx->scratch_cap >= n) return PCGC_OK;
  if (ctx->scratch) { CK(cudaStreamSynchronize(ctx->stream)); CK(cudaFree(ctx->scratch)); ctx->scratch = nullptr; }
  CK(cudaMalloc((void**)&ctx->scratch, n * sizeof(double)));
  ctx->scratch_cap = n;
  return PCGC_OK;
}

// pad-before of TF SAME for an even extent: stride 1 -> (k-1)/2 ; stride 2 -> (k-2)/2
int same_pad_before(int k, int stride) { return stride == 1 ? (k - 1) / 2 : (k - 2) / 2; }

int check_err_flag(pcgc_ctx* ctx, const char* what, bool force = false) {
  if (ctx->deferred_checks && !force) return PCGC_OK;       // the caller promised a pcgc_synchronize before it consumes results
  int h = 0;
  CK(cudaMemcpyAsync(&h, ctx->err_flag, sizeof(int), cudaMemcpyDeviceToHost, ctx->stream));
  CK(cudaStreamSynchronize(ctx->stream));
  if (h != 0) {
    CK(cudaMemsetAsync(ctx->err_flag, 0, sizeof(int), ctx->stream));
    return fail(ctx, h, "%s: device-side check failed (code %d)", what, h);
  }
  return PCGC_OK;
}

// ---------------------------------------------------------------------------------------------- tcgen05 program
int build_umma_program(pcgc_ctx* ctx, int kind) {
  Net& n = ctx->nets[kind];
  UmmaProgram& up = n.up;
  if (up.ready) return PCGC_OK;
  if (kind == PCGC_NET_HYPER_ENCODER || kind == PCGC_NET_HYPER_DECODER) {
    auto Lw = [&](const char* name) -> LayerW& { return n.w[n.find(name)]; };
    cudaError_t e;
    if (kind == PCGC_NET_HYPER_ENCODER) {
      LayerW& l = Lw("conv1");
      e = pack_umma_weights_dense(l.hk.data(), l.hb.data(), 16, 16, up.first);
    } else {
      LayerW &l3 = Lw("deconv3"), &l41 = Lw("deconv4_1"), &l42 = Lw("deconv4_2");
      e = pack_umma_weights_dense(l3.hk.data(), l3.hb.data(), 16, 32, up.first);
      // the two heads share their input: one GEMM with N = 16 (loc) + 16 (scale)
      std::vector<float> d((size_t)27 * 32 * 32), bb(32);
      for (int t = 0; t < 27; ++t) for (int ci = 0; ci < 32; ++ci) for (int co = 0; co < 16; ++co) {
        d[((size_t)t * 32 + ci) * 32 + co] = l41.hk[((size_t)t * 32 + ci) * 16 + co];
        d[((size_t)t * 32 + ci) * 32 + 16 + co] = l42.hk[((size_t)t * 32 + ci) * 16 + co];
      }
      for (int co = 0; co < 16; ++co) { bb[co] = l41.hb[co]; bb[16 + co] = l42.hb[co]; }
      if (e == cudaSuccess) e = pack_umma_weights_dense(d.data(), bb.data(), 32, 32, up.last);
      // the two 8^3 layers on the window kernel (8 x 8 x 2-voxel tiles): deconv1 = 3^3 conv 8 -> 16 (Keras [3,3,3,8,16]),
      // deconv2 = 3^3 stride-2 transposed conv 16 -> 16 (Keras [3,3,3,Cout,Cin]; out[2t + r] gathers x[t + c] W[r - 2c], c in {-1, 0})
      LayerW &l1 = Lw("deconv1"), &l2 = Lw("deconv2");
      auto w1 = [&](int tz, int ty, int tx, int ci, int co) -> float { return l1.hk[((((size_t)tz * 3 + ty) * 3 + tx) * 8 + ci) * 16 + co]; };
      if (e == cudaSuccess) e = pack_win_layer(8, 3, 3, 3, -1, -1, -1, 16, w1, l1.hb.data(), up.h_deconv1, 2);
      for (int g = 0; g < 2 && e == cudaSuccess; ++g) {
        auto w2 = [&](int tz, int ty, int tx, int ci, int col) -> float {
          const int cl = col / 16, co = col % 16;
          const int kz = g - 2 * (tz - 1), ky = ((cl >> 1) & 1) - 2 * (ty - 1), kx = (cl & 1) - 2 * (tx - 1);
          if (kz < 0 || kz > 2 || ky < 0 || ky > 2 || kx < 0 || kx > 2) return 0.f;
          return l2.hk[((((size_t)kz * 3 + ky) * 3 + kx) * 16 + co) * 16 + ci];
        };
        std::vector<float> b2(64);
        for (int i = 0; i < 64; ++i) b2[i] = l2.hb[i % 16];
        e = pack_win_layer(16, 2, 2, 2, -1, -1, -1, 64, w2, b2.data(), up.h_deconv2[g], 2);
        up.h_deconv2[g].up_ncls = 4; up.h_deconv2[g].up_cout = 16;
        for (int i = 0; i < 4; ++i) up.h_deconv2[g].up_cls[i] = 4 * g + i;
      }
    }
    if (e != cudaSuccess) return fail(ctx, PCGC_ERR_CUDA, "pack hyper net %d: %s", kind, cudaGetErrorString(e));
    up.ready = true;
    return PCGC_OK;
  }
  const bool ana = kind == PCGC_NET_VOX_ANALYSIS;
  const char* prefix = ana ? "vrn" : "dvrn";
  const int chans[3] = {ana ? 16 : 64, 32, ana ? 64 : 16};
  auto L = [&](const std::string& name) -> LayerW& { return n.w[n.find(name.c_str())]; };
  for (int s = 0; s < 3; ++s)
    for (int i = 0; i < 3; ++i) {
      const int C = chans[s], c4 = C / 4, c2 = C / 2, idx = s * 3 + i;
      const std::string p = std::string(prefix) + std::to_string(s + 1) + "_" + std::to_string(i + 1);
      LayerW &l11 = L(p + "_conv1_1"), &l12 = L(p + "_conv1_2"), &l21 = L(p + "_conv2_1"), &l22 = L(p + "_conv2_2"), &l23 = L(p + "_conv2_3");
      // K_a: dense [27][C][c2]
      std::vector<float> da((size_t)27 * C * c2, 0.f), ba(c2);
      for (int t = 0; t < 27; ++t) for (int ci = 0; ci < C; ++ci) for (int co = 0; co < c4; ++co)
        da[((size_t)t * C + ci) * c2 + co] = l11.hk[((size_t)t * C + ci) * c4 + co];
      for (int ci = 0; ci < C; ++ci) for (int co = 0; co < c4; ++co)
        da[((size_t)13 * C + ci) * c2 + c4 + co] = l21.hk[(size_t)ci * c4 + co];       // 1x1x1 conv = centre tap
      for (int co = 0; co < c4; ++co) { ba[co] = l11.hb[co]; ba[c4 + co] = l21.hb[co]; }
      // y-banded MMAs (umma_conv.cu) on the 64^3 and 32^3 grids: 9*(WT+2) A tiles per 128*WT outputs instead of 27*WT
      // measured on B200 (r01 sweep): the banded form pays for K_b at 64^3 (0.396 -> 0.325 ms), not for the other kernels
      static const int wt_env = getenv("PCGC_UMMA_WT") ? atoi(getenv("PCGC_UMMA_WT")) : -1;
      const int nn = ana ? (64 >> s) : (16 << s);
      const int wt_a = wt_env >= 0 ? ((nn >= 32 && wt_env >= 2) ? 2 : 1) : ((umma_stream_mode() && nn == 64) ? 2 : 1);   // K_a: banded only where it streams
      // K_b: y-banded tile kernel at 64^3.  Its z-banded form (wt 1, paired taps, 3 epilogue groups) is correct but measured slower
      // (0.359 vs 0.330 ms per 32 cubes: twice as many 128-voxel outputs, each with its fixed barrier / TMEM round trips) -> opt-in only
      static const bool kb16_zband = getenv("PCGC_KB16_ZBAND") && atoi(getenv("PCGC_KB16_ZBAND")) != 0;
      const int wt = wt_env >= 0 ? wt_a : ((nn == 64 && !(kb16_zband && umma_zband_mode())) ? 2 : 1);
      cudaError_t e = pack_umma_weights_dense(da.data(), ba.data(), C, c2, up.ka[idx], 27, wt_a);
      if (e != cudaSuccess) return fail(ctx, PCGC_ERR_CUDA, "pack K_a %s: %s", p.c_str(), cudaGetErrorString(e));
      // K_b: dense [27][c2][c2 + c4], block diagonal
      const int nb = c2 + c4;
      std::vector<float> db((size_t)27 * c2 * nb, 0.f), bb(nb);
      for (int t = 0; t < 27; ++t) for (int ci = 0; ci < c4; ++ci) {
        for (int co = 0; co < c2; ++co) db[((size_t)t * c2 + ci) * nb + co] = l12.hk[((size_t)t * c4 + ci) * c2 + co];
        for (int co = 0; co < c4; ++co) db[((size_t)t * c2 + c4 + ci) * nb + c2 + co] = l22.hk[((size_t)t * c4 + ci) * c4 + co];
      }
      for (int co = 0; co < c2; ++co) bb[co] = l12.hb[co];
      for (int co = 0; co < c4; ++co) bb[c2 + co] = l22.hb[co];
      UmmaWeights& kb = up.kb[idx];
      e = pack_umma_weights_dense(db.data(), bb.data(), c2, nb, kb, 27, wt);
      if (e != cudaSuccess) return fail(ctx, PCGC_ERR_CUDA, "pack K_b %s: %s", p.c_str(), cudaGetErrorString(e));
      CK(cudaMalloc((void**)&kb.w23, (size_t)c4 * c2 * sizeof(float)));
      CK(cudaMemcpy(kb.w23, l23.hk.data(), (size_t)c4 * c2 * sizeof(float), cudaMemcpyHostToDevice));
      CK(cudaMalloc((void**)&kb.b23, c2 * sizeof(float)));
      CK(cudaMemcpy(kb.b23, l23.hb.data(), c2 * sizeof(float), cudaMemcpyHostToDevice));
      kb.c4 = c4; kb.c2 = c2;
    }
  if (ana) {
    LayerW& lo = L("conv_out");
    cudaError_t e = pack_umma_weights_dense(lo.hk.data(), lo.hb.data(), 64, 16, up.last);
    if (e != cudaSuccess) return fail(ctx, PCGC_ERR_CUDA, "pack conv_out: %s", cudaGetErrorString(e));
    // Conv3D(k3, s2, same) = pads (0,1): out[t] = sum_k in[2t+k] W[k].  On the space-to-depth input X'[t][p*Cin+ci] = in[2t+p][ci]
    // it is a 2x2x2-tap stride-1 conv (offsets d in {0,1}^3, k = 2d+p, k <= 2) with 8*Cin channels.
    const char* dn[2] = {"down_1", "down_2"};
    for (int u = 0; u < 2; ++u) {
      LayerW& ld = L(dn[u]);
      const LayerSpec& sp = n.specs[n.find(dn[u])];
      const int cin = sp.cin, cout = sp.cout, K = 8 * cin;
      std::vector<float> d((size_t)8 * K * cout, 0.f);
      for (int tap = 0; tap < 8; ++tap) for (int par = 0; par < 8; ++par) {
        const int k[3] = {2 * ((tap >> 2) & 1) + ((par >> 2) & 1), 2 * ((tap >> 1) & 1) + ((par >> 1) & 1), 2 * (tap & 1) + (par & 1)};
        if (k[0] > 2 || k[1] > 2 || k[2] > 2) continue;
        const float* wk = ld.hk.data() + (((size_t)k[0] * 3 + k[1]) * 3 + k[2]) * cin * cout;       // [cin][cout]
        for (int ci = 0; ci < cin; ++ci) for (int co = 0; co < cout; ++co)
          d[((size_t)tap * K + par * cin + ci) * cout + co] = wk[(size_t)ci * cout + co];
      }
      e = pack_umma_weights_dense(d.data(), ld.hb.empty() ? nullptr : ld.hb.data(), K, cout, up.down[u], 8);
      if (e != cudaSuccess) return fail(ctx, PCGC_ERR_CUDA, "pack %s: %s", dn[u], cudaGetErrorString(e));
      up.down[u].origin = 0;
    }
  } else {
    LayerW &li = L("deconv_in"), &lo = L("deconv_out");
    cudaError_t e = pack_umma_weights_dense(li.hk.data(), li.hb.data(), 16, 64, up.first);
    if (e == cudaSuccess) e = pack_umma_weights_dense(lo.hk.data(), lo.hb.data(), 16, 1, up.last, 27,
                                                          getenv("PCGC_UMMA_WT") ? (atoi(getenv("PCGC_UMMA_WT")) >= 2 ? 4 : 1) : (umma_stream_mode() ? 2 : 1));
    if (e != cudaSuccess) return fail(ctx, PCGC_ERR_CUDA, "pack deconv_in/out: %s", cudaGetErrorString(e));
    // Conv3DTranspose(k3, s2, same): out[2t] = x[t] W[0] + x[t-1] W[2], out[2t+1] = x[t] W[1] per axis.  One GEMM over the
    // 2x2x2 input window {t-1,t}^3 (brick index 0/1) whose column blocks are the 8 output-parity classes.
    const char* up_names[2] = {"up_1", "up_2"};
    for (int u = 0; u < 2; ++u) {
      LayerW& lu = L(up_names[u]);
      const LayerSpec& sp = n.specs[n.find(up_names[u])];
      const int cin = sp.cin, cout = sp.cout;
      const int groups = (8 * cout) / 128;                  // up_1: 2 groups of 4 classes, up_2: 1 group of 8
      const int ncls = 8 / groups;
      up.up_groups[u] = groups;
      for (int g = 0; g < groups; ++g) {
        const int N = ncls * cout;
        std::vector<float> d((size_t)8 * cin * N, 0.f), bb(N);
        for (int tap = 0; tap < 8; ++tap) {
          const int idx[3] = {(tap >> 2) & 1, (tap >> 1) & 1, tap & 1};
          for (int cl = 0; cl < ncls; ++cl) {
            const int gc = g * ncls + cl;
            const int r[3] = {(gc >> 2) & 1, (gc >> 1) & 1, gc & 1};
            int k[3]; bool ok = true;
            for (int ax = 0; ax < 3; ++ax) {
              if (r[ax] == 0) k[ax] = idx[ax] ? 0 : 2; else if (idx[ax]) k[ax] = 1; else ok = false;
            }
            if (!ok) continue;
            const float* wk = lu.hk.data() + (((size_t)k[0] * 3 + k[1]) * 3 + k[2]) * cout * cin;     // [cout][cin]
            for (int ci = 0; ci < cin; ++ci) for (int co = 0; co < cout; ++co)
              d[((size_t)tap * cin + ci) * N + cl * cout + co] = wk[(size_t)co * cin + ci];
          }
        }
        for (int cl = 0; cl < ncls; ++cl) for (int co = 0; co < cout; ++co) bb[cl * cout + co] = lu.hb[co];
        UmmaWeights& w = up.up[u][g];
        e = pack_umma_weights_dense(d.data(), bb.data(), cin, N, w, 8);
        if (e != cudaSuccess) return fail(ctx, PCGC_ERR_CUDA, "pack %s: %s", up_names[u], cudaGetErrorString(e));
        w.up_ncls = ncls; w.up_cls0 = g * ncls; w.up_cout = cout;
      }
    }
  }
  up.ready = true;
  return PCGC_OK;
}

// Analysis / synthesis on the tcgen05 engine.  Internal activations are PM split-bf16 (same byte size as
// float32, so the float workspaces are reused); stride-2 / transposed / Cin=1 layers run on the FP32 CUDA-core
// kernel reading and writing PM directly.
int run_vox_umma(pcgc_ctx* ctx, int kind, const float* in_ext, const void* cubes, int cubes_dtype, int B, float* out0) {
  Net& n = ctx->nets[kind];
  for (size_t i = 0; i < n.w.size(); ++i)
    if (!n.w[i].loaded) return fail(ctx, PCGC_ERR_NOT_READY, "net %d: layer '%s' has no weights", kind, n.specs[i].name.c_str());
  int r = build_umma_program(ctx, kind);
  if (r) return r;
  if (B <= 0) return PCGC_OK;
  const bool ana = kind == PCGC_NET_VOX_ANALYSIS;
  const int SB = std::min(B, ctx->sub_batch);
  for (int bi = BUF_X0; bi < BUF_OUT0; ++bi) {
    size_t e = n.elems[bi];
    if (bi == BUF_X0) e = std::max(e, (size_t)64 * 64 * 64);
    if (bi == BUF_T2) continue;                       // t22 never leaves the K_b epilogue
    if (e) { r = ensure(ctx, &ctx->bufs[bi], &ctx->buf_cap[bi], e * SB); if (r) return r; }
  }
  UmmaProgram& up = n.up;
  auto pm = [&](int buf, int nn, int c, int nb) { PmTensor t; t.p = (__nv_bfloat16*)ctx->bufs[buf]; t.n = nn; t.c = c; t.B = nb; return t; };
  auto umma = [&](const char* what, const UmmaWeights& w, const PmTensor& in, int epi, int flags, const PmTensor& out, const PmTensor& res,
                  float* of32, int ocs, int s2d = 0, const uint8_t* ff_mask = nullptr, const uint8_t* ff_prev = nullptr,
                  const __nv_bfloat16* ff_src = nullptr, const int* ff_list = nullptr, int ff_list_zs = 0) -> int {
    UmmaCall c; c.out_s2d = s2d; c.in = in; c.epi = epi; c.flags = flags; c.out = out; c.res = res; c.out_f32 = of32; c.out_cs = ocs; c.out_co = 0;
    c.err = ctx->err_flag; c.ff_mask = ff_mask; c.ff_prev = ff_prev; c.ff_src = ff_src; c.ff_list = ff_list; c.ff_list_zs = ff_list_zs;
    char tag[96];
    snprintf(tag, sizeof tag, "conv_umma %s c%d->%d n%d", what, w.cin, w.n_real, in.n);
    // algorithmic MACs of the reference layers this kernel stands for
    double macs;
    const double vox = (double)in.n * in.n * in.n * in.B;
    if (epi == UEPI_VRN) { const double c4 = w.c4, c2 = w.c2; macs = vox * (27 * c4 * c2 + 27 * c4 * c4 + c4 * c2); }
    else if (epi == UEPI_UP) macs = vox * 27.0 * w.cin * w.up_cout * w.up_ncls / 8.0;
    else if (w.ntaps == 8) macs = vox * 27.0 * (w.cin / 8) * w.n_real;
    else if (!strcmp(what, "vrn_a")) { const double C = w.cin, c4 = C / 4; macs = vox * (27 * C * c4 + C * c4); }
    else macs = vox * 27.0 * w.cin * w.n_real;
    prof_begin(ctx, tag, 2.0 * macs, 0);
    cudaError_t e = launch_conv_umma_pm(c, w, ctx->stream, &ctx->launches);
    prof_end(ctx);
    if (e != cudaSuccess) return fail(ctx, PCGC_ERR_CUDA, "%s: %s", tag, cudaGetErrorString(e));
    return PCGC_OK;
  };
  auto ffma = [&](const char* name, const float* in_f32, const PmTensor& in, int in_n, const PmTensor& out) -> int {
    const int li = n.find(name);
    const LayerSpec& s = n.specs[li];
    LayerW& lw = n.w[li];
    const int out_n = s.transposed ? in_n * s.stride : in_n / s.stride;
    ConvCall c;
    c.in = in_f32; c.in_n = in_n; c.in_cs = s.cin; c.in_co = 0;
    c.out = nullptr; c.out_n = out_n; c.out_cs = s.cout; c.out_co = 0;
    c.bias = lw.bias; c.res = nullptr; c.res_cs = c.res_co = 0;
    c.flags = s.relu ? EPI_RELU : 0; c.floor_v = 0.f; c.B = out.B;
    c.in_pm = in_f32 ? nullptr : in.p; c.out_pm = out.p;
    char tag[96];
    snprintf(tag, sizeof tag, "conv_ffma k%d s%d%s c%d->%d n%d", s.k, s.stride, s.transposed ? "T" : "", s.cin, s.cout, in_n);
    const double tvox = (double)(s.transposed ? in_n : out_n);
    prof_begin(ctx, tag, 2.0 * out.B * tvox * tvox * tvox * s.k * s.k * s.k * s.cin * s.cout, 0);
    for (int k = 0; k < lw.n_classes; ++k) {
      c.d = lw.cls[k];
      c.tn = s.transposed ? in_n : out_n;
      cudaError_t e = launch_conv_ffma(c, ctx->stream, &ctx->launches);
      if (e != cudaSuccess) return fail(ctx, PCGC_ERR_CUDA, "conv '%s': %s", name, cudaGetErrorString(e));
    }
    prof_end(ctx);
    return PCGC_OK;
  };
  const PmTensor none;
  // The analysis 64^3 stage writes its layers into ff_act.  Far-field tiles (uint8 cubes): a tile of layer L whose receptive field (radius
  // L + 1: 1 for X0 .. 7 for X3) holds no occupied voxel equals the all-zero cube's value at the same position -- SAME padding included.
  // Per slot and layer: near tiles are computed; far tiles that the slot's previous cube left near are restored (K_b16 copies them from
  // the cached layer of the empty cube, conv_in and K_a16 compute them); the other far tiles already hold the empty cube's values and are
  // not touched.  Bit-identical to computing every tile (67-82 % of the tiles of the vox10 cloud are far).
  const int ff_ch[6] = {16, 8, 16, 8, 16, 8};
  if (ana)
    for (int L = 0; L < 6; ++L) {
      const size_t e = (size_t)ff_ch[L] * 64 * 64 * 64 * SB;      // PM: 4 bytes per channel and voxel
      if (ctx->ff_act_cap[L] < e) { ctx->ff_known = false; r = ensure(ctx, &ctx->ff_act[L], &ctx->ff_act_cap[L], e); if (r) return r; }
    }
  const char* ff_env = getenv("PCGC_FARFIELD");
  const bool ff = ana && cubes_dtype == PCGC_DTYPE_U8 && !ctx->ff_building && (ff_env ? atoi(ff_env) != 0 : PCGC_FARFIELD_DEFAULT);
  if (ana && !ff) ctx->ff_known = false;                          // every tile computed: the slots hold cubes no mask describes
  const size_t ff_cube_bytes = (size_t)4 * 64 * 64 * 64 * 8 * sizeof(__nv_bfloat16);      // one cube of a 16-channel PM tensor
  if (ff) {
    if (!ctx->ff_zero) { CK(cudaMalloc((void**)&ctx->ff_zero, 64 * 64 * 64)); CK(cudaMemsetAsync(ctx->ff_zero, 0, 64 * 64 * 64, ctx->stream)); }
    if (!ctx->ff_y) CK(cudaMalloc((void**)&ctx->ff_y, (size_t)16 * 16 * 16 * 16 * sizeof(float)));
    for (auto& e : ctx->ff_e) if (!e) CK(cudaMalloc((void**)&e, ff_cube_bytes));
    if (ctx->ff_cap < SB) {
      CK(cudaStreamSynchronize(ctx->stream));
      for (uint8_t** p : {&ctx->ff_rows, &ctx->ff_masks, &ctx->ff_prev}) if (*p) { cudaFree(*p); *p = nullptr; }
      if (ctx->ff_lists) { cudaFree(ctx->ff_lists); ctx->ff_lists = nullptr; }
      ctx->ff_cap = 0; ctx->ff_known = false;
      CK(cudaMalloc((void**)&ctx->ff_rows, (size_t)FF_LAYERS * SB * 4096));
      CK(cudaMalloc((void**)&ctx->ff_masks, (size_t)FF_LAYERS * SB * 128));
      CK(cudaMalloc((void**)&ctx->ff_prev, (size_t)6 * SB * 128));
      CK(cudaMalloc((void**)&ctx->ff_lists, (size_t)5 * ((size_t)SB * 1024 + 1) * sizeof(int)));
      ctx->ff_cap = SB;
    }
    if (!ctx->ff_ready) {                              // one pass of the empty cube with every tile computed; its block outputs are kept
      ctx->ff_building = true;
      const int rb = run_vox_umma(ctx, kind, nullptr, ctx->ff_zero, PCGC_DTYPE_U8, 1, ctx->ff_y);
      ctx->ff_building = false;
      if (rb) return rb;
      ctx->ff_ready = true;
    }
    if (!ctx->ff_known) {                              // unknown contents: every far tile of every slot is restored once
      CK(cudaMemsetAsync(ctx->ff_prev, 0xFF, (size_t)6 * ctx->ff_cap * 128, ctx->stream));
      ctx->ff_known = true;
    }
  }
  const size_t ff_ls = (size_t)ctx->ff_cap * 128;                // mask bytes per layer
  auto ff_cur = [&](int L) -> const uint8_t* { return ff ? ctx->ff_masks + L * ff_ls : nullptr; };
  auto ff_old = [&](int L) -> const uint8_t* { return ff && L < 6 ? ctx->ff_prev + L * ff_ls : nullptr; };
  // work list j: K_a16 of block i at j = 2i, K_b16 of blocks 1 and 2 at j = 1, 3
  auto ff_list = [&](int j) -> int* { return ff ? ctx->ff_lists + (size_t)j * ((size_t)ctx->ff_cap * 1024 + 1) : nullptr; };
  const int ff_list_zs[3] = {umma_zband_zs(64), ana ? umma_tile_zt(n.up.kb[0], 64, UEPI_VRN) : 0, ana ? umma_tile_zt(n.up.kb[1], 64, UEPI_VRN) : 0};
  for (int b0 = 0; b0 < B; b0 += SB) {
    const int nb = std::min(SB, B - b0);
    int cur = BUF_A, nxt = BUF_B;
    if (ff) {
      prof_begin(ctx, "ff_classify", 0, (double)nb * 64 * 64 * 64);
      CK(launch_ff_classify((const uint8_t*)cubes + (size_t)b0 * 64 * 64 * 64, nb, ctx->ff_rows, ctx->ff_masks, ff_ls, ctx->stream, &ctx->launches));
      // the units each kernel computes or restores, shared by its persistent CTAs (a static split over all units leaves some CTAs with
      // most of the near tiles)
      FfListJob jobs;
      for (int i = 0; i < 3; ++i) {
        jobs.l[2 * i] = {ff_cur(2 * i + 1), ff_old(2 * i + 1), ff_list(2 * i), ff_list_zs[0]};
        if (i < 2) jobs.l[2 * i + 1] = {ff_cur(2 * i + 2), ff_old(2 * i + 2), ff_list(2 * i + 1), ff_list_zs[1 + i]};
      }
      CK(launch_ff_list(jobs, 5, nb, ctx->stream, &ctx->launches));
      prof_end(ctx);
    }
    auto act = [&](int L) { PmTensor t; t.p = (__nv_bfloat16*)ctx->ff_act[L]; t.n = 64; t.c = ff_ch[L]; t.B = nb; return t; };
    auto vrn_stage = [&](int stage, int C, int nn, bool s2d_last = false) -> int {
      for (int i = 0; i < 3; ++i) {
        const int idx = stage * 3 + i;
        int rr = umma("vrn_a", up.ka[idx], pm(cur, nn, C, nb), UEPI_PM, EPI_RELU, pm(BUF_T1, nn, C / 2, nb), none, nullptr, 0);
        if (rr) return rr;
        const bool s2d = s2d_last && i == 2;          // the block feeding a stride-2 conv writes its output space-to-depth
        rr = umma("vrn_b", up.kb[idx], pm(BUF_T1, nn, C / 2, nb), UEPI_VRN, 0, s2d ? pm(nxt, nn / 2, 8 * C, nb) : pm(nxt, nn, C, nb),
                  pm(cur, nn, C, nb), nullptr, 0, s2d);
        if (rr) return rr;
        std::swap(cur, nxt);
      }
      return PCGC_OK;
    };
    if (ana) {
      const size_t in_elems = (size_t)64 * 64 * 64;
      const size_t esz = cubes_dtype == PCGC_DTYPE_U8 ? 1 : (cubes_dtype == PCGC_DTYPE_F32 ? 4 : 8);
      {
        // conv_in straight from the cube's own dtype into PM (the Keras [3,3,3,1,16] kernel is already [27][16])
        LayerW& lin = n.w[n.find("conv_in")];
        prof_begin(ctx, "conv_in_pm c1->16 n64", 2.0 * nb * in_elems * 27 * 16, 0);
        CK(launch_conv_in_pm((const char*)cubes + (size_t)b0 * in_elems * esz, cubes_dtype, lin.hk.data(), lin.hb.empty() ? nullptr : lin.hb.data(),
                             ctx->ff_act[0], nb, ff_cur(0), ff_old(0), ctx->stream, &ctx->launches));
        prof_end(ctx);
      }
      // the three VRN-16 blocks: X_{2i} -> K_a -> T = layer 2i+1 -> K_b (+ residual X_{2i}) -> layer 2i+2; X3 (space-to-depth for down_1)
      // goes to the shared buffer, every far tile of it copied
      for (int i = 0; i < 3; ++i) {
        const int L = 2 * i + 1;
        if ((r = umma("vrn_a", up.ka[i], act(L - 1), UEPI_PM, EPI_RELU, act(L), none, nullptr, 0, 0, nullptr, nullptr, nullptr, ff_list(2 * i),
                      ff_list_zs[0])))
          return r;
        const PmTensor out = i < 2 ? act(L + 1) : pm(BUF_B, 32, 128, nb);
        if ((r = umma("vrn_b", up.kb[i], act(L), UEPI_VRN, 0, out, act(L - 1), nullptr, 0, i == 2, ff_cur(L + 1), ff_old(L + 1), ctx->ff_e[i],
                      i < 2 ? ff_list(2 * i + 1) : nullptr, i < 2 ? ff_list_zs[1 + i] : 0)))
          return r;
        if (ctx->ff_building)                          // the empty cube's block output (one cube: nb == 1)
          CK(cudaMemcpyAsync(ctx->ff_e[i], out.p, ff_cube_bytes, cudaMemcpyDeviceToDevice, ctx->stream));
      }
      if (ff) {                                        // the masks of these cubes describe their slots now; later slots keep theirs
        CK(cudaMemcpy2DAsync(ctx->ff_prev, ff_ls, ctx->ff_masks, ff_ls, (size_t)nb * 128, 6, cudaMemcpyDeviceToDevice, ctx->stream));
      }
      if ((r = umma("down_1", up.down[0], pm(BUF_B, 32, 128, nb), UEPI_PM, EPI_RELU, pm(BUF_A, 32, 32, nb), none, nullptr, 0))) return r;
      if ((r = vrn_stage(1, 32, 32, true))) return r;
      if ((r = umma("down_2", up.down[1], pm(cur, 16, 256, nb), UEPI_PM, EPI_RELU, pm(nxt, 16, 64, nb), none, nullptr, 0))) return r;
      std::swap(cur, nxt);
      if ((r = vrn_stage(2, 64, 16))) return r;
      if ((r = umma("conv_out", up.last, pm(cur, 16, 64, nb), UEPI_F32, 0, none, none, out0 + (size_t)b0 * 16 * 16 * 16 * 16, 16))) return r;
    } else {
      // y (float32 NDHWC, 16 channels) -> PM in T1, deconv_in -> cur
      PmTensor yin = pm(BUF_T1, 16, 16, nb);
      prof_begin(ctx, "f32_to_pm", 0, 8.0 * nb * 16 * 16 * 16 * 16);
      CK(launch_f32_to_pm(in_ext + (size_t)b0 * 16 * 16 * 16 * 16, 16, 0, yin, ctx->stream, &ctx->launches));
      prof_end(ctx);
      if ((r = umma("deconv_in", up.first, yin, UEPI_PM, EPI_RELU, pm(cur, 16, 64, nb), none, nullptr, 0))) return r;
      if ((r = vrn_stage(0, 64, 16))) return r;
      for (int g = 0; g < up.up_groups[0]; ++g)
        if ((r = umma("up_1", up.up[0][g], pm(cur, 16, 64, nb), UEPI_UP, EPI_RELU, pm(nxt, 32, 32, nb), none, nullptr, 0))) return r;
      std::swap(cur, nxt);
      if ((r = vrn_stage(1, 32, 32))) return r;
      for (int g = 0; g < up.up_groups[1]; ++g)
        if ((r = umma("up_2", up.up[1][g], pm(cur, 32, 32, nb), UEPI_UP, EPI_RELU, pm(nxt, 64, 16, nb), none, nullptr, 0))) return r;
      std::swap(cur, nxt);
      if ((r = vrn_stage(2, 16, 64))) return r;
      if ((r = umma("deconv_out", up.last, pm(cur, 64, 16, nb), UEPI_F32, 0, none, none, out0 + (size_t)b0 * 64 * 64 * 64, 1))) return r;
    }
  }
  return PCGC_OK;
}

// Hyper encoder / decoder with their 16^3 layers on the tcgen05 engine (conv1; deconv3 and the fused loc|scale heads);
// the 8^3 layers and the stride-2 / transposed ones stay on the FP32 CUDA-core kernel (a few MMAC per cube).
int run_hyper_umma(pcgc_ctx* ctx, int kind, const float* in_ext, int B, float* out0, float* out1, float floor_v) {
  Net& n = ctx->nets[kind];
  for (size_t i = 0; i < n.w.size(); ++i)
    if (!n.w[i].loaded) return fail(ctx, PCGC_ERR_NOT_READY, "net %d: layer '%s' has no weights", kind, n.specs[i].name.c_str());
  int r = build_umma_program(ctx, kind);
  if (r) return r;
  if (B <= 0) return PCGC_OK;
  const int SB = std::min(B, 8 * ctx->sub_batch);
  const size_t big = (size_t)16 * 16 * 16 * 32;             // largest activation per cube (floats)
  for (int bi : {BUF_A, BUF_B, BUF_T1}) { r = ensure(ctx, &ctx->bufs[bi], &ctx->buf_cap[bi], big * SB); if (r) return r; }
  UmmaProgram& up = n.up;
  auto pm = [&](int buf, int nn, int c, int nb) { PmTensor t; t.p = (__nv_bfloat16*)ctx->bufs[buf]; t.n = nn; t.c = c; t.B = nb; return t; };
  const PmTensor none;
  auto ffma = [&](const char* name, const float* in_f32, const PmTensor* in_pm, int in_n, float* out_f32, const PmTensor* out_pm, int nb) -> int {
    const int li = n.find(name);
    const LayerSpec& s = n.specs[li];
    LayerW& lw = n.w[li];
    const int out_n = s.transposed ? in_n * s.stride : in_n / s.stride;
    ConvCall c;
    c.in = in_f32; c.in_n = in_n; c.in_cs = s.cin; c.in_co = 0;
    c.out = out_f32; c.out_n = out_n; c.out_cs = s.cout; c.out_co = 0;
    c.bias = lw.bias; c.res = nullptr; c.res_cs = c.res_co = 0;
    c.flags = s.relu ? EPI_RELU : 0; c.floor_v = 0.f; c.B = nb;
    c.in_pm = in_pm ? in_pm->p : nullptr; c.out_pm = out_pm ? out_pm->p : nullptr;
    char tag[96];
    snprintf(tag, sizeof tag, "conv_ffma k%d s%d%s c%d->%d n%d", s.k, s.stride, s.transposed ? "T" : "", s.cin, s.cout, in_n);
    const double tvox = (double)(s.transposed ? in_n : out_n);
    prof_begin(ctx, tag, 2.0 * nb * tvox * tvox * tvox * 27 * s.cin * s.cout, 0);
    for (int k = 0; k < lw.n_classes; ++k) {
      c.d = lw.cls[k];
      c.tn = s.transposed ? in_n : out_n;
      cudaError_t e = launch_conv_ffma(c, ctx->stream, &ctx->launches);
      if (e != cudaSuccess) return fail(ctx, PCGC_ERR_CUDA, "conv '%s': %s", name, cudaGetErrorString(e));
    }
    prof_end(ctx);
    return PCGC_OK;
  };
  auto umma = [&](const char* what, const UmmaWeights& w, const PmTensor& in, UmmaCall c) -> int {
    c.in = in; c.err = ctx->err_flag;
    char tag[96];
    snprintf(tag, sizeof tag, "conv_umma %s c%d->%d n%d", what, w.cin, w.n_real, in.n);
    prof_begin(ctx, tag, 2.0 * in.B * in.n * in.n * in.n * 27.0 * w.cin * w.n_real, 0);
    cudaError_t e = launch_conv_umma_pm(c, w, ctx->stream, &ctx->launches);
    prof_end(ctx);
    if (e != cudaSuccess) return fail(ctx, PCGC_ERR_CUDA, "%s: %s", tag, cudaGetErrorString(e));
    return PCGC_OK;
  };
  for (int b0 = 0; b0 < B; b0 += SB) {
    const int nb = std::min(SB, B - b0);
    if (kind == PCGC_NET_HYPER_ENCODER) {
      PmTensor yin = pm(BUF_T1, 16, 16, nb), f1 = pm(BUF_A, 16, 16, nb);
      CK(launch_f32_to_pm(in_ext + (size_t)b0 * 65536, 16, 0, yin, ctx->stream, &ctx->launches));
      UmmaCall c; c.epi = UEPI_PM; c.flags = EPI_RELU; c.out = f1;
      if ((r = umma("conv1", up.first, yin, c))) return r;
      if ((r = ffma("conv2", nullptr, &f1, 16, ctx->bufs[BUF_B], nullptr, nb))) return r;
      if ((r = ffma("conv3", ctx->bufs[BUF_B], nullptr, 8, out0 + (size_t)b0 * 4096, nullptr, nb))) return r;
    } else {
      PmTensor zin = pm(BUF_T1, 8, 8, nb), d1 = pm(BUF_A, 8, 16, nb), f2 = pm(BUF_B, 16, 16, nb), f3 = pm(BUF_T1, 16, 32, nb);
      auto win = [&](const char* what, const WinLayer& w, const PmTensor& in, WinCall c, bool open_tag, bool close_tag, double mult) -> int {
        c.in = in; c.err = ctx->err_flag;
        char tag[96];
        snprintf(tag, sizeof tag, "conv_umma_win %s c%d->%d n%d", what, w.cin, w.n_cols, in.n);
        if (open_tag) prof_begin(ctx, tag, 2.0 * in.B * (double)in.n * in.n * in.n * w.macs_per_row * mult, 0);
        cudaError_t e = launch_conv_umma_win(c, w, ctx->stream, &ctx->launches);
        if (close_tag) prof_end(ctx);
        if (e != cudaSuccess) return fail(ctx, PCGC_ERR_CUDA, "%s: %s", tag, cudaGetErrorString(e));
        return PCGC_OK;
      };
      // pinned kernels from here on: loc / scale feed the integer CDF tables, so the decoder process must reproduce the encoder's bits
      CK(launch_f32_to_pm(in_ext + (size_t)b0 * 4096, 8, 0, zin, ctx->stream, &ctx->launches));
      WinCall c1; c1.epi = WEPI_PM; c1.flags = EPI_RELU; c1.out = d1;
      if ((r = win("deconv1", up.h_deconv1, zin, c1, true, true, 1.0))) return r;
      for (int g = 0; g < 2; ++g) {
        WinCall c2; c2.epi = WEPI_UP_PM; c2.flags = EPI_RELU; c2.out = f2;
        if ((r = win("deconv2", up.h_deconv2[g], d1, c2, g == 0, g == 1, 2.0))) return r;
      }
      // pinned kernels: loc / scale feed the integer CDF tables, so the decoder process must reproduce the encoder's bits
      UmmaCall c; c.epi = UEPI_PM; c.flags = EPI_RELU; c.out = f3; c.pin_tile = true;
      if ((r = umma("deconv3", up.first, f2, c))) return r;
      UmmaCall h; h.epi = UEPI_F32; h.pin_tile = true; h.flags = 0; h.out_f32 = out0 + (size_t)b0 * 65536; h.out_cs = 16; h.out_co = 0;
      h.out2_f32 = out1 + (size_t)b0 * 65536; h.split = 16; h.flags2 = EPI_ABS | EPI_FLOOR; h.floor_v = floor_v;   // abs (:308) + max(., 1e-9)
      if ((r = umma("deconv4_1|4_2", up.last, f3, h))) return r;
    }
  }
  return PCGC_OK;
}


// model_simple, every layer on the tcgen05 window-GEMM kernel (umma_win.cu; the 8^3 grids in its 8 x 8 x 2-voxel tile form).
//   analysis : cube -> space-to-depth PM [32^3][8] -> conv_1 (5^3 cells) -> space-to-depth PM [16^3][256] -> conv_2 (3^3 cells)
//              -> space-to-depth PM [8^3][256] -> conv_3 (3^3 cells) -> y float32 [8^3][32]
//   synthesis: y -> PM [8^3][32] -> deconv_1 (4 launches x 2 parity classes) -> PM [16^3][32] -> deconv_2 (the same) -> PM [32^3][32]
//              -> deconv_3 (8 classes = 8 columns) -> logits float32 [64^3][1]
int build_simple_program(pcgc_ctx* ctx, int kind) {
  Net& n = ctx->nets[kind];
  UmmaProgram& up = n.up;
  if (up.ready) return PCGC_OK;
  auto Lw = [&](const char* name) -> LayerW& { return n.w[n.find(name)]; };
  cudaError_t e = cudaSuccess;
  if (kind == PCGC_NET_SIMPLE_ANALYSIS) {
    const LayerW &l1 = Lw("conv_1"), &l2 = Lw("conv_2");
    // conv_1: x index = 2(o + c) + p, tap k = 2c + p + 3 (SAME pads (3,4)); Keras [9,9,9,1,32]
    auto w1 = [&](int tz, int ty, int tx, int ci, int co) -> float {
      const int kz = 2 * (tz - 2) + ((ci >> 2) & 1) + 3, ky = 2 * (ty - 2) + ((ci >> 1) & 1) + 3, kx = 2 * (tx - 2) + (ci & 1) + 3;
      if (kz < 0 || kz > 8 || ky < 0 || ky > 8 || kx < 0 || kx > 8) return 0.f;
      return l1.hk[(((size_t)kz * 9 + ky) * 9 + kx) * 32 + co];
    };
    e = pack_win_layer(8, 5, 5, 5, -2, -2, -2, 32, w1, l1.hb.data(), up.s_conv1);
    // conv_2: tap k = 2c + p + 1 (SAME pads (1,2)); input channel = parity * 32 + c; Keras [5,5,5,32,32]
    auto w2 = [&](int tz, int ty, int tx, int ci, int co) -> float {
      const int par = ci / 32, c = ci % 32;
      const int kz = 2 * (tz - 1) + ((par >> 2) & 1) + 1, ky = 2 * (ty - 1) + ((par >> 1) & 1) + 1, kx = 2 * (tx - 1) + (par & 1) + 1;
      if (kz < 0 || kz > 4 || ky < 0 || ky > 4 || kx < 0 || kx > 4) return 0.f;
      return l2.hk[((((size_t)kz * 5 + ky) * 5 + kx) * 32 + c) * 32 + co];
    };
    if (e == cudaSuccess) e = pack_win_layer(256, 3, 3, 3, -1, -1, -1, 32, w2, l2.hb.data(), up.s_conv2);
    const LayerW& l3 = Lw("conv_3");                         // the same form on the 8^3 output grid, no bias, no activation
    auto w3 = [&](int tz, int ty, int tx, int ci, int co) -> float {
      const int par = ci / 32, c = ci % 32;
      const int kz = 2 * (tz - 1) + ((par >> 2) & 1) + 1, ky = 2 * (ty - 1) + ((par >> 1) & 1) + 1, kx = 2 * (tx - 1) + (par & 1) + 1;
      if (kz < 0 || kz > 4 || ky < 0 || ky > 4 || kx < 0 || kx > 4) return 0.f;
      return l3.hk[((((size_t)kz * 5 + ky) * 5 + kx) * 32 + c) * 32 + co];
    };
    if (e == cudaSuccess) e = pack_win_layer(256, 3, 3, 3, -1, -1, -1, 32, w3, nullptr, up.s_conv3, 2);
  } else {
    const LayerW &l1 = Lw("deconv_1"), &l2 = Lw("deconv_2"), &l3 = Lw("deconv_3");
    // Conv3DTranspose: out[2t + r] gathers x[t + c] W[k], k = r + pad_before - 2c; Keras [k,k,k,Cout,Cin]
    for (int layer = 0; layer < 2; ++layer) {
      const LayerW& l = layer == 0 ? l1 : l2;
      for (int g = 0; g < 4 && e == cudaSuccess; ++g) {
        auto w = [&](int tz, int ty, int tx, int ci, int col) -> float {
          const int rz = g >> 1, ry = g & 1, rx = col / 32, co = col % 32;
          const int kz = rz + 1 - 2 * (tz - 1), ky = ry + 1 - 2 * (ty - 1), kx = rx + 1 - 2 * (tx - 1);
          if (kz < 0 || kz > 4 || ky < 0 || ky > 4 || kx < 0 || kx > 4) return 0.f;
          return l.hk[((((size_t)kz * 5 + ky) * 5 + kx) * 32 + co) * 32 + ci];
        };
        std::vector<float> bb(64);
        for (int i = 0; i < 64; ++i) bb[i] = l.hb[i % 32];
        WinLayer& wl = layer == 0 ? up.s_deconv1[g] : up.s_deconv2[g];
        e = pack_win_layer(32, 3, 3, 3, -1, -1, -1, 64, w, bb.data(), wl, layer == 0 ? 2 : 1);
        wl.up_ncls = 2; wl.up_cout = 32;
        wl.up_cls[0] = 2 * g; wl.up_cls[1] = 2 * g + 1;
      }
    }
    auto w3 = [&](int tz, int ty, int tx, int ci, int col) -> float {
      const int kz = ((col >> 2) & 1) + 3 - 2 * (tz - 2), ky = ((col >> 1) & 1) + 3 - 2 * (ty - 2), kx = (col & 1) + 3 - 2 * (tx - 2);
      if (kz < 0 || kz > 8 || ky < 0 || ky > 8 || kx < 0 || kx > 8) return 0.f;
      return l3.hk[(((size_t)kz * 9 + ky) * 9 + kx) * 32 + ci];
    };
    std::vector<float> b3(8, l3.hb.empty() ? 0.f : l3.hb[0]);
    if (e == cudaSuccess) e = pack_win_layer(32, 5, 5, 5, -2, -2, -2, 8, w3, b3.data(), up.s_deconv3);
    up.s_deconv3.up_ncls = 8; up.s_deconv3.up_cout = 1;
    for (int i = 0; i < 8; ++i) up.s_deconv3.up_cls[i] = i;
  }
  if (e != cudaSuccess) return fail(ctx, PCGC_ERR_CUDA, "pack model_simple net %d: %s", kind, cudaGetErrorString(e));
  up.ready = true;
  return PCGC_OK;
}

int run_simple_umma(pcgc_ctx* ctx, int kind, const float* in_ext, const void* cubes, int cubes_dtype, int B, float* out0) {
  Net& n = ctx->nets[kind];
  for (size_t i = 0; i < n.w.size(); ++i)
    if (!n.w[i].loaded) return fail(ctx, PCGC_ERR_NOT_READY, "net %d: layer '%s' has no weights", kind, n.specs[i].name.c_str());
  int r = build_simple_program(ctx, kind);
  if (r) return r;
  if (B <= 0) return PCGC_OK;
  const int SB = std::min(B, ctx->sub_batch);
  for (int bi = BUF_X0; bi < BUF_OUT0; ++bi) {
    size_t e = n.elems[bi];
    if (bi == BUF_X0) e = std::max(e, (size_t)64 * 64 * 64);
    if (e) { r = ensure(ctx, &ctx->bufs[bi], &ctx->buf_cap[bi], e * SB); if (r) return r; }
  }
  UmmaProgram& up = n.up;
  auto pm = [&](int buf, int nn, int c, int nb) { PmTensor t; t.p = (__nv_bfloat16*)ctx->bufs[buf]; t.n = nn; t.c = c; t.B = nb; return t; };
  auto ffma = [&](const char* name, const float* in_f32, const PmTensor* in_pm, int in_n, float* out_f32, const PmTensor* out_pm, int nb) -> int {
    const int li = n.find(name);
    const LayerSpec& s = n.specs[li];
    LayerW& lw = n.w[li];
    const int out_n = s.transposed ? in_n * s.stride : in_n / s.stride;
    ConvCall c;
    c.in = in_f32; c.in_n = in_n; c.in_cs = s.cin; c.in_co = 0;
    c.out = out_f32; c.out_n = out_n; c.out_cs = s.cout; c.out_co = 0;
    c.bias = lw.bias; c.res = nullptr; c.res_cs = c.res_co = 0;
    c.flags = s.relu ? EPI_RELU : 0; c.floor_v = 0.f; c.B = nb;
    c.in_pm = in_pm ? in_pm->p : nullptr; c.out_pm = out_pm ? out_pm->p : nullptr;
    char tag[96];
    snprintf(tag, sizeof tag, "conv_ffma k%d s%d%s c%d->%d n%d", s.k, s.stride, s.transposed ? "T" : "", s.cin, s.cout, in_n);
    const double tvox = (double)(s.transposed ? in_n : out_n);
    prof_begin(ctx, tag, 2.0 * nb * tvox * tvox * tvox * s.k * s.k * s.k * s.cin * s.cout, 0);
    for (int k = 0; k < lw.n_classes; ++k) {
      c.d = lw.cls[k];
      c.tn = s.transposed ? in_n : out_n;
      cudaError_t e = launch_conv_ffma(c, ctx->stream, &ctx->launches);
      if (e != cudaSuccess) return fail(ctx, PCGC_ERR_CUDA, "conv '%s': %s", name, cudaGetErrorString(e));
    }
    prof_end(ctx);
    return PCGC_OK;
  };
  auto win = [&](const char* what, const WinLayer& w, const PmTensor& in, WinCall c, bool open_tag = true, bool close_tag = true) -> int {
    c.in = in; c.err = ctx->err_flag;
    char tag[96];
    snprintf(tag, sizeof tag, "conv_umma_win %s c%d->%d n%d", what, w.cin, w.n_cols, in.n);
    if (open_tag) prof_begin(ctx, tag, 2.0 * in.B * (double)in.n * in.n * in.n * w.macs_per_row * (close_tag ? 1.0 : 4.0), 0);
    cudaError_t e = launch_conv_umma_win(c, w, ctx->stream, &ctx->launches);
    if (close_tag) prof_end(ctx);
    if (e != cudaSuccess) return fail(ctx, PCGC_ERR_CUDA, "%s: %s", tag, cudaGetErrorString(e));
    return PCGC_OK;
  };
  for (int b0 = 0; b0 < B; b0 += SB) {
    const int nb = std::min(SB, B - b0);
    if (kind == PCGC_NET_SIMPLE_ANALYSIS) {
      const size_t esz = cubes_dtype == PCGC_DTYPE_U8 ? 1 : (cubes_dtype == PCGC_DTYPE_F32 ? 4 : 8);
      const void* src = cubes ? (const void*)((const char*)cubes + (size_t)b0 * 262144 * esz) : (const void*)(in_ext + (size_t)b0 * 262144);
      PmTensor x = pm(BUF_X0, 32, 8, nb), f1 = pm(BUF_A, 16, 256, nb), f2 = pm(BUF_B, 8, 256, nb);
      CK(launch_cubes_to_s2d_pm(src, cubes ? cubes_dtype : PCGC_DTYPE_F32, x, ctx->stream, &ctx->launches));
      WinCall c1; c1.epi = WEPI_PM; c1.flags = EPI_RELU; c1.out = f1; c1.out_s2d = 1;
      if ((r = win("conv_1", up.s_conv1, x, c1))) return r;
      WinCall c2; c2.epi = WEPI_PM; c2.flags = EPI_RELU; c2.out = f2; c2.out_s2d = 1;
      if ((r = win("conv_2", up.s_conv2, f1, c2))) return r;
      WinCall c3; c3.epi = WEPI_F32; c3.flags = 0; c3.out_f32 = out0 + (size_t)b0 * 8 * 8 * 8 * 32; c3.out_cs = 32; c3.out_co = 0;
      if ((r = win("conv_3", up.s_conv3, f2, c3))) return r;
    } else {
      PmTensor yin = pm(BUF_B, 8, 32, nb), f1 = pm(BUF_A, 16, 32, nb), f2 = pm(BUF_B, 32, 32, nb);
      CK(launch_f32_to_pm(in_ext + (size_t)b0 * 8 * 8 * 8 * 32, 32, 0, yin, ctx->stream, &ctx->launches));
      for (int g = 0; g < 4; ++g) {
        WinCall c; c.epi = WEPI_UP_PM; c.flags = EPI_RELU; c.out = f1;
        if ((r = win("deconv_1", up.s_deconv1[g], yin, c, g == 0, g == 3))) return r;
      }
      for (int g = 0; g < 4; ++g) {
        WinCall c; c.epi = WEPI_UP_PM; c.flags = EPI_RELU; c.out = f2;
        if ((r = win("deconv_2", up.s_deconv2[g], f1, c, g == 0, g == 3))) return r;
      }
      WinCall c3; c3.epi = WEPI_UP_F32; c3.flags = 0; c3.out_f32 = out0 + (size_t)b0 * 262144; c3.out_cs = 1; c3.out_co = 0;
      if ((r = win("deconv_3", up.s_deconv3, f2, c3))) return r;
    }
  }
  return PCGC_OK;
}

int run_net(pcgc_ctx* ctx, int kind, const float* in_ext, const void* cubes, int cubes_dtype, int B, float* out0,
            float* out1, float floor_v) {
  Net& n = ctx->nets[kind];
  for (size_t i = 0; i < n.w.size(); ++i)
    if (!n.w[i].loaded) return fail(ctx, PCGC_ERR_NOT_READY, "net %d: layer '%s' has no weights", kind, n.specs[i].name.c_str());
  if (B <= 0) return PCGC_OK;
  // the hyper nets work on 16^3 / 8^3 grids: a 32-cube sub-batch leaves most SMs idle, their activations are tiny
  const bool small_net = kind == PCGC_NET_HYPER_ENCODER || kind == PCGC_NET_HYPER_DECODER;
  const int SB = std::min(B, small_net ? 8 * ctx->sub_batch : ctx->sub_batch);
  for (int bi = BUF_X0; bi < BUF_OUT0; ++bi) {
    size_t e = n.elems[bi];
    if (bi == BUF_X0 && cubes) e = std::max(e, (size_t)n.in_n * n.in_n * n.in_n * n.in_c);
    if (e) { int r = ensure(ctx, &ctx->bufs[bi], &ctx->buf_cap[bi], e * SB); if (r) return r; }
  }
  const size_t in_elems = (size_t)n.in_n * n.in_n * n.in_n * n.in_c;
  // output sizes per cube
  size_t out_elems[2] = {0, 0};
  for (const Op& op : n.ops) {
    const LayerSpec& s = n.specs[op.layer];
    const int out_n = s.transposed ? op.in_n * s.stride : op.in_n / s.stride;
    if (op.out == BUF_OUT0) out_elems[0] = (size_t)out_n * out_n * out_n * op.out_cs;
    if (op.out == BUF_OUT1) out_elems[1] = (size_t)out_n * out_n * out_n * op.out_cs;
  }
  for (int b0 = 0; b0 < B; b0 += SB) {
    const int nb = std::min(SB, B - b0);
    float* ptr[BUF_COUNT];
    for (int i = 0; i < BUF_COUNT; ++i) ptr[i] = ctx->bufs[i];
    ptr[BUF_OUT0] = out0 ? out0 + (size_t)b0 * out_elems[0] : nullptr;
    ptr[BUF_OUT1] = out1 ? out1 + (size_t)b0 * out_elems[1] : nullptr;
    if (cubes) {
      const size_t esz = cubes_dtype == PCGC_DTYPE_U8 ? 1 : (cubes_dtype == PCGC_DTYPE_F32 ? 4 : 8);
      CK(launch_u8_to_f32((const char*)cubes + (size_t)b0 * in_elems * esz, cubes_dtype, ctx->bufs[BUF_X0],
                          (int64_t)nb * in_elems, ctx->stream, &ctx->launches));
      ptr[BUF_IN] = ctx->bufs[BUF_X0];
    } else {
      ptr[BUF_IN] = const_cast<float*>(in_ext) + (size_t)b0 * in_elems;
    }
    for (const Op& op : n.ops) {
      const LayerSpec& s = n.specs[op.layer];
      LayerW& lw = n.w[op.layer];
      const int out_n = s.transposed ? op.in_n * s.stride : op.in_n / s.stride;
      ConvCall c;
      c.in = ptr[op.in]; c.in_n = op.in_n; c.in_cs = op.in_cs; c.in_co = op.in_co;
      c.out = ptr[op.out]; c.out_n = out_n; c.out_cs = op.out_cs; c.out_co = op.out_co;
      c.bias = lw.bias;
      c.res = op.res >= 0 ? ptr[op.res] : nullptr; c.res_cs = op.res_cs; c.res_co = op.res_co;
      c.flags = op.flags; c.floor_v = floor_v;
      c.B = nb;
      if (!c.out) return fail(ctx, PCGC_ERR_BAD_ARG, "net %d: missing output pointer", kind);
      bool done = false;
      char tag[96];
      const double flops = 2.0 * nb * (double)(s.transposed ? op.in_n : out_n) * (s.transposed ? op.in_n : out_n) *
                           (s.transposed ? op.in_n : out_n) * s.k * s.k * s.k * s.cin * s.cout;
      if (!done) {
        snprintf(tag, sizeof tag, "conv_ffma k%d s%d%s c%d->%d n%d", s.k, s.stride, s.transposed ? "T" : "", s.cin, s.cout, op.in_n);
        prof_begin(ctx, tag, flops, 0);
        for (int k = 0; k < lw.n_classes; ++k) {
          c.d = lw.cls[k];
          c.tn = s.transposed ? op.in_n : out_n;
          cudaError_t e = launch_conv_ffma(c, ctx->stream, &ctx->launches);
          if (e != cudaSuccess) return fail(ctx, PCGC_ERR_CUDA, "conv '%s': %s", s.name.c_str(), cudaGetErrorString(e));
        }
        prof_end(ctx);
      }
    }
  }
  return PCGC_OK;
}

}  // namespace

// ---- accessors for train.cu (the ctx layout stays private to this file) ----
namespace pcgc {
cudaStream_t ctx_stream(pcgc_ctx* c) { return c->stream; }
int64_t* ctx_launches(pcgc_ctx* c) { return &c->launches; }
int ctx_device(pcgc_ctx* c) { return c->device; }
int* ctx_err_flag(pcgc_ctx* c) { return c->err_flag; }
int ctx_fail(pcgc_ctx* c, int code, const char* msg) { return fail(c, code, "%s", msg); }
float* ctx_workspace(pcgc_ctx* c, int slot, size_t floats) {
  if (slot < 0 || slot > 3) return nullptr;
  if (c->train_cap[slot] < floats) {
    if (c->train_ws[slot]) { cudaStreamSynchronize(c->stream); cudaFree(c->train_ws[slot]); c->train_ws[slot] = nullptr; c->train_cap[slot] = 0; }
    const size_t want = floats + floats / 4 + 1024;
    if (cudaMalloc((void**)&c->train_ws[slot], want * sizeof(float)) != cudaSuccess) return nullptr;
    c->train_cap[slot] = want;
  }
  return c->train_ws[slot];
}
void ctx_prof_begin(pcgc_ctx* c, const char* tag, double flops, double bytes) { prof_begin(c, tag, flops, bytes); }
void ctx_prof_end(pcgc_ctx* c) { prof_end(c); }
MeshWorkspace** ctx_mesh_workspace(pcgc_ctx* c) { return &c->mesh_ws; }
}  // namespace pcgc

extern "C" {

int pcgc_create(pcgc_ctx** out, int device) {
  if (!out) return PCGC_ERR_BAD_ARG;
  *out = nullptr;
  int count = 0;
  if (cudaGetDeviceCount(&count) != cudaSuccess || device < 0 || device >= count) return PCGC_ERR_CUDA;
  pcgc_ctx* ctx = new pcgc_ctx();
  ctx->device = device;
  DeviceGuard g(device);
  cudaDeviceProp prop;
  if (cudaGetDeviceProperties(&prop, device) != cudaSuccess || prop.major != 10) {
    // sm_100a SASS only: refuse loudly instead of failing at the first launch
    delete ctx;
    return PCGC_ERR_CUDA;
  }
  for (int k = 0; k < PCGC_NET_COUNT; ++k) build_net(ctx->nets[k], k);
  if (const char* sb = getenv("PCGC_SUB_BATCH")) { const int v = atoi(sb); if (v >= 1 && v <= 512) ctx->sub_batch = v; }
  if (cudaMalloc((void**)&ctx->err_flag, sizeof(int)) != cudaSuccess ||
      cudaMemset(ctx->err_flag, 0, sizeof(int)) != cudaSuccess ||
      cudaMalloc((void**)&ctx->pmf_dev, 32 * 512 * sizeof(float)) != cudaSuccess) {
    delete ctx;
    return PCGC_ERR_CUDA;
  }
  *out = ctx;
  return PCGC_OK;
}

void pcgc_destroy(pcgc_ctx* ctx) {
  if (!ctx) return;
  DeviceGuard g(ctx->device);
  cudaDeviceSynchronize();
  for (int i = 0; i < BUF_COUNT; ++i) if (ctx->bufs[i]) cudaFree(ctx->bufs[i]);
  for (auto& n : ctx->nets) {
    for (int i = 0; i < 9; ++i) { free_umma_weights(n.up.ka[i]); free_umma_weights(n.up.kb[i]); }
    free_umma_weights(n.up.first); free_umma_weights(n.up.last);
    for (int u = 0; u < 2; ++u) for (int g = 0; g < 2; ++g) free_umma_weights(n.up.up[u][g]);
    free_umma_weights(n.up.down[0]); free_umma_weights(n.up.down[1]);
    if (n.up.conv_in_w) cudaFree(n.up.conv_in_w);
    free_win_layer(n.up.s_conv1); free_win_layer(n.up.s_conv2); free_win_layer(n.up.s_conv3); free_win_layer(n.up.s_deconv3);
    free_win_layer(n.up.h_deconv1); free_win_layer(n.up.h_deconv2[0]); free_win_layer(n.up.h_deconv2[1]);
    for (int g2 = 0; g2 < 4; ++g2) { free_win_layer(n.up.s_deconv1[g2]); free_win_layer(n.up.s_deconv2[g2]); }
  }
  for (auto& n : ctx->nets)
    for (auto& lw : n.w) {
      for (int k = 0; k < lw.n_classes; ++k) if (lw.cls[k].w) cudaFree((void*)lw.cls[k].w);
      if (lw.bias) cudaFree(lw.bias);
      free_umma_weights(lw.umma);
    }
  for (auto& b : ctx->bn) if (b.params) cudaFree(b.params);
  free_geometry_workspace(ctx->geo_ws);
  free_mesh_workspace(ctx->mesh_ws);
  if (ctx->ff_zero) cudaFree(ctx->ff_zero);
  if (ctx->ff_y) cudaFree(ctx->ff_y);
  for (auto e : ctx->ff_e) if (e) cudaFree(e);
  if (ctx->ff_rows) cudaFree(ctx->ff_rows);
  if (ctx->ff_masks) cudaFree(ctx->ff_masks);
  if (ctx->ff_prev) cudaFree(ctx->ff_prev);
  if (ctx->ff_lists) cudaFree(ctx->ff_lists);
  for (auto a : ctx->ff_act) if (a) cudaFree(a);
  if (ctx->scratch) cudaFree(ctx->scratch);
  if (ctx->pmf_dev) cudaFree(ctx->pmf_dev);
  if (ctx->err_flag) cudaFree(ctx->err_flag);
  if (ctx->mm_dev) cudaFree(ctx->mm_dev);
  if (ctx->off_dev) cudaFree(ctx->off_dev);
  if (ctx->chunk_dev) cudaFree(ctx->chunk_dev);
  for (auto p : ctx->train_ws) if (p) cudaFree(p);
  for (auto& r : ctx->prof) { cudaEventDestroy(r.a); cudaEventDestroy(r.b); }
  for (auto e : ctx->ev_pool) cudaEventDestroy(e);
  delete ctx;
}

const char* pcgc_last_error(const pcgc_ctx* ctx) { return ctx ? ctx->err.c_str() : "null ctx"; }

int pcgc_set_stream(pcgc_ctx* ctx, void* stream) {
  if (!ctx) return PCGC_ERR_BAD_ARG;
  ctx->stream = (cudaStream_t)stream;
  return PCGC_OK;
}

int pcgc_set_engine(pcgc_ctx* ctx, int engine) {
  if (!ctx || engine < 0 || engine > 2) return PCGC_ERR_BAD_ARG;
  ctx->engine = engine;
  return PCGC_OK;
}

int64_t pcgc_launch_count(const pcgc_ctx* ctx) { return ctx ? ctx->launches : 0; }

int pcgc_profile_enable(pcgc_ctx* ctx, int on) {
  if (!ctx) return PCGC_ERR_BAD_ARG;
  ctx->profiling = on != 0;
  return PCGC_OK;
}

int pcgc_profile_report(pcgc_ctx* ctx, char* buf, int64_t cap) {
  if (!ctx || !buf || cap < 3) return PCGC_ERR_BAD_ARG;
  DeviceGuard g(ctx->device);
  CK(cudaStreamSynchronize(ctx->stream));
  struct Agg { std::string tag; int count; double ms, flops, bytes; };
  std::vector<Agg> aggs;
  if (getenv("PCGC_PROF_TIMELINE") && !ctx->prof.empty()) {
    // dev form (tools/timeline.py): one entry per record with its start relative to the first record, so that the gaps
    // between launches and the overlap of the streams can be read off
    std::string out = "[";
    for (size_t i = 0; i < ctx->prof.size(); ++i) {
      auto& r = ctx->prof[i];
      float t0 = 0.f, ms = 0.f;
      cudaEventSynchronize(r.b);
      cudaEventElapsedTime(&t0, ctx->prof[0].a, r.a);
      cudaEventElapsedTime(&ms, r.a, r.b);
      char line[256];
      snprintf(line, sizeof line, "%s{\"tag\":\"%s\",\"count\":1,\"t0\":%.4f,\"ms\":%.4f,\"flops\":%.6e,\"bytes\":%.6e}", i ? "," : "",
               r.tag.c_str(), t0, ms, r.flops, r.bytes);
      out += line;
    }
    out += "]";
    for (auto& r : ctx->prof) { ctx->ev_pool.push_back(r.a); ctx->ev_pool.push_back(r.b); }
    ctx->prof.clear();
    if ((int64_t)out.size() + 1 > cap) return fail(ctx, PCGC_ERR_OVERFLOW, "profile report needs %zu bytes", out.size() + 1);
    memcpy(buf, out.c_str(), out.size() + 1);
    return PCGC_OK;
  }
  for (auto& r : ctx->prof) {
    float ms = 0.f;
    cudaEventElapsedTime(&ms, r.a, r.b);
    Agg* a = nullptr;
    for (auto& x : aggs) if (x.tag == r.tag) { a = &x; break; }
    if (!a) { aggs.push_back({r.tag, 0, 0, 0, 0}); a = &aggs.back(); }
    a->count++; a->ms += ms; a->flops += r.flops; a->bytes += r.bytes;
    ctx->ev_pool.push_back(r.a); ctx->ev_pool.push_back(r.b);
  }
  ctx->prof.clear();
  std::string out = "[";
  for (size_t i = 0; i < aggs.size(); ++i) {
    char line[256];
    snprintf(line, sizeof line, "%s{\"tag\":\"%s\",\"count\":%d,\"ms\":%.6f,\"flops\":%.6e,\"bytes\":%.6e}", i ? "," : "",
             aggs[i].tag.c_str(), aggs[i].count, aggs[i].ms, aggs[i].flops, aggs[i].bytes);
    out += line;
  }
  out += "]";
  if ((int64_t)out.size() + 1 > cap) return fail(ctx, PCGC_ERR_OVERFLOW, "profile report needs %zu bytes", out.size() + 1);
  memcpy(buf, out.c_str(), out.size() + 1);
  return PCGC_OK;
}

int pcgc_synchronize(pcgc_ctx* ctx) {
  if (!ctx) return PCGC_ERR_BAD_ARG;
  DeviceGuard g(ctx->device);
  return check_err_flag(ctx, "pcgc_synchronize", true);      // also surfaces device-side timeouts of the tcgen05 engine
}

int pcgc_load_conv(pcgc_ctx* ctx, int net, const char* layer, const float* kernel, const int64_t kshape[5],
                   const float* bias) {
  if (!ctx || net < 0 || net >= PCGC_NET_COUNT || !layer || !kernel || !kshape) return fail(ctx, PCGC_ERR_BAD_ARG, "pcgc_load_conv: bad argument");
  DeviceGuard g(ctx->device);
  Net& n = ctx->nets[net];
  const int li = n.find(layer);
  if (li < 0) return fail(ctx, PCGC_ERR_BAD_ARG, "net %d has no layer '%s'", net, layer);
  const LayerSpec& s = n.specs[li];
  const int k = s.k;
  const int64_t want[5] = {k, k, k, s.transposed ? s.cout : s.cin, s.transposed ? s.cin : s.cout};
  for (int i = 0; i < 5; ++i)
    if (kshape[i] != want[i]) return fail(ctx, PCGC_ERR_BAD_ARG, "layer '%s': kernel dim %d is %lld, expected %lld", layer, i, (long long)kshape[i], (long long)want[i]);
  if ((bias != nullptr) != s.bias) return fail(ctx, PCGC_ERR_BAD_ARG, "layer '%s': use_bias=%d in the reference", layer, (int)s.bias);
  LayerW& lw = n.w[li];
  CK(cudaStreamSynchronize(ctx->stream));
  lw.hk.assign(kernel, kernel + (size_t)k * k * k * s.cin * s.cout);
  if (bias) lw.hb.assign(bias, bias + s.cout); else lw.hb.clear();
  n.up.ready = false;
  if (net == PCGC_NET_VOX_ANALYSIS) ctx->ff_ready = ctx->ff_known = false;   // the empty cube's activations and the slots belong to the old weights
  if (n.up.conv_in_w) { cudaFree(n.up.conv_in_w); n.up.conv_in_w = nullptr; }
  for (int c = 0; c < lw.n_classes; ++c) if (lw.cls[c].w) { cudaFree((void*)lw.cls[c].w); lw.cls[c].w = nullptr; }
  if (lw.bias) { cudaFree(lw.bias); lw.bias = nullptr; }
  free_umma_weights(lw.umma);
  lw.loaded = false;

  auto K = [&](int kz, int ky, int kx, int ci, int co) -> float {   // value of tap (kz,ky,kx) from ci to co
    if (s.transposed) return kernel[((((size_t)kz * k + ky) * k + kx) * s.cout + co) * s.cin + ci];
    return kernel[((((size_t)kz * k + ky) * k + kx) * s.cin + ci) * s.cout + co];
  };
  std::vector<float> packed;
  if (!s.transposed) {
    lw.n_classes = 1;
    ConvDesc& d = lw.cls[0];
    d.kz = d.ky = d.kx = k; d.stride = s.stride;
    d.pz = d.py = d.px = same_pad_before(k, s.stride);
    d.ostride = 1; d.oz = d.oy = d.ox = 0; d.cin = s.cin; d.cout = s.cout;
    packed.resize((size_t)k * k * k * s.cin * s.cout);
    for (int ky = 0; ky < k; ++ky) for (int kx = 0; kx < k; ++kx) for (int ci = 0; ci < s.cin; ++ci)
      for (int kz = 0; kz < k; ++kz) for (int co = 0; co < s.cout; ++co)
        packed[((((size_t)ky * k + kx) * s.cin + ci) * k + kz) * s.cout + co] = K(kz, ky, kx, ci, co);
    float* dw = nullptr;
    CK(cudaMalloc((void**)&dw, packed.size() * sizeof(float)));
    CK(cudaMemcpy(dw, packed.data(), packed.size() * sizeof(float), cudaMemcpyHostToDevice));
    d.w = dw;
  } else {
    // stride-2 Conv3DTranspose = 8 output-parity classes, each a stride-1 gather conv over the input grid
    const int pb = same_pad_before(k, 2);
    if (s.cout == 1) {
      // One output channel (model_simple deconv_3, k9): the 8 classes become the 8 "output channels" of ONE conv over the union
      // tap box, so the input brick is staged once instead of 8 times and every staged value feeds 8 FMAs instead of 1
      // (r01: 15.4 ms -> per 64 cubes for this layer alone as 8 single-channel launches).
      int km[2], q0[2], o0[2], P[2];
      for (int r = 0; r < 2; ++r) {
        km[r] = (k - r + 1) / 2;
        q0[r] = std::max(0, (pb - r + 1) / 2);
        o0[r] = 2 * q0[r] + r - pb;
        P[r] = (km[r] - 1) - q0[r];
      }
      const int PU = std::max(P[0], P[1]);
      const int KM = std::max(km[0] + PU - P[0], km[1] + PU - P[1]);
      lw.n_classes = 1;
      ConvDesc& d = lw.cls[0];
      d.kz = d.ky = d.kx = KM; d.stride = 1; d.pz = d.py = d.px = PU;
      d.ostride = 2; d.oz = d.oy = d.ox = 0; d.cin = s.cin; d.cout = 8;
      d.class_mode = 1; d.cls_o0[0] = o0[0]; d.cls_o0[1] = o0[1];
      packed.assign((size_t)KM * KM * KM * s.cin * 8, 0.f);
      for (int cls = 0; cls < 8; ++cls) {
        const int r[3] = {(cls >> 2) & 1, (cls >> 1) & 1, cls & 1};
        for (int jz = 0; jz < km[r[0]]; ++jz) for (int jy = 0; jy < km[r[1]]; ++jy) for (int jx = 0; jx < km[r[2]]; ++jx) {
          const int uz = jz + PU - P[r[0]], uy = jy + PU - P[r[1]], ux = jx + PU - P[r[2]];
          const int kz = r[0] + 2 * (km[r[0]] - 1 - jz), ky = r[1] + 2 * (km[r[1]] - 1 - jy), kx = r[2] + 2 * (km[r[2]] - 1 - jx);
          for (int ci = 0; ci < s.cin; ++ci)
            packed[((((size_t)uy * KM + ux) * s.cin + ci) * KM + uz) * 8 + cls] = K(kz, ky, kx, ci, 0);
        }
      }
      float* dw = nullptr;
      CK(cudaMalloc((void**)&dw, packed.size() * sizeof(float)));
      CK(cudaMemcpy(dw, packed.data(), packed.size() * sizeof(float), cudaMemcpyHostToDevice));
      d.w = dw;
    } else {
    lw.n_classes = 8;
    for (int cls = 0; cls < 8; ++cls) {
      const int r[3] = {(cls >> 2) & 1, (cls >> 1) & 1, cls & 1};   // parity of (o+pb) per axis z,y,x
      int km[3], q0[3], o0[3], P[3];
      for (int a = 0; a < 3; ++a) {
        km[a] = (k - r[a] + 1) / 2;
        q0[a] = std::max(0, (pb - r[a] + 1) / 2);
        o0[a] = 2 * q0[a] + r[a] - pb;
        P[a] = (km[a] - 1) - q0[a];
      }
      ConvDesc& d = lw.cls[cls];
      d.kz = km[0]; d.ky = km[1]; d.kx = km[2]; d.stride = 1;
      d.pz = P[0]; d.py = P[1]; d.px = P[2];
      d.ostride = 2; d.oz = o0[0]; d.oy = o0[1]; d.ox = o0[2]; d.cin = s.cin; d.cout = s.cout;
      packed.assign((size_t)km[0] * km[1] * km[2] * s.cin * s.cout, 0.f);
      for (int jy = 0; jy < km[1]; ++jy) for (int jx = 0; jx < km[2]; ++jx) for (int ci = 0; ci < s.cin; ++ci)
        for (int jz = 0; jz < km[0]; ++jz) for (int co = 0; co < s.cout; ++co) {
          const int kz = r[0] + 2 * (km[0] - 1 - jz), ky = r[1] + 2 * (km[1] - 1 - jy), kx = r[2] + 2 * (km[2] - 1 - jx);
          packed[((((size_t)jy * km[2] + jx) * s.cin + ci) * km[0] + jz) * s.cout + co] = K(kz, ky, kx, ci, co);
        }
      float* dw = nullptr;
      CK(cudaMalloc((void**)&dw, packed.size() * sizeof(float)));
      CK(cudaMemcpy(dw, packed.data(), packed.size() * sizeof(float), cudaMemcpyHostToDevice));
      d.w = dw;
    }
    }
  }
  if (bias) {
    CK(cudaMalloc((void**)&lw.bias, s.cout * sizeof(float)));
    CK(cudaMemcpy(lw.bias, bias, s.cout * sizeof(float), cudaMemcpyHostToDevice));
  }
  lw.loaded = true;
  return PCGC_OK;
}

int pcgc_load_bottleneck(pcgc_ctx* ctx, int slot, int channels, const float* matrices, const float* biases,
                         const float* factors) {
  if (!ctx || slot < 0 || slot > 1 || channels < 1 || channels > 512 || !matrices || !biases || !factors)
    return fail(ctx, PCGC_ERR_BAD_ARG, "pcgc_load_bottleneck: bad argument");
  DeviceGuard g(ctx->device);
  const int C = channels;
  // input: matrix_0 [C,3,1], matrix_1 [C,3,3], matrix_2 [C,3,3], matrix_3 [C,1,3]; bais/factor [C,3,1]x3,[C,1,1]
  const float* m[4] = {matrices, matrices + 3 * C, matrices + 12 * C, matrices + 21 * C};
  const float* bb[4] = {biases, biases + 3 * C, biases + 6 * C, biases + 9 * C};
  const float* ff[4] = {factors, factors + 3 * C, factors + 6 * C, factors + 9 * C};
  auto softplus = [](float x) -> float {   // tf.nn.softplus in float32 (entropy_model.py:87)
    if (x > 20.f) return x;
    if (x < -20.f) return expf(x);
    return log1pf(expf(x));
  };
  std::vector<float> p((size_t)C * 44);
  for (int c = 0; c < C; ++c) {
    float* q = p.data() + (size_t)c * 44;
    for (int j = 0; j < 3; ++j) { q[j] = softplus(m[0][c * 3 + j]); q[3 + j] = bb[0][c * 3 + j]; q[6 + j] = tanhf(ff[0][c * 3 + j]); }
    q += 9;
    for (int l = 1; l <= 2; ++l) {
      for (int j = 0; j < 9; ++j) q[j] = softplus(m[l][c * 9 + j]);
      for (int j = 0; j < 3; ++j) { q[9 + j] = bb[l][c * 3 + j]; q[12 + j] = tanhf(ff[l][c * 3 + j]); }
      q += 15;
    }
    for (int j = 0; j < 3; ++j) q[j] = softplus(m[3][c * 3 + j]);
    q[3] = bb[3][c]; q[4] = tanhf(ff[3][c]);
  }
  BottleneckDev& bn = ctx->bn[slot];
  CK(cudaStreamSynchronize(ctx->stream));
  if (bn.params) { cudaFree(bn.params); bn.params = nullptr; }
  CK(cudaMalloc((void**)&bn.params, p.size() * sizeof(float)));
  CK(cudaMemcpy(bn.params, p.data(), p.size() * sizeof(float), cudaMemcpyHostToDevice));
  bn.channels = C;
  ctx->bn_host[slot] = p;
  return PCGC_OK;
}

int pcgc_debug_conv3_umma(pcgc_ctx* ctx, const float* in_dev, int n, int cin, int cout, const float* kernel_host,
                          const float* bias_host, int relu, int B, int wt, float* out_dev) {
  if (!ctx || !in_dev || !kernel_host || !out_dev || B < 1) return fail(ctx, PCGC_ERR_BAD_ARG, "pcgc_debug_conv3_umma: bad argument");
  DeviceGuard g(ctx->device);
  UmmaWeights w;
  cudaError_t e = pack_umma_weights_dense(kernel_host, bias_host, cin, cout, w, 27, wt < 1 ? 1 : wt);
  if (e != cudaSuccess) return fail(ctx, PCGC_ERR_BAD_ARG, "pack_umma_weights_dense: %s", cudaGetErrorString(e));
  PmTensor t; t.n = n; t.c = cin; t.B = B;
  CK(cudaMalloc((void**)&t.p, t.cube_elems() * B * sizeof(__nv_bfloat16)));
  CK(launch_f32_to_pm(in_dev, cin, 0, t, ctx->stream, &ctx->launches));
  UmmaCall c; c.in = t; c.epi = UEPI_F32; c.flags = relu ? EPI_RELU : 0; c.out_f32 = out_dev; c.out_cs = cout; c.out_co = 0;
  c.err = ctx->err_flag;
  e = launch_conv_umma_pm(c, w, ctx->stream, &ctx->launches);
  cudaError_t e2 = cudaStreamSynchronize(ctx->stream);
  cudaFree(t.p);
  free_umma_weights(w);
  if (e != cudaSuccess) return fail(ctx, PCGC_ERR_CUDA, "launch_conv_umma_pm: %s", cudaGetErrorString(e));
  if (e2 != cudaSuccess) return fail(ctx, PCGC_ERR_CUDA, "conv_umma kernel: %s", cudaGetErrorString(e2));
  return check_err_flag(ctx, "pcgc_debug_conv3_umma");
}

int pcgc_analysis(pcgc_ctx* ctx, int net, const void* cubes_dev, int dtype, int B, float* y_dev) {
  if (!ctx || !cubes_dev || !y_dev || (net != PCGC_NET_VOX_ANALYSIS && net != PCGC_NET_SIMPLE_ANALYSIS) || dtype < 0 || dtype > 2)
    return fail(ctx, PCGC_ERR_BAD_ARG, "pcgc_analysis: bad argument");
  DeviceGuard g(ctx->device);
  if (net == PCGC_NET_VOX_ANALYSIS && ctx->engine != PCGC_ENGINE_FFMA) return run_vox_umma(ctx, net, nullptr, cubes_dev, dtype, B, y_dev);
  if (net == PCGC_NET_SIMPLE_ANALYSIS && ctx->engine != PCGC_ENGINE_FFMA) return run_simple_umma(ctx, net, nullptr, cubes_dev, dtype, B, y_dev);
  return run_net(ctx, net, nullptr, cubes_dev, dtype, B, y_dev, nullptr, 0.f);
}

int pcgc_synthesis(pcgc_ctx* ctx, int net, const float* y_dev, int B, float* logits_dev) {
  if (!ctx || !y_dev || !logits_dev || (net != PCGC_NET_VOX_SYNTHESIS && net != PCGC_NET_SIMPLE_SYNTHESIS))
    return fail(ctx, PCGC_ERR_BAD_ARG, "pcgc_synthesis: bad argument");
  DeviceGuard g(ctx->device);
  if (net == PCGC_NET_VOX_SYNTHESIS && ctx->engine != PCGC_ENGINE_FFMA) return run_vox_umma(ctx, net, y_dev, nullptr, 0, B, logits_dev);
  if (net == PCGC_NET_SIMPLE_SYNTHESIS && ctx->engine != PCGC_ENGINE_FFMA) return run_simple_umma(ctx, net, y_dev, nullptr, 0, B, logits_dev);
  return run_net(ctx, net, y_dev, nullptr, 0, B, logits_dev, nullptr, 0.f);
}

int pcgc_hyper_encode(pcgc_ctx* ctx, const float* y_dev, int B, float* z_dev) {
  if (!ctx || !y_dev || !z_dev) return fail(ctx, PCGC_ERR_BAD_ARG, "pcgc_hyper_encode: bad argument");
  DeviceGuard g(ctx->device);
  if (ctx->engine != PCGC_ENGINE_FFMA) return run_hyper_umma(ctx, PCGC_NET_HYPER_ENCODER, y_dev, B, z_dev, nullptr, 0.f);
  return run_net(ctx, PCGC_NET_HYPER_ENCODER, y_dev, nullptr, 0, B, z_dev, nullptr, 0.f);
}

int pcgc_hyper_decode(pcgc_ctx* ctx, const float* z_hat_dev, int B, float scale_floor, float* loc_dev, float* scale_dev) {
  if (!ctx || !z_hat_dev || !loc_dev || !scale_dev) return fail(ctx, PCGC_ERR_BAD_ARG, "pcgc_hyper_decode: bad argument");
  DeviceGuard g(ctx->device);
  // ONE fixed program whatever pcgc_set_engine / the PCGC_UMMA_* tuning switches say: loc and scale become integer CDF tables,
  // and a last-bit difference between the encoding and the decoding process desynchronises the range decoder.
  return run_hyper_umma(ctx, PCGC_NET_HYPER_DECODER, z_hat_dev, B, loc_dev, scale_dev, scale_floor);
}

int pcgc_factorized_quantize_likelihood(pcgc_ctx* ctx, int slot, const float* x_dev, int64_t n_vox, int C,
                                        float likelihood_bound, float* x_hat_dev, float* p_dev, double* bits_dev,
                                        int32_t* minmax_dev) {
  if (!ctx || slot < 0 || slot > 1 || !x_dev || n_vox < 0) return fail(ctx, PCGC_ERR_BAD_ARG, "pcgc_factorized_quantize_likelihood: bad argument");
  DeviceGuard g(ctx->device);
  if (!ctx->bn[slot].params) return fail(ctx, PCGC_ERR_NOT_READY, "bottleneck slot %d not loaded", slot);
  if (C != ctx->bn[slot].channels || C % 4) return fail(ctx, PCGC_ERR_BAD_ARG, "channels %d != loaded %d (must be a multiple of 4)", C, ctx->bn[slot].channels);
  if (n_vox == 0) return PCGC_OK;
  int r = ensure_scratch(ctx, 148 * 8 + 8); if (r) return r;
  prof_begin(ctx, "factorized_quantize_likelihood", 0, 4.0 * n_vox * C * (1 + (x_hat_dev != nullptr) + (p_dev != nullptr)));
  CK(launch_factorized(ctx->bn[slot], x_dev, n_vox, C, likelihood_bound, x_hat_dev, p_dev, bits_dev, minmax_dev,
                       ctx->scratch, ctx->stream, &ctx->launches, ctx->quant_noise, ctx->quant_seed));
  prof_end(ctx);
  return PCGC_OK;
}

int pcgc_factorized_cdf(pcgc_ctx* ctx, int slot, int min_v, int max_v, float likelihood_bound, int precision,
                        int32_t* cdf_host) {
  if (!ctx || slot < 0 || slot > 1 || !cdf_host) return fail(ctx, PCGC_ERR_BAD_ARG, "pcgc_factorized_cdf: bad argument");
  DeviceGuard g(ctx->device);
  const BottleneckDev& bn = ctx->bn[slot];
  if (!bn.params) return fail(ctx, PCGC_ERR_NOT_READY, "bottleneck slot %d not loaded", slot);
  const int N = max_v - min_v + 1;
  if (N < 2) return fail(ctx, PCGC_ERR_BAD_RANGE, "single-symbol alphabet [%d,%d]: pmf_to_quantized_cdf needs >= 2 symbols (entropy_model.py:192-193)", min_v, max_v);
  if ((size_t)N * bn.channels > 32 * 512) return fail(ctx, PCGC_ERR_BAD_RANGE, "symbol range too large");
  CK(launch_factorized_pmf(bn, min_v, max_v, likelihood_bound, ctx->pmf_dev, ctx->stream, &ctx->launches));
  std::vector<float> pmf((size_t)N * bn.channels);
  CK(cudaMemcpyAsync(pmf.data(), ctx->pmf_dev, pmf.size() * sizeof(float), cudaMemcpyDeviceToHost, ctx->stream));
  int r = check_err_flag(ctx, "pcgc_factorized_cdf (earlier kernels on this stream)", true);     // synchronises; surfaces tcgen05 timeouts of the transforms
  if (r) return r;
  r = pcgc_pmf_to_quantized_cdf(pmf.data(), bn.channels, N, precision, cdf_host);
  if (r) return fail(ctx, r, "pmf_to_quantized_cdf failed");
  return PCGC_OK;
}

int pcgc_laplace_quantize_likelihood(pcgc_ctx* ctx, const float* y_dev, const float* loc_dev, const float* scale_dev,
                                     int B, int64_t E, float likelihood_bound, float* y_hat_dev, float* p_dev,
                                     double* bits_dev, int32_t* minmax_dev) {
  if (!ctx || !y_dev || !loc_dev || !scale_dev || B < 0 || E <= 0 || E % 4) return fail(ctx, PCGC_ERR_BAD_ARG, "pcgc_laplace_quantize_likelihood: bad argument");
  DeviceGuard g(ctx->device);
  if (B == 0) return PCGC_OK;
  int r = ensure_scratch(ctx, (size_t)B * 16 + 8); if (r) return r;
  prof_begin(ctx, "laplace_quantize_likelihood", 0, 4.0 * B * E * (3 + (y_hat_dev != nullptr) + (p_dev != nullptr)));
  CK(launch_laplace(y_dev, loc_dev, scale_dev, B, E, likelihood_bound, y_hat_dev, p_dev, bits_dev, minmax_dev,
                    ctx->scratch, ctx->stream, &ctx->launches, ctx->quant_noise, ctx->quant_seed + 0x9E3779B97F4A7C15ull));
  prof_end(ctx);
  return PCGC_OK;
}

int pcgc_laplace_intervals(pcgc_ctx* ctx, const float* y_hat_dev, const float* loc_dev, const float* scale_dev, int B,
                           int64_t E, const int32_t* minmax_dev, float likelihood_bound, int precision,
                           uint32_t* intervals_dev) {
  if (!ctx || !y_hat_dev || !loc_dev || !scale_dev || !minmax_dev || !intervals_dev || B < 0 || precision != 16)
    return fail(ctx, PCGC_ERR_BAD_ARG, "pcgc_laplace_intervals: bad argument (precision must be 16)");
  DeviceGuard g(ctx->device);
  if (B == 0) return PCGC_OK;
  prof_begin(ctx, "laplace_intervals", 0, 4.0 * B * E * 4);
  CK(launch_laplace_intervals(y_hat_dev, loc_dev, scale_dev, B, E, minmax_dev, likelihood_bound, precision,
                              intervals_dev, ctx->err_flag, ctx->stream, &ctx->launches));
  prof_end(ctx);
  return check_err_flag(ctx, "pcgc_laplace_intervals");
}

int pcgc_laplace_cdf(pcgc_ctx* ctx, const float* loc_dev, const float* scale_dev, int B, int64_t E,
                     const int32_t* minmax_host, float likelihood_bound, int precision,
                     const int64_t* row_offset_host, uint16_t* cdf_dev) {
  if (!ctx || !loc_dev || !scale_dev || !minmax_host || !row_offset_host || !cdf_dev || B < 0 || precision != 16)
    return fail(ctx, PCGC_ERR_BAD_ARG, "pcgc_laplace_cdf: bad argument (precision must be 16)");
  DeviceGuard g(ctx->device);
  if (B == 0) return PCGC_OK;
  for (int b = 0; b < B; ++b) {
    const int N = minmax_host[2 * b + 1] - minmax_host[2 * b] + 1;
    if (N < 2 || N > PCGC_MAX_SYMBOLS) return fail(ctx, PCGC_ERR_BAD_RANGE, "cube %d: symbol range [%d,%d] unsupported", b, minmax_host[2 * b], minmax_host[2 * b + 1]);
  }
  if (ctx->mm_cap < (size_t)2 * B) {
    if (ctx->mm_dev) { CK(cudaStreamSynchronize(ctx->stream)); cudaFree(ctx->mm_dev); }
    CK(cudaMalloc((void**)&ctx->mm_dev, sizeof(int32_t) * 2 * B)); ctx->mm_cap = 2 * B;
  }
  if (ctx->off_cap < (size_t)B + 1) {
    if (ctx->off_dev) { CK(cudaStreamSynchronize(ctx->stream)); cudaFree(ctx->off_dev); }
    CK(cudaMalloc((void**)&ctx->off_dev, sizeof(int64_t) * (B + 1))); ctx->off_cap = B + 1;
  }
  CK(cudaMemcpyAsync(ctx->mm_dev, minmax_host, sizeof(int32_t) * 2 * B, cudaMemcpyHostToDevice, ctx->stream));
  CK(cudaMemcpyAsync(ctx->off_dev, row_offset_host, sizeof(int64_t) * (B + 1), cudaMemcpyHostToDevice, ctx->stream));
  prof_begin(ctx, "laplace_cdf", 0, 8.0 * B * E + 2.0 * (double)row_offset_host[B]);
  CK(launch_laplace_cdf(loc_dev, scale_dev, B, E, ctx->mm_dev, ctx->off_dev, likelihood_bound, precision, cdf_dev,
                        ctx->err_flag, ctx->stream, &ctx->launches));
  prof_end(ctx);
  // the host arrays were pageable: make sure the copies are done before the caller reuses them
  return check_err_flag(ctx, "pcgc_laplace_cdf");
}

int pcgc_debug_quantize_pmf(pcgc_ctx* ctx, const float* pmf_dev, int64_t rows, int N, int precision, int32_t* cdf_dev) {
  if (!ctx || !pmf_dev || !cdf_dev || rows < 0 || N < 2 || N > PCGC_MAX_SYMBOLS) return fail(ctx, PCGC_ERR_BAD_ARG, "pcgc_debug_quantize_pmf: bad argument");
  DeviceGuard g(ctx->device);
  if (rows == 0) return PCGC_OK;
  if (ctx->mm_cap < 2) { CK(cudaMalloc((void**)&ctx->mm_dev, sizeof(int32_t) * 2)); ctx->mm_cap = 2; }
  const int32_t mm[2] = {0, N - 1};
  CK(cudaMemcpyAsync(ctx->mm_dev, mm, sizeof mm, cudaMemcpyHostToDevice, ctx->stream));
  CK(launch_debug_quantize_pmf(pmf_dev, rows, ctx->mm_dev, precision, cdf_dev, ctx->err_flag, ctx->stream, &ctx->launches));
  return check_err_flag(ctx, "pcgc_debug_quantize_pmf");
}

int pcgc_topk_select(pcgc_ctx* ctx, const float* logits_dev, int B, int64_t V, const int32_t* ks_dev, uint8_t* mask_dev,
                     float* thres_dev, int32_t* count_dev) {
  if (!ctx || !logits_dev || !ks_dev || !mask_dev || B < 0 || V <= 0 || V % 4) return fail(ctx, PCGC_ERR_BAD_ARG, "pcgc_topk_select: bad argument");
  DeviceGuard g(ctx->device);
  if (B == 0) return PCGC_OK;
  prof_begin(ctx, "topk_select", 0, 5.0 * B * V);
  CK(launch_topk(logits_dev, B, V, ks_dev, mask_dev, thres_dev, count_dev, ctx->err_flag, ctx->stream, &ctx->launches));
  prof_end(ctx);
  return check_err_flag(ctx, "pcgc_topk_select");
}

int pcgc_threshold_select(pcgc_ctx* ctx, const float* logits_dev, int B, int64_t V, float thres, uint8_t* mask_dev,
                          int32_t* count_dev) {
  if (!ctx || !logits_dev || !mask_dev || B < 0 || V <= 0 || V % 4) return fail(ctx, PCGC_ERR_BAD_ARG, "pcgc_threshold_select: bad argument");
  DeviceGuard g(ctx->device);
  if (B == 0) return PCGC_OK;
  CK(launch_threshold(logits_dev, B, V, thres, mask_dev, count_dev, ctx->stream, &ctx->launches));
  return PCGC_OK;
}

int pcgc_voxelize(pcgc_ctx* ctx, const int16_t* local_dev, const int64_t* offsets_host, int B, int S, uint8_t* cubes_dev) {
  if (!ctx || !offsets_host || !cubes_dev || B < 0 || S < 1 || S > 1024) return fail(ctx, PCGC_ERR_BAD_ARG, "pcgc_voxelize: bad argument");
  DeviceGuard g(ctx->device);
  if (B == 0) return PCGC_OK;
  const int64_t n = offsets_host[B];
  if (n < 0 || (n > 0 && !local_dev)) return fail(ctx, PCGC_ERR_BAD_ARG, "pcgc_voxelize: bad offsets");
  if (ctx->chunk_cap < (size_t)(B + 1)) {
    if (ctx->chunk_dev) { CK(cudaStreamSynchronize(ctx->stream)); cudaFree(ctx->chunk_dev); ctx->chunk_dev = nullptr; ctx->chunk_cap = 0; }
    CK(cudaMalloc((void**)&ctx->chunk_dev, sizeof(int64_t) * (size_t)(B + 1))); ctx->chunk_cap = (size_t)(B + 1);
  }
  CK(cudaMemcpyAsync(ctx->chunk_dev, offsets_host, sizeof(int64_t) * (size_t)(B + 1), cudaMemcpyHostToDevice, ctx->stream));
  prof_begin(ctx, "voxelize", 0, 6.0 * n + (double)B * S * S * S);
  CK(launch_voxelize(local_dev, ctx->chunk_dev, B, S, n, cubes_dev, ctx->err_flag, ctx->stream, &ctx->launches));
  prof_end(ctx);
  return check_err_flag(ctx, "pcgc_voxelize");
}

int pcgc_extract_points(pcgc_ctx* ctx, const uint8_t* mask_dev, int B, int S, int32_t* counts_dev, int16_t* points_dev, int64_t cap,
                        int64_t* total_dev) {
  if (!ctx || !mask_dev || !counts_dev || !total_dev || (!points_dev && cap) || B < 0 || cap < 0 || S < 16 || S % 16 || S > 1024)
    return fail(ctx, PCGC_ERR_BAD_ARG, "pcgc_extract_points: bad argument (S must be a multiple of 16)");
  DeviceGuard g(ctx->device);
  if (B == 0) { CK(cudaMemsetAsync(total_dev, 0, sizeof(int64_t), ctx->stream)); return PCGC_OK; }
  const size_t n_chunks = (size_t)B * ((size_t)S * S * S / 4096);
  if (ctx->chunk_cap < n_chunks) {
    if (ctx->chunk_dev) { CK(cudaStreamSynchronize(ctx->stream)); cudaFree(ctx->chunk_dev); ctx->chunk_dev = nullptr; ctx->chunk_cap = 0; }
    CK(cudaMalloc((void**)&ctx->chunk_dev, sizeof(int64_t) * n_chunks)); ctx->chunk_cap = n_chunks;
  }
  prof_begin(ctx, "extract_points", 0, 2.0 * B * S * S * S);
  CK(launch_extract_points(mask_dev, B, S, ctx->chunk_dev, counts_dev, points_dev, cap, total_dev, ctx->stream, &ctx->launches));
  prof_end(ctx);
  return PCGC_OK;
}

int pcgc_geometry_sums(pcgc_ctx* ctx, const double* a_dev, int64_t n_a, const double* b_dev, int64_t n_b, const double* normals_a_dev,
                       double* out_dev) {
  if (!ctx || !a_dev || !b_dev || !out_dev || n_a <= 0 || n_b <= 0 || n_a > ((int64_t)1 << 27) || n_b > ((int64_t)1 << 27))
    return fail(ctx, PCGC_ERR_BAD_ARG, "pcgc_geometry_sums: bad argument (both sets need 1 .. 2^27 points)");
  DeviceGuard g(ctx->device);
  prof_begin(ctx, "geometry_grid", 0, 24.0 * (double)(n_a + n_b) + 32.0 * (double)(n_a + n_b));
  CK(launch_geometry_grids(&ctx->geo_ws, a_dev, n_a, b_dev, n_b, ctx->stream, &ctx->launches));
  prof_end(ctx);
  prof_begin(ctx, "geometry_query", 0, 2.0 * 32.0 * (double)(n_a + n_b) + (normals_a_dev ? 48.0 * (double)(n_a + n_b) : 0.0));
  CK(launch_geometry_queries(ctx->geo_ws, a_dev, b_dev, normals_a_dev, out_dev, ctx->stream, &ctx->launches));
  prof_end(ctx);
  return PCGC_OK;
}

int pcgc_estimate_normals(pcgc_ctx* ctx, const double* pts_dev, int64_t n, int k, double* normals_dev, int32_t* knn_idx_dev) {
  if (!ctx || !pts_dev || !normals_dev || n <= 0 || n > ((int64_t)1 << 27) || k < 1 || k > 64)
    return fail(ctx, PCGC_ERR_BAD_ARG, "pcgc_estimate_normals: bad argument (1 .. 2^27 points, 1 <= k <= 64)");
  DeviceGuard g(ctx->device);
  prof_begin(ctx, "normals_grid", 0, 24.0 * (double)n + 32.0 * (double)n);
  CK(launch_normals_grid(&ctx->geo_ws, pts_dev, n, ctx->stream, &ctx->launches));
  prof_end(ctx);
  const int kk = (int)std::min<int64_t>(k, n);
  prof_begin(ctx, "normals_query", 0, (double)n * (32.0 + 2.0 * 24.0 * kk + 24.0 + (knn_idx_dev ? 4.0 * k : 0.0)));
  CK(launch_normals_query(ctx->geo_ws, pts_dev, n, k, normals_dev, knn_idx_dev, ctx->stream, &ctx->launches));
  prof_end(ctx);
  return PCGC_OK;
}

int pcgc_widen_symbol_ranges(pcgc_ctx* ctx, int32_t* minmax_dev, int n_pairs) {
  if (!ctx || !minmax_dev || n_pairs < 0) return fail(ctx, PCGC_ERR_BAD_ARG, "pcgc_widen_symbol_ranges: bad argument");
  DeviceGuard g(ctx->device);
  CK(launch_widen_minmax(minmax_dev, n_pairs, ctx->stream, &ctx->launches));
  return PCGC_OK;
}

int pcgc_set_deferred_checks(pcgc_ctx* ctx, int on) {
  if (!ctx) return PCGC_ERR_BAD_ARG;
  ctx->deferred_checks = on != 0;
  return PCGC_OK;
}

int pcgc_set_quantize_mode(pcgc_ctx* ctx, int noise, uint64_t seed) {
  if (!ctx || noise < 0 || noise > 1) return fail(ctx, PCGC_ERR_BAD_ARG, "pcgc_set_quantize_mode: bad argument");
  ctx->quant_noise = noise; ctx->quant_seed = seed;
  return PCGC_OK;
}

int pcgc_factorized_cdf_host(pcgc_ctx* ctx, int slot, int min_v, int max_v, float likelihood_bound, int precision,
                             int32_t* cdf_host) {
  if (!ctx || slot < 0 || slot > 1 || !cdf_host) return fail(ctx, PCGC_ERR_BAD_ARG, "pcgc_factorized_cdf_host: bad argument");
  const std::vector<float>& hp = ctx->bn_host[slot];
  if (hp.empty()) return fail(ctx, PCGC_ERR_NOT_READY, "bottleneck slot %d not loaded", slot);
  const int C = (int)(hp.size() / 44), N = max_v - min_v + 1;
  if (N < 2) return fail(ctx, PCGC_ERR_BAD_RANGE, "single-symbol alphabet [%d,%d]", min_v, max_v);
  std::vector<float> pmf((size_t)C * N);
  for (int c = 0; c < C; ++c)
    for (int k = 0; k < N; ++k) pmf[(size_t)c * N + k] = fmaxf(det_bn_likelihood((float)(min_v + k), hp.data() + (size_t)c * 44), likelihood_bound);
  int r = pcgc_pmf_to_quantized_cdf(pmf.data(), C, N, precision, cdf_host);
  if (r) return fail(ctx, r, "pmf_to_quantized_cdf failed");
  return PCGC_OK;
}

int pcgc_laplace_cdf_dev(pcgc_ctx* ctx, const float* loc_dev, const float* scale_dev, int B, int64_t E,
                         const int32_t* minmax_dev, const int64_t* row_offset_dev, double rows_total, float likelihood_bound,
                         int precision, uint16_t* cdf_dev) {
  if (!ctx || !loc_dev || !scale_dev || !minmax_dev || !row_offset_dev || !cdf_dev || B < 0 || precision != 16)
    return fail(ctx, PCGC_ERR_BAD_ARG, "pcgc_laplace_cdf_dev: bad argument (precision must be 16)");
  DeviceGuard g(ctx->device);
  if (B == 0) return PCGC_OK;
  prof_begin(ctx, "laplace_cdf", 0, 8.0 * B * E + 2.0 * rows_total);
  CK(launch_laplace_cdf(loc_dev, scale_dev, B, E, minmax_dev, row_offset_dev, likelihood_bound, precision, cdf_dev,
                        ctx->err_flag, ctx->stream, &ctx->launches));
  prof_end(ctx);
  return PCGC_OK;
}

int pcgc_range_encode_intervals_dev(pcgc_ctx* ctx, const uint32_t* intervals_dev, int B, int64_t E, int precision,
                                    uint8_t* scratch_dev, int64_t stride, int64_t* lens_dev, uint8_t* packed_dev, int64_t cap,
                                    int64_t* offsets_dev) {
  if (!ctx || !intervals_dev || !scratch_dev || !lens_dev || !packed_dev || !offsets_dev || B < 0 || E <= 0 || E % 32 || E > 65536 ||
      stride < 6 * E + 32 || (stride & 15) || precision != 16)
    return fail(ctx, PCGC_ERR_BAD_ARG, "pcgc_range_encode_intervals_dev: bad argument (E %% 32 == 0, E <= 65536, stride %% 16 == 0, stride >= 6*E + 32, precision 16)");
  DeviceGuard g(ctx->device);
  if (B == 0) { CK(cudaMemsetAsync(offsets_dev, 0, sizeof(int64_t), ctx->stream)); return PCGC_OK; }
  prof_begin(ctx, "range_encode_gpu", 0, 4.0 * B * E);
  CK(launch_range_encode_intervals(intervals_dev, B, E, precision, scratch_dev, stride, lens_dev, packed_dev, cap, offsets_dev,
                                   ctx->err_flag, ctx->stream, &ctx->launches));
  prof_end(ctx);
  return PCGC_OK;
}

int pcgc_range_decode_rows_dev(pcgc_ctx* ctx, const uint8_t* packed_dev, const int64_t* offsets_dev, int B, int64_t E,
                               const uint16_t* rows_dev, const int64_t* row_offset_dev, double rows_total, const int32_t* minmax_dev,
                               int max_n, int precision, float* y_hat_dev) {
  if (!ctx || max_n < 1 || max_n > PCGC_MAX_SYMBOLS || !packed_dev || !offsets_dev || !rows_dev || !row_offset_dev || !minmax_dev || !y_hat_dev || B < 0 || E <= 0 || E % 32 ||
      precision < 1 || precision > 16)
    return fail(ctx, PCGC_ERR_BAD_ARG, "pcgc_range_decode_rows_dev: bad argument (E must be a multiple of 32)");
  DeviceGuard g(ctx->device);
  if (B == 0) return PCGC_OK;
  prof_begin(ctx, "range_decode_gpu", 0, 2.0 * rows_total + 4.0 * B * E);
  CK(launch_range_decode_rows(packed_dev, offsets_dev, B, E, rows_dev, row_offset_dev, minmax_dev, max_n, precision, y_hat_dev,
                              ctx->err_flag, ctx->stream, &ctx->launches));
  prof_end(ctx);
  return PCGC_OK;
}

}  // extern "C"
