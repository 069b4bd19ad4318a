/* pcgc_b200.h -- C ABI of libpcgc_b200.so: the B200 (sm_100a) implementation of PCGCv1's per-cube
 * compress/decompress hot path.  Plain pointers and sizes only; no torch / C++ types.
 *
 * Every entry point names the reference interface it replaces (paths into NJUVISION/PCGCv1).
 * The reference has no FFI of its own (it is Python on TF 1.13); the binding a maintainer adds
 * is the ctypes stub shown in INTEGRATION.md (pcgcv1_b200/_lib.py is that stub).
 *
 * Conventions
 *   - every function returns 0 on success or a negative pcgc_status; pcgc_last_error(ctx) gives text.
 *   - "dev" pointers are CUDA device pointers on the ctx's device, "host" pointers are CPU memory.
 *   - tensors are dense, channels-last NDHWC float32 unless stated (the reference's layout).
 *   - all device work is enqueued on the ctx stream (pcgc_set_stream); nothing synchronises unless
 *     the function returns a host value (documented per function).
 *   - a ctx is not thread-safe; different ctxs (one per GPU) are independent.  Host coder entry
 *     points (pcgc_range_*) take no ctx and are re-entrant.
 */
#ifndef PCGC_B200_H_
#define PCGC_B200_H_

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define PCGC_B200_ABI_VERSION 1

typedef struct pcgc_ctx pcgc_ctx;

typedef enum {
  PCGC_OK = 0,
  PCGC_ERR_BAD_ARG = -1,    /* null pointer, unknown enum, shape mismatch */
  PCGC_ERR_BAD_RANGE = -2,  /* symbol range unsupported (single-symbol alphabet, N > PCGC_MAX_SYMBOLS) or k out of range */
  PCGC_ERR_CUDA = -3,       /* a CUDA call failed; text in pcgc_last_error */
  PCGC_ERR_OOM = -4,
  PCGC_ERR_NOT_READY = -5,  /* weights of a required layer were never loaded */
  PCGC_ERR_OVERFLOW = -6,   /* output buffer too small */
  PCGC_ERR_CORRUPT = -7     /* bitstream inconsistent with the CDFs */
} pcgc_status;

/* Nets = the reference's Keras models (checkpoint top-level keys, transform.py:107-111). */
typedef enum {
  PCGC_NET_VOX_ANALYSIS = 0,   /* models/model_voxception.py:71-144  AnalysisTransform  */
  PCGC_NET_VOX_SYNTHESIS = 1,  /* models/model_voxception.py:147-214 SynthesisTransform */
  PCGC_NET_HYPER_ENCODER = 2,  /* models/model_voxception.py:217-252 HyperEncoder       */
  PCGC_NET_HYPER_DECODER = 3,  /* models/model_voxception.py:255-308 HyperDecoder       */
  PCGC_NET_SIMPLE_ANALYSIS = 4,  /* models/model_simple.py:12-51  AnalysisTransform  */
  PCGC_NET_SIMPLE_SYNTHESIS = 5, /* models/model_simple.py:54-95  SynthesisTransform */
  PCGC_NET_COUNT = 6
} pcgc_net;

typedef enum { PCGC_DTYPE_U8 = 0, PCGC_DTYPE_F32 = 1, PCGC_DTYPE_F64 = 2 } pcgc_dtype;

/* Mesh file formats of pcgc_mesh_parse. */
typedef enum { PCGC_MESH_OBJ = 0, PCGC_MESH_OFF = 1, PCGC_MESH_PLY = 2 } pcgc_mesh_format;

/* Conv engines.  AUTO = tcgen05 implicit GEMM where a layer qualifies, FP32 CUDA-core kernel elsewhere. */
typedef enum { PCGC_ENGINE_AUTO = 0, PCGC_ENGINE_FFMA = 1, PCGC_ENGINE_UMMA = 2 } pcgc_engine;

#define PCGC_MAX_SYMBOLS 64   /* largest max_v-min_v+1 the conditional CDF kernels accept */

/* ---- context ------------------------------------------------------------------------------- */
int pcgc_abi_version(void);
int pcgc_create(pcgc_ctx** out, int device);
void pcgc_destroy(pcgc_ctx* ctx);
const char* pcgc_last_error(const pcgc_ctx* ctx);
/* stream: a cudaStream_t cast to void* (NULL = legacy default stream). */
int pcgc_set_stream(pcgc_ctx* ctx, void* stream);
int pcgc_set_engine(pcgc_ctx* ctx, int engine);
/* number of kernels this library has launched on ctx since creation (bench "gpu_launches"). */
int64_t pcgc_launch_count(const pcgc_ctx* ctx);
int pcgc_synchronize(pcgc_ctx* ctx);
/* Pipelining aid.  Several entry points synchronise the stream only to read the device-side error flag (bad symbol range,
 * tcgen05 barrier timeout ...).  With deferred checks ON they return right after enqueueing; the caller MUST call
 * pcgc_synchronize (which reports the flag) before it consumes any result.  Default OFF. */
int pcgc_set_deferred_checks(pcgc_ctx* ctx, int on);
/* Measurement aid (bench.py roofline): when on, every kernel launch group is bracketed by CUDA events
 * on the ctx stream.  pcgc_profile_report synchronises, writes a JSON array of
 * {"tag","count","ms","flops","bytes"} (algorithmic work per tag) into buf and clears the records. */
int pcgc_profile_enable(pcgc_ctx* ctx, int on);
int pcgc_profile_report(pcgc_ctx* ctx, char* buf, int64_t cap);

/* ---- weights (replaces tf.train.Checkpoint.restore, transform.py:36-38,70-72,107-112,214-218) -- */
/* kernel: HOST float32 in the Keras layout ([k,k,k,Cin,Cout]; Conv3DTranspose [k,k,k,Cout,Cin]),
 * kshape = its 5 dims, bias: HOST float32 [Cout] or NULL for use_bias=False layers.
 * layer = the Keras name= of the layer ("conv_in", "vrn1_1_conv1_1", "up_1", ...). */
int pcgc_load_conv(pcgc_ctx* ctx, int net, const char* layer, const float* kernel, const int64_t kshape[5],
                   const float* bias);
/* EntropyBottleneck variables (models/entropy_model.py:42-68), HOST float32:
 * matrices = matrix_0..3 concatenated ([C,3,1],[C,3,3],[C,3,3],[C,1,3]), biases = bais_0..3
 * ([C,3,1]x3,[C,1,1]), factors = factor_0..3 (same shapes as biases).  slot 0 = "estimator"
 * of the checkpoint; slot 1 is free for a second bottleneck. */
int pcgc_load_bottleneck(pcgc_ctx* ctx, int slot, int channels, const float* matrices, const float* biases,
                         const float* factors);

/* Test hook for the tcgen05 engine: one 3x3x3 stride-1 SAME conv (+bias, optional ReLU) of a float32 NDHWC
 * batch [B,n,n,n,cin] (cin in {8,16,32,64}, cout <= 64, n in {16,32,64}) with a HOST Keras kernel
 * [3,3,3,cin,cout]; converts to the engine's split-bf16 format, runs the UMMA kernel, writes float32
 * [B,n,n,n,cout].  wt = 1 | 2 | 4 selects the y-banded form of the kernel (each M row produces wt output lines).
 * Synchronises.  Compared against a plain FP32 conv in tests/test_gpu_umma.py. */
int pcgc_debug_conv3_umma(pcgc_ctx* ctx, const float* in_dev, int n, int cin, int cout, const float* kernel_host,
                          const float* bias_host, int relu, int B, int wt, float* out_dev);

/* ---- transforms (dev pointers) --------------------------------------------------------------- */
/* AnalysisTransform()(x), one call for B cubes instead of tf.map_fn(parallel_iterations=1)
 * (transform.py:42-48,116-122).  cubes: [B,64,64,64,1] of `dtype`; y: [B,16,16,16,16] (voxception)
 * or [B,8,8,8,32] (simple).  net = PCGC_NET_VOX_ANALYSIS | PCGC_NET_SIMPLE_ANALYSIS. */
int pcgc_analysis(pcgc_ctx* ctx, int net, const void* cubes_dev, int dtype, int B, float* y_dev);
/* SynthesisTransform()(y) (transform.py:79-84,181-183,251-256): logits [B,64,64,64,1]. */
int pcgc_synthesis(pcgc_ctx* ctx, int net, const float* y_dev, int B, float* logits_dev);
/* HyperEncoder()(y) (transform.py:125-131): y [B,16,16,16,16] -> z [B,8,8,8,8]. */
int pcgc_hyper_encode(pcgc_ctx* ctx, const float* y_dev, int B, float* z_dev);
/* HyperDecoder()(z_hat) followed by scales = max(scales, 1e-9) (transform.py:138-146,225-233):
 * z_hat [B,8,8,8,8] -> loc, scale [B,16,16,16,16]; scale = max(|.|, scale_floor).
 * Bit-reproducible across calls, batch sizes, devices of the same type, pcgc_set_engine settings and the PCGC_UMMA_* tuning
 * switches (one pinned kernel program: the outputs become integer CDF tables on both sides of the stream). */
int pcgc_hyper_decode(pcgc_ctx* ctx, const float* z_hat_dev, int B, float scale_floor, float* loc_dev,
                      float* scale_dev);

/* ---- factorized entropy model (models/entropy_model.py) ---------------------------------------- */
/* EntropyBottleneck.__call__(x, training=False) (:153-181): x_hat = round-half-even(x),
 * p = max(|sigmoid(s*u)-sigmoid(s*l)|, bound).  x: [n_vox, C] (C fastest).  Optional outputs
 * (NULL to skip): x_hat_dev, p_dev [n_vox*C]; bits_dev (double, sum(log2 p) * -1);
 * minmax_dev int32[2] = {floor(min x_hat), ceil(max x_hat)} (:249-250).  No host sync. */
int pcgc_factorized_quantize_likelihood(pcgc_ctx* ctx, int slot, const float* x_dev, int64_t n_vox, int C,
                                        float likelihood_bound, float* x_hat_dev, float* p_dev,
                                        double* bits_dev, int32_t* minmax_dev);
/* EntropyBottleneck._get_cdf (:183-221): int32 cdf [C, N+1] to HOST, N = max_v-min_v+1 >= 2.
 * Synchronises the ctx stream. */
int pcgc_factorized_cdf(pcgc_ctx* ctx, int slot, int min_v, int max_v, float likelihood_bound, int precision,
                        int32_t* cdf_host);

/* ---- conditional (Laplace) entropy model (models/conditional_entropy_model.py) ------------------ */
/* SymmetricConditional.__call__(y, loc, scale, training=False) (:71-93) per cube.
 * y, loc, scale: [B, E] (E elements per cube, 65536 for voxception).  Optional outputs:
 * y_hat_dev, p_dev [B,E]; bits_dev double[B]; minmax_dev int32[2B] = {min_v, max_v} per cube
 * (:153-154).  No host sync. */
int pcgc_laplace_quantize_likelihood(pcgc_ctx* ctx, const float* y_dev, const float* loc_dev,
                                     const float* scale_dev, int B, int64_t E, float likelihood_bound,
                                     float* y_hat_dev, float* p_dev, double* bits_dev, int32_t* minmax_dev);
/* Makes per-cube symbol ranges codable and storable before the tables are built: min_v <- min(min_v, 0), max_v <- max(max_v, 0)
 * (the container packs max*16 - min with min <= 0 <= max, dataprocess/inout_bitstream.py:95-96) and max_v <- 1 for the
 * one-symbol range {0} (pmf_to_quantized_cdf needs two symbols, entropy_model.py:192-193).  minmax_dev int32[2*n_pairs]. */
int pcgc_widen_symbol_ranges(pcgc_ctx* ctx, int32_t* minmax_dev, int n_pairs);
/* Encoder side of SymmetricConditional._get_cdf + range_encode's table lookup (:95-124,142-161):
 * for every element builds its quantised CDF row over min_v[b]..max_v[b] and emits only the
 * interval of the element's own symbol: interval = lower | (upper-lower-1) << 16.
 * y_hat: [B,E] rounded latents; minmax_dev int32[2B] (device, e.g. from the call above). */
int pcgc_laplace_intervals(pcgc_ctx* ctx, const float* y_hat_dev, const float* loc_dev, const float* scale_dev,
                           int B, int64_t E, const int32_t* minmax_dev, float likelihood_bound, int precision,
                           uint32_t* intervals_dev);
/* Decoder side (:186-195): full rows.  Cube b's rows start at row_offset[b] (in uint16 units,
 * HOST array of B+1 prefix sums of E*N_b) and hold cdf[0..N_b-1] as uint16 (cdf[N_b] = 2^precision
 * is implied).  minmax_host int32[2B]. */
int pcgc_laplace_cdf(pcgc_ctx* ctx, const float* loc_dev, const float* scale_dev, int B, int64_t E,
                     const int32_t* minmax_host, float likelihood_bound, int precision,
                     const int64_t* row_offset_host, uint16_t* cdf_dev);

/* Test hook: the DEVICE copy of the 16-bit normaliser on given pmf rows (device float32 [rows,N], 2 <= N <=
 * PCGC_MAX_SYMBOLS) -> device int32 cdf [rows,N+1]; must equal pcgc_pmf_to_quantized_cdf bit for bit.  Synchronises. */
int pcgc_debug_quantize_pmf(pcgc_ctx* ctx, const float* pmf_dev, int64_t rows, int N, int precision, int32_t* cdf_dev);

/* "noise" quantisation of the training graph (entropy_model.py:105-107, conditional_entropy_model.py:62-64): when noise = 1
 * the two *_quantize_likelihood entry points return x + U(-1/2, 1/2) (counter-based Philox4x32-10 keyed by `seed`, element
 * index as the counter: reproducible, independent of the launch shape) and the likelihood AT that value instead of round(x);
 * minmax outputs are then meaningless.  noise = 0 (default) is "symbols" = round half to even. */
int pcgc_set_quantize_mode(pcgc_ctx* ctx, int noise, uint64_t seed);
/* Test hook (host, no ctx): the four draws of elements 4*v .. 4*v+3 for `seed` as the kernels make them (the conditional
 * model's launch uses seed + 0x9E3779B97F4A7C15 so that y and z do not share a stream). */
int pcgc_debug_noise(uint64_t seed, uint64_t v, float* out4);

/* ---- GPU-side range coding of the per-cube strings (SURVEY.md 8(f) rank 2; models/conditional_entropy_model.py:126-201) ----
 * All pointers are DEVICE pointers, nothing synchronises; device-side failures (overflow, bad range) set the ctx error flag
 * that pcgc_synchronize reports.  The strings are byte-identical to the host coder's (same state machine source). */
/* pcgc_laplace_cdf with device-resident headers: minmax_dev int32[2B], row_offset_dev int64[B+1] (uint16 units);
 * rows_total = row_offset[B] (only used for the profile's byte count). */
int pcgc_laplace_cdf_dev(pcgc_ctx* ctx, const float* loc_dev, const float* scale_dev, int B, int64_t E,
                         const int32_t* minmax_dev, const int64_t* row_offset_dev, double rows_total, float likelihood_bound,
                         int precision, uint16_t* cdf_dev);
/* range_encode of B cubes from pcgc_laplace_intervals' output (precision 16, E % 32 == 0): cube b is coded into
 * scratch_dev + b*stride (E <= 65536; stride a multiple of 16 and >= 6*E + 32: the string, at most one 16-bit word per symbol,
 * followed by the encoder's 32-bit digit sums), lens_dev[b] receives its length, then the strings are concatenated into
 * packed_dev (capacity cap; 2*E + 2 bytes per cube always suffice) with offsets_dev int64[B+1] (offsets[B] = total bytes). */
int pcgc_range_encode_intervals_dev(pcgc_ctx* ctx, const uint32_t* intervals_dev, int B, int64_t E, int precision,
                                    uint8_t* scratch_dev, int64_t stride, int64_t* lens_dev, uint8_t* packed_dev, int64_t cap,
                                    int64_t* offsets_dev);
/* range_decode of B cubes: string b = packed_dev[offsets[b] .. offsets[b+1]), rows as written by pcgc_laplace_cdf(_dev),
 * y_hat_dev float32 [B,E] = symbol + min_v (conditional_entropy_model.py:196-199).  E % 32 == 0; max_n = the largest
 * N_b = max_v - min_v + 1 of the call (<= PCGC_MAX_SYMBOLS; sizes the shared-memory row window). */
int pcgc_range_decode_rows_dev(pcgc_ctx* ctx, const uint8_t* packed_dev, const int64_t* offsets_dev, int B, int64_t E,
                               const uint16_t* rows_dev, const int64_t* row_offset_dev, double rows_total, const int32_t* minmax_dev,
                               int max_n, int precision, float* y_hat_dev);

/* ---- host twins of the CDF builders (bit-identical tables: det_math.h + cdf_norm.h are shared by host and device) ---------
 * Interoperability / test aids: a CPU that has (loc, scale) or the bottleneck parameters can build exactly the tables the GPU
 * coded with, and decode the stream with pcgc_range_decode_rows / pcgc_range_decode.  Not on the product path. */
int pcgc_host_laplace_cdf(const float* loc, const float* scale, int B, int64_t E, const int32_t* minmax, float likelihood_bound,
                          int precision, const int64_t* row_offset, uint16_t* rows, int threads);
int pcgc_factorized_cdf_host(pcgc_ctx* ctx, int slot, int min_v, int max_v, float likelihood_bound, int precision,
                             int32_t* cdf_host);

/* ---- top-k occupancy classification (dataprocess/inout_points.py:147-179) ---------------------- */
/* select_voxels: per cube k = ks[b] (caller computes int(rho * n_points)); threshold = k-th
 * largest logit; mask = logits >= threshold (ties kept).  k == 0 reproduces the reference's
 * values[-0] quirk (threshold = smallest logit > -2.0).  Outputs: mask_dev uint8 [B,V],
 * thres_dev float[B] (optional), count_dev int32[B] (optional, voxels set). */
int pcgc_topk_select(pcgc_ctx* ctx, const float* logits_dev, int B, int64_t V, const int32_t* ks_dev,
                     uint8_t* mask_dev, float* thres_dev, int32_t* count_dev);
/* fixed_thres bypass of select_voxels (:157-160). */
int pcgc_threshold_select(pcgc_ctx* ctx, const float* logits_dev, int B, int64_t V, float thres,
                          uint8_t* mask_dev, int32_t* count_dev);

/* ---- host range coder (replaces coder_ops.range_encode / range_decode / pmf_to_quantized_cdf,
 *      models/entropy_model.py:218,258,298; models/conditional_entropy_model.py:122,161,195) ------ */
/* pmf float32 [rows,N] -> cdf int32 [rows,N+1]. */
int pcgc_pmf_to_quantized_cdf(const float* pmf, int64_t rows, int N, int precision, int32_t* cdf);
/* Symbols sym[i] coded with row (i % cdf_rows) of cdf [cdf_rows, N+1] (the EntropyBottleneck
 * broadcast [1,C,N+1] against data [M,C]).  out/cap: caller buffer; *len receives the size. */
int pcgc_range_encode(const int16_t* sym, int64_t n, const int32_t* cdf, int cdf_rows, int N, int precision,
                      uint8_t* out, int64_t cap, int64_t* len);
int pcgc_range_decode(const uint8_t* data, int64_t nbytes, int64_t n, const int32_t* cdf, int cdf_rows, int N,
                      int precision, int16_t* sym);
/* As pcgc_range_decode, publishing progress: after every `step` symbols (and at the end) the count of symbols already
 * written to sym is stored to *progress (release order; -1 on a bad argument), so a second thread can start on the head of
 * one long string -- decompress_hyper starts the hyper decoder on the first cubes while the rest of z is still decoded. */
int pcgc_range_decode_progress(const uint8_t* data, int64_t nbytes, int64_t n, const int32_t* cdf, int cdf_rows, int N,
                               int precision, int16_t* sym, int64_t* progress, int64_t step);
/* Per-element intervals from pcgc_laplace_intervals -> one string. */
int pcgc_range_encode_intervals(const uint32_t* intervals, int64_t n, int precision, uint8_t* out, int64_t cap,
                                int64_t* len);
/* Per-element rows from pcgc_laplace_cdf (N uint16 per element, last implied) -> symbols. */
int pcgc_range_decode_rows(const uint8_t* data, int64_t nbytes, int64_t n, const uint16_t* rows, int N,
                           int precision, int16_t* sym);
/* Many independent strings at once on a host thread pool (threads <= 0: all cores).
 * Cube b: intervals + b*E, output written at out + b*stride, length in lens[b]. */
int pcgc_range_encode_intervals_batch(const uint32_t* intervals, int B, int64_t E, int precision, uint8_t* out,
                                      int64_t stride, int64_t* lens, int threads);
int pcgc_range_decode_rows_batch(const uint8_t* const* data, const int64_t* nbytes, int B, int64_t E,
                                 const uint16_t* rows, const int64_t* row_offset, const int32_t* minmax,
                                 int precision, int16_t* sym, int threads);

/* Same, writing y_hat = symbol + min_v as float32 [B,E] (conditional_entropy_model.py:196-199). */
int pcgc_range_decode_rows_batch_f32(const uint8_t* const* data, const int64_t* nbytes, int B, int64_t E,
                                     const uint16_t* rows, const int64_t* row_offset, const int32_t* minmax,
                                     int precision, float* y_hat, int threads);

/* ---- training step primitives (train_hyper.py:184-214, loss.py:8-33; SURVEY.md 8a row a22) -------------------------------
 * Exact FP32 on CUDA cores, deterministic (fixed reduction orders, no atomics).  All pointers are DEVICE pointers, float32
 * NDHWC activations, kernels in the Keras layouts ([k,k,k,Cin,Cout]; Conv3DTranspose [k,k,k,Cout,Cin]); nothing synchronises.
 * pcgcv1_b200/training.py strings them into the reference's training graph (torch.autograd is only the tape). */
/* y = act(conv(x) + bias): x [B,n,n,n,cin] -> out [B,m,m,m,cout], m = n/stride (conv) or n*stride (transposed); k odd, SAME. */
int pcgc_train_conv_forward(pcgc_ctx* ctx, const float* x, int B, int n, int cin, int cout, int k, int stride, int transposed,
                            const float* w_keras, const float* bias, int relu, float* out);
/* dx [B,n,n,n,cin] from the output gradient g [B,m,m,m,cout] of the same layer (n = the layer's INPUT grid). */
int pcgc_train_conv_dgrad(pcgc_ctx* ctx, const float* g, int B, int n, int cin, int cout, int k, int stride, int transposed,
                          const float* w_keras, float* dx);
/* dw (the layer's Keras layout) and db [cout] (NULL for use_bias=False layers) from the layer input x and g.
 * The form of dW follows from the shape alone.  k <= 3 (every Voxception layer): the tile kernel, one partial per anchor tile
 * (2x4x4 anchors at stride 2, 4x8x8 at stride 1), summed in groups of 64 tiles and then over the groups; the workspace grows with
 * the batch; also k = 5, where it measured faster than the slice kernel.  k = 9 with <= 64 anchor channels (the anchor side is g
 * for a conv, x for a transposed conv; conv_1 and deconv_3 of model_simple): the slice kernel.  Its anchor tiles (2x4x8) are cut
 * into S contiguous runs, S = min(128, ceil(592 / Y)) with Y = ceil(min(cg, 8) * ceil(ca / 4) * k^2 / 128) * ceil(cg / 8) (cg = the other side's channels), a function of the shape only;
 * every dW element is summed over the tiles of a run in increasing order (voxels in z, y, x order within a tile), then over the
 * runs in increasing order.  Its workspace is S * k^3 * cin * cout floats <= 128 * k^3 * cin * cout, whatever the batch.
 * Neither form uses atomics: two calls return the same bits. */
int pcgc_train_conv_wgrad(pcgc_ctx* ctx, const float* x, const float* g, int B, int n, int cin, int cout, int k, int stride,
                          int transposed, float* dw, float* db);
/* pcgc_train_conv_wgrad with the dW form forced: 0 = tile kernel (any odd k), 1 = slice kernel (k in {3, 5, 9}, <= 64 anchor
 * channels, else PCGC_ERR_BAD_ARG).  *partial_floats (nullable) = the size of the partial buffer the form used.  Test / benchmark
 * hook: the product path never calls it. */
int pcgc_debug_train_wgrad(pcgc_ctx* ctx, int form, const float* x, const float* g, int B, int n, int cin, int cout, int k, int stride,
                           int transposed, float* dw, float* db, int64_t* partial_floats);
/* out = g where y > 0 else 0 (gradient through a fused ReLU; y = the layer output). */
int pcgc_train_relu_backward(pcgc_ctx* ctx, const float* g, const float* y, int64_t n, float* out);
/* _VoxceptionResNet merge (model_voxception.py:64-67): out = relu(x + concat[t12, t23]) over nvox voxels of c channels. */
int pcgc_train_vrn_merge(pcgc_ctx* ctx, const float* x, const float* t12, const float* t23, int64_t nvox, int c, float* out);
int pcgc_train_vrn_merge_backward(pcgc_ctx* ctx, const float* g, const float* out, int64_t nvox, int c, float* gx, float* g12, float* g23);
/* scale = max(|s|, floor) (model_voxception.py:308, train_hyper.py:191) and its gradient. */
int pcgc_train_abs_floor(pcgc_ctx* ctx, const float* s, int64_t n, float floor_v, float* out);
int pcgc_train_abs_floor_backward(pcgc_ctx* ctx, const float* g, const float* s, int64_t n, float floor_v, float* out);
/* Gradients of coef * sum(log max(likelihood, bound)) w.r.t. the (noisy) latents, loc and scale of the conditional model. */
int pcgc_train_laplace_backward(pcgc_ctx* ctx, const float* y_t, const float* loc, const float* scale, int64_t n, float bound, float coef,
                                float* gy, float* gloc, float* gscale);
/* EntropyBottleneck(z, training=True) from the RAW variables (matrices / biases / factors concatenated in the pcgc_load_bottleneck
 * order): z_t = z + U(-1/2, 1/2) (Philox, `seed`), logsum_dev double[1] = sum(log max(likelihood, bound)). */
int pcgc_train_factorized_forward(pcgc_ctx* ctx, const float* matrices, const float* biases, const float* factors, int C, const float* z,
                                  int64_t nvox, uint64_t seed, float bound, float* z_t, double* logsum_dev);
/* The same for the EntropyBottleneck on z_t [nvox, C], with the gradients of its RAW variables (the pcgc_load_bottleneck order). */
int pcgc_train_factorized_backward(pcgc_ctx* ctx, const float* matrices, const float* biases, const float* factors, int C, const float* z_t,
                                   int64_t nvox, float bound, float coef, float* gz, float* gmatrices, float* gbiases, float* gfactors);
/* get_bce_loss (loss.py:8-33): sums_dev double[4] = {sum_empty -log(1-occ), sum_full -log(occ), #empty, #full}. */
int pcgc_train_bce(pcgc_ctx* ctx, const float* logits, const uint8_t* label, int64_t n, double* sums_dev);
int pcgc_train_bce_backward(pcgc_ctx* ctx, const float* logits, const uint8_t* label, int64_t n, const double* sums_dev, float w_empty,
                            float w_full, float* g);
/* get_focal_loss (loss.py:83-93; BASELINE config 5's "focal occupancy loss") on y_pred = sigmoid(logits), label in {0, 1}:
 * sums_dev double[2] = {-sum(alpha (1 - pt_1)^gamma log pt_1), -sum((1 - alpha) pt_0^gamma log(1 - pt_0))} with the reference's
 * clip to [1e-3, .999] (the constant "other" branch of each tf.where included); the loss is their sum.  The backward entry
 * writes g = weight * d loss / d logits (zero where the clip is active).  gamma >= 1. */
int pcgc_train_focal(pcgc_ctx* ctx, const float* logits, const uint8_t* label, int64_t n, float gamma, float alpha, double* sums_dev);
int pcgc_train_focal_backward(pcgc_ctx* ctx, const float* logits, const uint8_t* label, int64_t n, float gamma, float alpha, float weight,
                              float* g);
/* tf.train.AdamOptimizer update with the bias-corrected step lr_t = lr * sqrt(1 - beta2^t) / (1 - beta1^t). */
int pcgc_train_adam(pcgc_ctx* ctx, float* p, const float* g, float* m, float* v, int64_t n, float lr_t, float beta1, float beta2, float eps);

/* ---- point-cloud I/O either side of the codec (SURVEY.md section 8(f) rank 1) ----------------------- */
/* Multithreaded memcpy of a large host buffer (a pinned staging buffer -> the NumPy array handed to the caller; first-touch
 * page faults of the fresh destination are spread over the threads).  No reference counterpart: plumbing of this build. */
int pcgc_host_copy(void* dst, const void* src, int64_t nbytes, int threads);
/* load_ply_data (dataprocess/inout_points.py:8-28): every line of the ASCII text whose first three single-space
 * separated tokens parse as floats is a point, truncated to int32; other lines (header, comments) are skipped.
 * xyz: HOST int32 [cap,3]; *n = points found (set even when PCGC_ERR_OVERFLOW says cap was too small).  A line with a
 * numeric first token but fewer than three tokens returns PCGC_ERR_CORRUPT (the reference raises IndexError there). */
int pcgc_ply_parse(const char* text, int64_t nbytes, int32_t* xyz, int64_t cap, int64_t* n, int threads);
/* write_ply_data (inout_points.py:30-46) for integer coordinates: header + "x y z\n" per point, byte-identical to the
 * reference's output.  out: HOST buffer of at least 160 + 36*n bytes. */
int pcgc_ply_format(const int32_t* xyz, int64_t n, char* out, int64_t cap, int64_t* len, int threads);
/* The cube partition of load_points (inout_points.py:50-90): cube = point // cube_size, local = point % cube_size, cubes
 * with fewer than min_num points dropped (a single-point cube counts as 3, the reference's 1-D shape quirk), kept cubes
 * ordered by x + y*step + z*step^2 with step = max kept cube coordinate + 1, file order inside a cube.
 * Outputs (HOST, caller-allocated): local_sorted int16 [local_cap,3] (points of the kept cubes, grouped in sorted cube
 * order; local_cap = n suffices unless negative coordinates make the reference repeat a cube -- PCGC_ERR_OVERFLOW then
 * reports the needed size in *n_points), cube_pos_seen int64 [n,3] (kept cubes in first-appearance order = the reference's cube_positions
 * return value), cube_pos_sorted int64 [n,3], counts_sorted int64 [n], *n_cubes, *n_points. */
int pcgc_partition_points(const int32_t* xyz, int64_t n, int cube_size, int min_num, int16_t* local_sorted, int64_t local_cap,
                          int64_t* cube_pos_seen, int64_t* cube_pos_sorted, int64_t* counts_sorted, int64_t* n_cubes,
                          int64_t* n_points);
/* points2voxels (inout_points.py:116-132) on the device: local_dev int16 [n,3] grouped per cube, offsets_host int64
 * [B+1] -> cubes_dev uint8 [B,S,S,S] (0/1).  Coordinates outside [0,S) return an error (the reference raises
 * IndexError).  Synchronises (error flag). */
int pcgc_voxelize(pcgc_ctx* ctx, const int16_t* local_dev, const int64_t* offsets_host, int B, int S, uint8_t* cubes_dev);
/* voxels2points (inout_points.py:134-143) on the device: mask_dev uint8 [B,S,S,S] -> counts_dev int32 [B], points_dev
 * int16 [cap,3] (non-zero voxels as (d,h,w), lexicographic per cube, cubes in order = np.where order) and *total_dev
 * (int64, may exceed cap: only the first cap points are written).  S must be a multiple of 16.  Does not synchronise. */
int pcgc_extract_points(pcgc_ctx* ctx, const uint8_t* mask_dev, int B, int S, int32_t* counts_dev, int16_t* points_dev,
                        int64_t cap, int64_t* total_dev);

/* ---- D1 / D2 geometry metrics (myutils/pc_error_wrapper.py geometry_metrics; MPEG pc_error's definitions) ------------------
 * a_dev float64 [n_a,3], b_dev float64 [n_b,3], normals_a_dev float64 [n_a,3] (unit normals of A) or NULL for p2point only; all
 * DEVICE pointers.  For direction 1 every a against its nearest b, for direction 2 every b against its nearest a; e = query - neighbour:
 *   p2point |e|^2,  p2plane (e . n)^2 with n = normal of a (direction 1) or of the nearest a (direction 2).
 * out_dev double[8] = [direction 1, 2][p2point, p2plane][sum, max]; the p2plane entries are 0 when normals_a_dev is NULL.
 * Exact search (uniform grid over each set, ring-by-ring, no cap).  TIE RULE: among equidistant neighbours the lowest index of the
 * searched array wins.  Per-point arithmetic as NumPy's ((x0 + x1) + x2, no contraction); sums in a fixed order (deterministic;
 * exact for integer coordinates).  Empty sets or more than 2^27 points: PCGC_ERR_BAD_ARG.  Enqueued on the ctx stream, does not
 * synchronise (except when the per-ctx workspace grows). */
int pcgc_geometry_sums(pcgc_ctx* ctx, const double* a_dev, int64_t n_a, const double* b_dev, int64_t n_b, const double* normals_a_dev,
                       double* out_dev);

/* ---- k-nearest-neighbour PCA normals of one point set (the normals file D2 reads) ---------------------------------------------
 * pts_dev float64 [n,3], normals_dev float64 [n,3] (out), knn_idx_dev int32 [n,k] (out, optional: NULL = not written); all DEVICE
 * pointers.  1 <= n <= 2^27, 1 <= k <= 64 (k > n: all n points); otherwise PCGC_ERR_BAD_ARG.
 *   NEIGHBOURHOOD of point i: the m = min(k, n) points of the set with the smallest (d2, index), compared lexicographically, with
 *     e = p_i - p_j and d2 = (e0*e0 + e1*e1) + e2*e2 (as pcgc_geometry_sums).  The point itself is included (d2 = 0); equidistant
 *     points are taken in ascending index (the LOWEST index wins at the k-th distance).  knn_idx_dev row i lists them in that
 *     order; slots m .. k-1 hold -1.  Exact search over one uniform grid (pcgc_geometry_sums' grid and ring-by-ring search, no cap).
 *   COVARIANCE, in (d2, index) order, on u_j = p_j - p_i (relative to the point, which leaves C unchanged mathematically and keeps
 *     it exactly 0 when all neighbours coincide): mu = (sum u_j) / m, then C = sum (u_j - mu)(u_j - mu)^T / m; two passes, running
 *     sums in that fixed order, every multiply and add rounded on its own (no FMA).
 *   NORMAL: the unit eigenvector of the smallest eigenvalue of C by cyclic Jacobi (at most 32 sweeps; lowest axis on an exact
 *     eigenvalue tie), scaled to unit length; sign: its component of largest magnitude is positive (lowest axis on an exact tie).
 *     C == 0 (one point, or all neighbours at the same coordinates) gives (0, 0, 1).
 * Deterministic (two calls give the same bits).  Enqueued on the ctx stream, does not synchronise (except when the per-ctx
 * workspace, shared with pcgc_geometry_sums, grows). */
int pcgc_estimate_normals(pcgc_ctx* ctx, const double* pts_dev, int64_t n, int k, double* normals_dev, int32_t* knn_idx_dev);

/* ---- training data from meshes (pcgcv1_b200/dataset.py) ----------------------------------------------------------------------
 * Triangle mesh reader.  format: PCGC_MESH_OBJ = 0, PCGC_MESH_OFF = 1, PCGC_MESH_PLY = 2.  verts: HOST float64 [vcap,3]; tris: HOST
 * int32 [tcap,3] (0-based).  *nv / *nt are set even when PCGC_ERR_OVERFLOW reports a capacity too small; malformed input ->
 * PCGC_ERR_CORRUPT.  Every polygon with n >= 3 corners becomes the fan (v0, v_i, v_{i+1}) in file order; a face with fewer than 3
 * corners, an index out of range or a truncated file is PCGC_ERR_CORRUPT.
 *   OBJ: "v x y z [w]" (further values ignored); "f" tokens i, i/j, i//k, i/j/k, negative indices counting back from the vertices
 *        read so far, index 0 an error; vt, vn, g, o, s, usemtl, mtllib, l, p and # lines ignored, any other statement CORRUPT.
 *   OFF: "OFF" or "COFF" header (the counts may be glued on: "OFF490 518 0"), # comments, "nv nf ne", vertex lines "x y z ..."
 *        (values after z ignored), face lines "n i0 .. i{n-1} ..." (colour values after the indices ignored).
 *   PLY: "ascii 1.0" or "binary_little_endian 1.0" (any other format: PCGC_ERR_BAD_ARG); element vertex with x / y / z of any
 *        scalar type (other properties skipped), element face with "property list <count> <index> vertex_indices|vertex_index"
 *        (other properties skipped); other elements skipped, in binary files only when all their properties are scalars. */
int pcgc_mesh_parse(const char* data, int64_t nbytes, int format, double* verts, int64_t vcap, int32_t* tris, int64_t tcap,
                    int64_t* nv, int64_t* nt);

/* Uniform surface sampling of a triangle mesh, grid quantisation and deduplication.  verts_dev float64 [nv,3], tris_dev int32 [nt,3],
 * points_dev int32 [n,3] (out), samples_dev float64 [n,3] and face_dev int32 [n] (optional outputs, NULL = not written): DEVICE
 * pointers; rot_host float64 [9] (row-major R) and *n_unique: HOST.  This project's own exact rule (no external sampler's):
 *   1. FACE WEIGHT: e1 = B - A, e2 = C - A, c = e1 x e2 component-wise (cx = e1y*e2z - e1z*e2y, ...), a2 = sqrt((cx*cx + cy*cy) + cz*cz)
 *      (twice the area).  With M = max a2 and frexp(M) = (m, e): w = (uint64) floor(ldexp(a2, 32 - e)) < 2^32 (exact scaling).
 *      w = 0 exactly when a2 < 2^(e-32): every degenerate face and every face below 2^-32 of the largest (faces up to 2^-31 of the
 *      largest may fall under it too) is NEVER drawn.  P = exclusive prefix sum of w (uint64, exact), W = total.
 *   2. SAMPLE j (0 <= j < n): r = philox4x32_10(counter (j_lo, j_hi), key (seed_lo, seed_hi)); t = r1 * 2^32 + r0;
 *      target = mulhi64(t, W); face f = the largest f with P[f] <= target.  u1 = (r2 + 0.5) 2^-32, u2 = (r3 + 0.5) 2^-32, s = sqrt(u1),
 *      a = 1 - s, b = s*(1 - u2), c = s*u2; p = (a*A + b*B) + c*C per coordinate (uniform density on the triangle).
 *   3. ROTATION AND GRID: q = R p, row r = (R[r][0]*p0 + R[r][1]*p1) + R[r][2]*p2.  [lo, hi] = box of the rotated vertices that a
 *      face references (unreferenced vertices are ignored; the box depends only on the mesh and R, not on n or the seed);
 *      E = max over axes of (hi - lo), scale = (resolution - 1) / E; g = clamp(rint((q - lo) * scale), 0, resolution - 1), rint
 *      rounding half to even.
 *   4. DEDUPLICATION: key (gx*R + gy)*R + gz (R = resolution), radix-sorted over 3*ceil(log2 R) bits, unique.  points_dev[0 .. *n_unique)
 *      = the distinct grid points in ascending key order (lexicographic (x, y, z)); samples_dev = q and face_dev = f in sample order.
 * Every multiply and add is rounded on its own (no FMA).  PCGC_ERR_BAD_ARG: 2 <= resolution <= 4096, 1 <= n <= 2^28,
 * 1 <= nt <= 2^30, 1 <= nv < 2^31 violated; a face index outside [0, nv); a non-finite a2; W == 0; a zero or non-finite box extent E
 * (the last four detected on the device).  Runs on the ctx stream and synchronises once (n_unique and the error flags); the per-ctx
 * workspace grows as needed.  Deterministic: two calls give the same bits. */
int pcgc_mesh_sample(pcgc_ctx* ctx, const double* verts_dev, int64_t nv, const int32_t* tris_dev, int64_t nt, const double* rot_host,
                     int64_t n, uint64_t seed, int resolution, int32_t* points_dev, int64_t* n_unique, double* samples_dev,
                     int32_t* face_dev);

#ifdef __cplusplus
}
#endif
#endif /* PCGC_B200_H_ */
