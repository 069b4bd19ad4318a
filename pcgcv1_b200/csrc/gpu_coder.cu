// GPU-side range coding of the per-cube latent strings (SURVEY.md section 8(f) rank 2): the byte streams of
// SymmetricConditional.compress / decompress (models/conditional_entropy_model.py:126-201) are written and read on the
// device, so neither the per-element CDF rows (65 536 x N uint16 per cube) nor the per-element intervals cross PCIe and no
// host thread pool sits between the transforms.  Cubes are independent strings (transform.py:157-168): the coder is
// sequential inside a string and parallel over cubes.
//
// The state machines are range_coder.h's -- the SAME source as the host coder (coder.cpp) -- so a string written here is
// byte-identical to pcgc_range_encode_intervals' and decodes with pcgc_range_decode_rows (tests/test_gpu_coder.py).
//   encode: one WARP per cube with the state replicated in every lane: coalesced interval loads handed round by shuffles, a
//           warp-uniform renormalisation branch, lane 0 stores the words.
//   decode: one WARP per cube.  The symbol search is lane-parallel: lane k holds cdf[k] of the current symbol's row and
//           tests size*cdf[k] <= offset; a ballot gives the symbol without a division or a serial scan.  Rows stream
//           through a double-buffered shared-memory window (cp.async), the next 16-bit word of the string is prefetched.
#include <stdint.h>

#include "common.cuh"
#include "range_coder.h"

namespace pcgc {

namespace {

// Encoder, one WARP per cube, precision 16.  A range encoder is sequential only in its SIZE: size_{i+1} depends on size_i and the
// interval of symbol i, nothing else.  The base -- the number the string spells -- is a SUM,
//     string = sum_i  a_i * 2^(-16 R_i),      a_i = (size_i * lower_i) >> 16,   R_i = renormalisations before symbol i,
// whose cache / pending-0xFFFF bookkeeping in RangeEncoder16 is just lazy carry propagation.  So the kernel splits the work:
//   1. chain   : 32 symbols at a time, state replicated in every lane, NOTHING but the size recurrence on the serial path
//                (two IMAD.WIDE, two funnel shifts, one IADD3, one compare, one select); lane j keeps a_j, a bit mask keeps the
//                renormalisation flags.  The intervals of the group come from shared memory as broadcast 8-byte loads.
//   2. digits  : lane j adds hi16(a_j) to 16-bit digit R_j and lo16(a_j) to digit R_j + 1 of a 128-digit shared-memory window
//                (R_j from a popcount of the flag mask); digits the chain has moved past are flushed to the cube's scratch as
//                32-bit sums (Sum a_i < 2^32 between two renormalisations and E <= 65536 bound a digit below 2^32).
//   3. carries : after the last symbol the digits are resolved right to left, 32 per step with shuffles (the loop runs until
//                no lane carries: twice in expectation), byte-swapped into the string; the length follows the upstream Finalize rule.
// finish() of range_coder.h = the upstream Finalize rule on the last two digits (see the end of the kernel).
// Same bytes as RangeEncoder16 / the host coder for every input (tests/test_gpu_coder.py); measured 3.8 -> see DESIGN.md.
// The r02 first form ran the whole RangeEncoder16 per symbol on the serial path (~104 cycles per symbol).
__device__ __forceinline__ void cp_async4(uint32_t dst, const void* src) {
  asm volatile("cp.async.ca.shared.global [%0], [%1], 4;" ::"r"(dst), "l"(src) : "memory");
}

constexpr int ENC_W = 128;                      // digit window: 31 unflushed + 32 new + 2 < 128

__global__ void __launch_bounds__(32)
range_encode_intervals_kernel(const uint32_t* __restrict__ iv, int B, int64_t E, uint8_t* __restrict__ out,
                              int64_t stride, int64_t dig_off, int64_t* __restrict__ lens) {
  __shared__ uint32_t s_win[ENC_W];
  __shared__ uint4 s_lu[2][32];
  __shared__ uint32_t s_w[4][32];
  const int lane = threadIdx.x;
  const int b = blockIdx.x;
  const unsigned FULL = 0xffffffffu;
  const uint32_t* src = iv + (size_t)b * E;
  uint16_t* o16 = reinterpret_cast<uint16_t*>(out + (size_t)b * stride);          // stride and the buffer are 16-byte aligned
  uint32_t* dig = reinterpret_cast<uint32_t*>(out + (size_t)b * stride + dig_off);
  for (int i = lane; i < ENC_W; i += 32) s_win[i] = 0;
  uint32_t sm1 = 0xFFFFFFFFu;                    // size - 1, identical in every lane
  uint32_t R = 0, Rfl = 0;                       // renormalisations so far; digits [0, Rfl) are in the scratch
  const int64_t groups = E / 32;                 // E % 32 == 0 (checked by the launcher)
  // interval words reach the lanes through a 4-slot shared-memory ring filled by cp.async two groups ahead (a register
  // prefetch put a false scoreboard wait on every iteration: 13 % of the kernel in the r02 ncu capture)
  const uint32_t s_w_addr = (uint32_t)__cvta_generic_to_shared(&s_w[0][lane]);
  auto prefetch = [&](int64_t g) {
    if (g < groups) cp_async4(s_w_addr + (uint32_t)(g & 3) * 128u, src + g * 32 + lane);
    asm volatile("cp.async.commit_group;" ::: "memory");
  };
  prefetch(0);
  prefetch(1);
  for (int64_t g = 0; g < groups; ++g) {
    prefetch(g + 2);
    asm volatile("cp.async.wait_group 2;" ::: "memory");
    const uint32_t w = s_w[g & 3][lane];
    // Operands pre-shifted by the lanes so that the products' HIGH words are the interval ends (no shift on the chain):
    //   a = (size*lower) >> 16 = hi32(sm1*L + L),  L = lower << 16;
    //   (size*upper) >> 16 = hi32(sm1*Ul + Ul) + Uh*(sm1 + 1),  upper << 16 = Uh*2^32 + Ul  (Uh = 1 only for upper = 2^16, Ul = 0 then)
    //   t = b - a = hi32(sm1*Ul + Ul) + (Uh*sm1 + Uh - 1) - a          -- all mod 2^32, as in range_coder.h
    const uint32_t lower = w & 0xFFFFu, upper = lower + (w >> 16) + 1u;
    s_lu[g & 1][lane] = make_uint4(lower << 16, upper << 16, upper >> 16, (upper >> 16) - 1u);
    __syncwarp();
    uint32_t a_keep = 0, rmask = 0;
#pragma unroll
    for (int j = 0; j < 32; ++j) {
      const uint4 lu = s_lu[g & 1][j];                                            // broadcast
      const uint32_t a = (uint32_t)(((uint64_t)sm1 * lu.x + lu.x) >> 32);
      const uint32_t x = (uint32_t)(((uint64_t)sm1 * lu.y + lu.y) >> 32);
      const uint32_t y = sm1 * lu.z + lu.w;
      const uint32_t t = x + y - a;
      const bool renorm = t < 0x10000u;
      sm1 = renorm ? ((t << 16) | 0xFFFFu) : t;
      a_keep = lane == j ? a : a_keep;
      rmask |= renorm ? (1u << j) : 0u;
    }
    const uint32_t Rj = R + __popc(rmask & ((1u << lane) - 1u));
    atomicAdd(&s_win[Rj & (ENC_W - 1)], a_keep >> 16);
    atomicAdd(&s_win[(Rj + 1) & (ENC_W - 1)], a_keep & 0xFFFFu);
    R += __popc(rmask);
    __syncwarp();
    while (R - Rfl >= 32) {
      const uint32_t idx = Rfl + lane;
      dig[idx] = s_win[idx & (ENC_W - 1)];
      s_win[idx & (ENC_W - 1)] = 0;
      Rfl += 32;
    }
    __syncwarp();
  }
  // finish() of range_coder.h (the upstream Finalize rule).  Digits R and R + 1 are the coder's current 32-bit window and have nothing to
  // their right, so their exact value mod 2^32 is local: low32.  If [low32, low32 + size - 1] wraps, the interval still holds a multiple
  // of 2^32 and THAT is the value written (+ (2^32 - low32): both digits become zero, one carry leaves to the left); otherwise the base
  // is rounded up to a multiple of 2^16 at digit R (+0xFFFF on digit R + 1).  Words 0..R are produced either way.
  const uint32_t w1 = s_win[(R + 1) & (ENC_W - 1)], w0 = s_win[R & (ENC_W - 1)] + (w1 >> 16);
  const uint32_t low32 = (w0 << 16) | (w1 & 0xFFFFu);
  const bool straddle = (uint32_t)(low32 + sm1) < low32;
  __syncwarp();
  if (lane == 0) {
    if (straddle) {
      const uint32_t x = 0u - low32;
      s_win[R & (ENC_W - 1)] += x >> 16;
      s_win[(R + 1) & (ENC_W - 1)] += x & 0xFFFFu;
    } else {
      s_win[(R + 1) & (ENC_W - 1)] += 0xFFFFu;
    }
  }
  __syncwarp();
  const uint32_t n_dig = R + 2;
  for (uint32_t idx = Rfl + lane; idx < n_dig; idx += 32) dig[idx] = s_win[idx & (ENC_W - 1)];
  __syncwarp();
  // carries, right to left: lane l of block k holds digit 32k + l (more significant = lower lane)
  const int nb = (int)((n_dig + 31) / 32);
  uint32_t cb = 0;                               // carry out of the block to the right
  uint32_t found = 0;                            // string length once the last non-zero byte is known
  for (int k0 = nb - 1; k0 >= 0; k0 -= 8) {       // 8 blocks' loads in flight at a time (the digits sit in L2)
    uint32_t vv[8];
#pragma unroll
    for (int q = 0; q < 8; ++q) {
      const int p = 32 * (k0 - q) + lane;
      vv[q] = (k0 - q >= 0 && (uint32_t)p < n_dig) ? dig[p] : 0u;
    }
#pragma unroll
    for (int q = 0; q < 8; ++q) {
      const int k = k0 - q;
      if (k < 0) break;
      const uint32_t p = (uint32_t)(32 * k + lane);
      uint32_t v = vv[q];
      uint32_t c = v >> 16, cbn = __shfl_sync(FULL, c, 0);
      uint32_t cin = __shfl_down_sync(FULL, c, 1);
      v = (v & 0xFFFFu) + (lane == 31 ? cb : cin);
      while (__any_sync(FULL, v >> 16)) {
        c = v >> 16;
        cbn += __shfl_sync(FULL, c, 0);
        cin = __shfl_down_sync(FULL, c, 1);
        v = (v & 0xFFFFu) + (lane == 31 ? 0u : cin);
      }
      cb = cbn;
      if (p <= R) o16[p] = (uint16_t)(((v & 0xFF) << 8) | (v >> 8));              // big-endian 16-bit word
      if (!found) {
        const uint32_t cand = (p <= R && v) ? ((v & 0xFF) ? 2 * p + 2 : 2 * p + 1) : 0u;
        found = __reduce_max_sync(FULL, cand);
      }
    }
  }
  // length: the words before the last one are written in full (upstream emits them while coding), the last word loses a zero low byte
  // and is left out when it is zero; after a straddle everything from the delayed word's last non-zero byte on is zero and left out
  if (!straddle && found < 2u * R) found = 2u * R;
  if (lane == 0) lens[b] = (int64_t)found;
}

// Concatenates the B strings: offsets[b] = sum of lens[0..b), offsets[B] = total; bytes beyond cap are dropped (error flag).
__global__ void __launch_bounds__(256)
pack_strings_kernel(const uint8_t* __restrict__ in, int64_t stride, const int64_t* __restrict__ lens, int B,
                    uint8_t* __restrict__ packed, int64_t cap, int64_t* __restrict__ offsets, int* __restrict__ err) {
  __shared__ int64_t s_part[256];
  const int b = blockIdx.x;
  int64_t acc = 0;
  for (int j = threadIdx.x; j < b; j += 256) acc += lens[j];
  s_part[threadIdx.x] = acc;
  __syncthreads();
  for (int o = 128; o > 0; o >>= 1) { if (threadIdx.x < o) s_part[threadIdx.x] += s_part[threadIdx.x + o]; __syncthreads(); }
  const int64_t off = s_part[0], n = lens[b];
  if (threadIdx.x == 0) { offsets[b] = off; if (b == B - 1) offsets[B] = off + n; }
  if (off + n > cap) { if (threadIdx.x == 0) atomicExch(err, PCGC_ERR_OVERFLOW); return; }
  const uint8_t* src = in + (size_t)b * stride;
  for (int64_t i = threadIdx.x; i < n; i += 256) packed[off + i] = src[i];
}

constexpr int DEC_G = 32;                       // symbols per shared-memory window
constexpr int DEC_MAXN = 64;                    // lane-parallel search: lane k tests entry k (and k + 32 in the WIDE form)


// One warp per cube, precision 16.  Per symbol the serial chain is: size -> one 32x32->64 multiply per lane -> compare with
// value - base -> two warp reductions (REDUX max / min) -> new base / size.  Derivation (range_coder.h RangeDecoder):
//   size*cdf[k] <= offset = ((d+1) << 16) - 1  with d = value - base   <=>   a_k := (size*cdf[k]) >> 16 <= d,
//   so the decoded symbol s is the LAST lane whose a_k <= d, its interval starts at a_s = max{a_k : a_k <= d} (a_k is
//   monotone) and ends at a_{s+1} - 1 = min{a_k - 1 : a_k > d}; lanes >= N hold cdf = 2^16, i.e. a_k - 1 = size - 1.
// Nothing inside the 32-symbol loop touches memory: the lane's CDF entries are read into registers first, the next 16-bit
// words of the string are prefetched one per lane and handed out by shuffles.
template <bool WIDE>
__global__ void __launch_bounds__(32)
range_decode_rows_kernel(const uint8_t* __restrict__ packed, const int64_t* __restrict__ offsets, int B, int64_t E,
                         const uint16_t* __restrict__ rows, const int64_t* __restrict__ row_offset,
                         const int32_t* __restrict__ minmax, float* __restrict__ y_hat, int* __restrict__ err, int win_elems) {
  extern __shared__ __align__(16) uint16_t s_rows[];              // [2][win_elems], win_elems >= DEC_G * max N of the launch
  const int lane = threadIdx.x;
  const int b = blockIdx.x;
  const unsigned FULL = 0xffffffffu;
  const int min_v = minmax[2 * b], N = minmax[2 * b + 1] - min_v + 1;
  if (N < 1 || N > (WIDE ? DEC_MAXN : 32) || DEC_G * N > win_elems) { if (lane == 0) atomicExch(err, PCGC_ERR_BAD_RANGE); return; }
  const uint8_t* str = packed + offsets[b];
  const int64_t nbytes = offsets[b + 1] - offsets[b];
  const uint32_t* rsrc = reinterpret_cast<const uint32_t*>(rows + row_offset[b]);    // E*N is even: 4-byte aligned windows
  const int words = DEC_G * N / 2;                                                   // uint32 words per window
  uint16_t* const wbuf[2] = {s_rows, s_rows + win_elems};
  const uint32_t sbuf[2] = {(uint32_t)__cvta_generic_to_shared(wbuf[0]), (uint32_t)__cvta_generic_to_shared(wbuf[1])};
  const int64_t groups = E / DEC_G;                                                  // E % 32 == 0 (checked by the host)
  auto fetch = [&](int64_t g, int buf) {
    const uint32_t* src = rsrc + (size_t)g * words;
    for (int w = lane; w < words; w += 32) cp_async4(sbuf[buf] + 4u * w, src + w);
    asm volatile("cp.async.commit_group;" ::: "memory");
  };
  // big-endian 16-bit word `i` of the string (zero beyond its end), i counted from the start of the string
  auto word_at = [&](int64_t i) -> uint32_t {
    const int64_t p = 2 * i;
    const uint32_t hi = p < nbytes ? (uint32_t)__ldg(str + p) : 0u, lo = p + 1 < nbytes ? (uint32_t)__ldg(str + p + 1) : 0u;
    return (hi << 8) | lo;
  };
  // decoder state, identical in every lane
  uint32_t value = (word_at(0) << 16) | word_at(1);
  int64_t wpos = 2;                                   // index of the next unread word
  uint32_t w0 = word_at(wpos + lane), w1 = word_at(wpos + 32 + lane);      // words wpos + [0, 64) spread over the lanes
  uint32_t base = 0, sm1 = 0xFFFFFFFFu;
  fetch(0, 0);
  for (int64_t g = 0; g < groups; ++g) {
    const int buf = (int)(g & 1);
    if (g + 1 < groups) { fetch(g + 1, buf ^ 1); asm volatile("cp.async.wait_group 1;" ::: "memory"); }
    else asm volatile("cp.async.wait_group 0;" ::: "memory");
    __syncwarp();
    const uint32_t wb = sbuf[buf];
    uint32_t c[DEC_G], c2[WIDE ? DEC_G : 1];
#pragma unroll
    for (int j = 0; j < DEC_G; ++j) {
      uint32_t v = 0x10000u;
      if (lane < N) { uint16_t t; asm volatile("ld.shared.u16 %0, [%1];" : "=h"(t) : "r"(wb + 2u * (uint32_t)(j * N + lane))); v = t; }
      c[j] = v;
      if (WIDE) {
        uint32_t v2 = 0x10000u;
        if (lane + 32 < N) { uint16_t t; asm volatile("ld.shared.u16 %0, [%1];" : "=h"(t) : "r"(wb + 2u * (uint32_t)(j * N + lane + 32))); v2 = t; }
        c2[j] = v2;
      }
    }
    uint32_t r = 0;                                   // renormalisations (= words consumed) in this group
    uint32_t nxt = __shfl_sync(FULL, w0, 0);
    int mine = 0;
#pragma unroll
    for (int j = 0; j < DEC_G; ++j) {
      const uint32_t d = value - base;
      const uint64_t q = ((uint64_t)sm1 * c[j] + c[j]) >> 16;                        // (size * cdf[lane]) >> 16
      const uint32_t a_l = (uint32_t)q;
      const bool pred = a_l <= d && c[j] < 0x10000u;
      uint32_t va = pred ? a_l : 0u, vu = pred ? 0xFFFFFFFFu : a_l - 1u;
      unsigned cnt = __ballot_sync(FULL, pred);
      int s = __popc(cnt) - 1;
      if (WIDE) {
        const uint32_t a2 = (uint32_t)(((uint64_t)sm1 * c2[j] + c2[j]) >> 16);
        const bool pred2 = a2 <= d && c2[j] < 0x10000u;
        va = pred2 ? a2 : va;
        vu = pred2 ? vu : min(vu, a2 - 1u);
        s += __popc(__ballot_sync(FULL, pred2));
      }
      const uint32_t a = __reduce_max_sync(FULL, va);
      const uint32_t bm1 = min(__reduce_min_sync(FULL, vu), sm1);
      base += a;
      const uint32_t t = bm1 - a;
      const bool renorm = t < 0x10000u;                                             // warp-uniform; selects instead of a branch keep the
      sm1 = renorm ? ((t << 16) | 0xFFFFu) : t;                                     // 32 symbols one basic block for the scheduler
      base = renorm ? (base << 16) : base;
      value = renorm ? ((value << 16) | nxt) : value;
      r += renorm ? 1u : 0u;
      nxt = __shfl_sync(FULL, w0, r & 31);
      if (lane == j) mine = s;
    }
    y_hat[(size_t)b * E + g * DEC_G + lane] = (float)(mine + min_v);
    // advance the word window by r (<= 32): new w0 = words [r, r + 32) of the old 64, new w1 is fetched (latency hidden by the
    // next group)
    {
      const uint32_t t = r + (uint32_t)lane;
      const uint32_t x0 = __shfl_sync(FULL, w0, t & 31), x1 = __shfl_sync(FULL, w1, t & 31);
      w0 = t < 32 ? x0 : x1;
      wpos += r;
      // w1 must become words [wpos + 32, wpos + 64): those below old wpos + 64 are already in w1 (shifted), the rest are new
      const uint32_t y1 = __shfl_sync(FULL, w1, t & 31);
      w1 = t < 32 ? y1 : word_at(wpos + 32 + lane);
    }
    __syncwarp();                                                                     // window `buf` is refilled two iterations later
  }
}


// Decoder for alphabets of at most 31 symbols (every cube of the reference's models; wider ones take the kernel above).  Same
// stream, same decisions as RangeDecoder of range_coder.h, with the serial path cut to what the recurrence needs.  State: size - 1
// and D = value - base (base and value themselves never matter).  Lane l holds C_l = cdf[l] << 16 of the current row, so
//     q_l = (size * cdf[l]) >> 16 = hi32(sm1 * C_l + C_l)                       (one IMAD.HI, no shift)
// and with q_N := size (lane N: C = 0 plus a per-lane constant) the decoded symbol s is the last lane with q_l <= D, its interval
// [a, b] = [q_s, q_{s+1} - 1].  Both ends come out of UNSIGNED MINIMA without a compare or select in front of the reductions:
//     D - a = min_l (D - q_l)            lanes with q_l > D wrap to >= 2^32 - size + D >= D
//     b - D = min_l (q_l - 1 - D)        lanes with q_l <= D wrap to >= 2^32 - 1 - D >= size - 1 - D (lane N)
// (ties only at size = 2^32 and only between equal values), so  t = b - a = min + min,  D' = D - a = the first minimum.  Chain per
// symbol: IMAD.HI -> IADD -> REDUX.MIN -> IADD -> ISETP -> SEL.  Off the chain: the symbol index (ballot, stored as a mask; the
// popcount is taken lane-parallel after 32 symbols), the next 16-bit word (broadcast load from a shared-memory ring of the string's
// words), the CDF rows (cp.async ring, two groups ahead).  No divergent branch inside the 32-symbol block.
constexpr int DECN_SLOTS = 4;

__device__ __forceinline__ void cp_async16(uint32_t dst, const void* src) {
  asm volatile("cp.async.cg.shared.global [%0], [%1], 16;" ::"r"(dst), "l"(src) : "memory");
}

__global__ void __launch_bounds__(32)
range_decode_rows_narrow_kernel(const uint8_t* __restrict__ packed, const int64_t* __restrict__ offsets, int B, int64_t E,
                                const uint16_t* __restrict__ rows, const int64_t* __restrict__ row_offset,
                                const int32_t* __restrict__ minmax, float* __restrict__ y_hat, int* __restrict__ err, int slot_elems) {
  extern __shared__ __align__(16) uint16_t s_rows_n[];            // [DECN_SLOTS][slot_elems], slot_elems >= 32 * max N + 32, multiple of 8
  __shared__ uint32_t s_words[128];                              // ring of the string's 16-bit words, indexed by word number & 127
  __shared__ uint32_t s_mask[32];
  const int lane = threadIdx.x;
  const int b = blockIdx.x;
  const unsigned FULL = 0xffffffffu;
  const int min_v = minmax[2 * b], N = minmax[2 * b + 1] - min_v + 1;
  if (N < 1 || N > 31 || 32 * N + 32 > slot_elems) { if (lane == 0) atomicExch(err, PCGC_ERR_BAD_RANGE); return; }
  const uint8_t* str = packed + offsets[b];
  const int64_t nbytes = offsets[b + 1] - offsets[b];
  const uint4* rsrc = reinterpret_cast<const uint4*>(rows + row_offset[b]);          // 64 * N bytes per group, 16-byte aligned (launcher)
  const int chunks = 4 * N;                                                          // 16-byte chunks per group
  const uint32_t slot0 = (uint32_t)__cvta_generic_to_shared(s_rows_n);
  const int64_t groups = E / 32;                                                     // E % 32 == 0 (checked by the host)
  auto fetch = [&](int64_t g) {
    if (g < groups) {
      const uint4* src = rsrc + (size_t)g * chunks;
      const uint32_t dst = slot0 + (uint32_t)(g & (DECN_SLOTS - 1)) * (uint32_t)slot_elems * 2u;
      for (int c = lane; c < chunks; c += 32) cp_async16(dst + 16u * c, src + c);
    }
    asm volatile("cp.async.commit_group;" ::: "memory");
  };
  // big-endian 16-bit word `i` of the string (zero beyond its end)
  auto word_at = [&](int64_t i) -> uint32_t {
    const int64_t p = 2 * i;
    const uint32_t hi = p < nbytes ? (uint32_t)__ldg(str + p) : 0u, lo = p + 1 < nbytes ? (uint32_t)__ldg(str + p + 1) : 0u;
    return (hi << 8) | lo;
  };
  fetch(0);
  fetch(1);
  // per-lane constants: valid lanes carry cdf << 16; lane N stands for cdf[N] = 2^16 (q_N - 1 = size - 1); lanes above never win
  const bool valid = lane < N;
  const uint32_t mul = valid ? 0x10000u : 0u, uh = lane == N ? 1u : 0u, um1 = uh - 1u;
  uint32_t sm1 = 0xFFFFFFFFu;
  uint32_t D = (word_at(0) << 16) | word_at(1);                  // value - base
  uint32_t wpos = 2;                                             // next unread word
  s_words[(2 + lane) & 127] = word_at(2 + lane);
  s_words[(34 + lane) & 127] = word_at(34 + lane);
  uint32_t filled = 66;                                          // words [.., filled) are in the ring
  uint32_t pend = word_at(filled + lane);                        // words [filled, filled + 32), stored when the ring has room
  __syncwarp();
  for (int64_t g = 0; g < groups; ++g) {
    if (filled - wpos <= 64) {                                   // uniform; keeps 32 <= filled - wpos <= 96 at every group start
      s_words[(filled + lane) & 127] = pend;
      filled += 32;
      pend = word_at(filled + lane);                             // consumed a group later at the earliest
    }
    fetch(g + 2);
    asm volatile("cp.async.wait_group 2;" ::: "memory");
    __syncwarp();
    const uint16_t* slot = s_rows_n + (size_t)(g & (DECN_SLOTS - 1)) * slot_elems;
    uint32_t C[32];
#pragma unroll
    for (int j = 0; j < 32; ++j) C[j] = (uint32_t)slot[j * N + lane] * mul;
    uint32_t nxt = s_words[wpos & 127];
#pragma unroll
    for (int j = 0; j < 32; ++j) {
      const uint32_t q = (uint32_t)(((uint64_t)sm1 * C[j] + C[j]) >> 32);
      const uint32_t e = D - q;
      const uint32_t z = q + (sm1 * uh + um1) - D;
      const uint32_t emin = __reduce_min_sync(FULL, e);
      const uint32_t zmin = __reduce_min_sync(FULL, z);
      const unsigned m = __ballot_sync(FULL, valid && q <= D);
      if (lane == 0) s_mask[j] = m;
      const uint32_t t = zmin + emin;
      const bool renorm = t < 0x10000u;
      sm1 = renorm ? ((t << 16) | 0xFFFFu) : t;
      D = renorm ? ((emin << 16) | nxt) : emin;
      wpos += renorm ? 1u : 0u;
      nxt = s_words[wpos & 127];
    }
    __syncwarp();
    y_hat[(size_t)b * E + g * 32 + lane] = (float)(__popc(s_mask[lane]) - 1 + min_v);
    __syncwarp();                                                // s_mask, the row slot and the word ring are rewritten next
  }
}

}  // namespace

// One-warp CTAs are placed wherever a slot is free.  Measured (r02): launched with no shared-memory
// request the 191 encoder CTAs of the vox10 cloud ran in one of two regimes, 1.7 ms or ~6-7 ms per launch, depending on what
// the device was finishing when the launch became runnable: the hardware scheduler stacks up to 32 such CTAs on the SMs that
// are free at that moment and they stay there for the whole launch, so a latency-bound warp shares its scheduler with 7
// others.  Unused dynamic shared memory per CTA caps the CTAs per SM (about B / 148 + 1, at least 2) and so forces a launch
// to spread over the device: 1.7 ms every time.  Large launches (thousands of cubes) keep up to 32 CTAs per SM: there the
// throughput of the SM counts, not the latency of one string.  The decoder gets no padding: its slowdown beside the synthesis is
// issue-slot contention with the conv CTAs of the same SM, which spreading it does not change (DESIGN.md §4.3).
static size_t encoder_pad_bytes(int B) {
  static const int max_kb = 200;
  int per_sm = (B + 147) / 148 + 1;
  if (per_sm < 2) per_sm = 2;
  if (per_sm >= 32) return 0;
  cudaFuncSetAttribute(range_encode_intervals_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, max_kb * 1024);
  return (size_t)(max_kb / per_sm - 2) * 1024;
}

cudaError_t launch_range_encode_intervals(const uint32_t* iv, int B, int64_t E, int precision, uint8_t* scratch, int64_t stride,
                                          int64_t* lens, uint8_t* packed, int64_t cap, int64_t* offsets, int* err,
                                          cudaStream_t s, int64_t* launches) {
  if (B <= 0) return cudaSuccess;
  // per cube: the string (at most 2 * (E + 1) bytes) then E + 2 digit sums of 4 bytes
  const int64_t dig_off = (2 * E + 2 + 15) / 16 * 16;
  if (precision != 16 || E % 32 || E > 65536 || stride < dig_off + 4 * (E + 2) || (stride & 15)) return cudaErrorInvalidValue;
  PCGC_CARVEOUT_ONCE(range_encode_intervals_kernel);
  PCGC_CARVEOUT_ONCE(pack_strings_kernel);
  range_encode_intervals_kernel<<<B, 32, encoder_pad_bytes(B), s>>>(iv, B, E, scratch, stride, dig_off, lens);
  pack_strings_kernel<<<B, 256, 0, s>>>(scratch, stride, lens, B, packed, cap, offsets, err);
  if (launches) *launches += 2;
  return cudaGetLastError();
}

cudaError_t launch_range_decode_rows(const uint8_t* packed, const int64_t* offsets, int B, int64_t E, const uint16_t* rows,
                                     const int64_t* row_offset, const int32_t* minmax, int max_n, int precision, float* y_hat, int* err,
                                     cudaStream_t s, int64_t* launches) {
  if (B <= 0) return cudaSuccess;
  if (E % DEC_G || max_n < 1 || max_n > DEC_MAXN || precision != 16) return cudaErrorInvalidValue;
  if (max_n <= 31 && (reinterpret_cast<uintptr_t>(rows) & 15) == 0) {
    // every row window is a multiple of 64 bytes (E % 32 == 0), so 16-byte cp.async needs only the base pointer aligned
    const int slot_elems = (32 * max_n + 32 + 7) / 8 * 8;
    PCGC_CARVEOUT_ONCE(range_decode_rows_narrow_kernel);
    range_decode_rows_narrow_kernel<<<B, 32, (size_t)DECN_SLOTS * slot_elems * sizeof(uint16_t), s>>>(packed, offsets, B, E, rows, row_offset,
                                                                                                      minmax, y_hat, err, slot_elems);
    if (launches) ++*launches;
    return cudaGetLastError();
  }
  const int win_elems = DEC_G * ((max_n + 7) / 8 * 8);              // 16-byte multiple per window
  const size_t smem = 2 * (size_t)win_elems * sizeof(uint16_t);
  PCGC_CARVEOUT_ONCE(range_decode_rows_kernel<true>);
  PCGC_CARVEOUT_ONCE(range_decode_rows_kernel<false>);
  if (max_n > 32)
    range_decode_rows_kernel<true><<<B, 32, smem, s>>>(packed, offsets, B, E, rows, row_offset, minmax, y_hat, err, win_elems);
  else
    range_decode_rows_kernel<false><<<B, 32, smem, s>>>(packed, offsets, B, E, rows, row_offset, minmax, y_hat, err, win_elems);
  if (launches) ++*launches;
  return cudaGetLastError();
}

}  // namespace pcgc
