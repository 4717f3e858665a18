// Hand-written sm_100a kernels for the CTC "extended" beam-search decode.
//
// The sections of this header are compiled by different translation units: define CTCX_WITH_NORM
// (normaliser kernels), CTCX_WITH_GENERIC (the generic beam kernel) and / or CTCX_WITH_POST (trace-back,
// scan, pack) before including it; the common helpers at the top are always available.
//
// What each kernel replaces in the reference (paths relative to
// tensorflow_ctc_ext_beam_search_decoder/cc/):
//   LogNormKernel   util/ctc_ext_beam_search_decoder.h:71-80   softmax normaliser of Step()
//   BeamKernel      util/ctc_ext_beam_search_decoder.h:84-209  Step(): extract/sort, member update,
//                   grow + prune; util/ctc_beam_entry.h (BeamEntry trie, BeamProbability,
//                   AddAlignmentCandidate); gtl::TopN; util/ctc_loss_util.h LogSumExp
//   TraceKernel     util/ctc_ext_beam_search_decoder.h:229-261 TopPaths +
//                   util/ctc_beam_entry.h:123-152 LabelSeq / AlignmentLabelSeq
//   ScanKernel/PackKernel  kernels/ctc_ext_beam_search_decoder_kernels.cc:163-257
//                   StoreAllDecodedSequences
//
// The beam kernel does NOT translate the reference's sequential trie walk. It implements the
// parallel formulation derived in DESIGN.md (validated on the CPU by tests/model/ctcx_model.cc):
// one CTA per utterance, the beam as sorted structure-of-arrays in shared memory, prefix identity by
// 64-bit hash, fresh children as a filtered candidate list, the reference's order-dependent
// "revisit-wipe" side effect as a count-based fixed point, the next beam by radix select + rank,
// and 8-byte back-pointer records per (frame, slot) in HBM for the device trace-back.
#pragma once
#include <cuda_runtime.h>
#include <cstdint>

#include <cuda_bf16.h>
#include <cuda_fp16.h>

#include "ctcx_math.cuh"
#include "ctcx_params.h"

namespace ctcx {

constexpr unsigned kFull = 0xffffffffu;
constexpr unsigned long long kRootHash = 0x243F6A8885A308D3ull;

// back-pointer record, word 0: [0,11) prev_self slot | [11,22) an_src slot | [22] ab_kind | [23,25) an_kind
constexpr unsigned kInvalidSlot = 0x7ffu;
enum { kAbFromAb = 0, kAbFromAn = 1 };
enum { kAnSelfAn = 0, kAnParAb = 1, kAnParAn = 2, kAnNone = 3 };

__device__ __forceinline__ unsigned PackRec(unsigned prev_self, unsigned an_src, unsigned ab_kind,
                                            unsigned an_kind) {
  return prev_self | (an_src << 11) | (ab_kind << 22) | (an_kind << 23);
}

__device__ __forceinline__ float NegInf() { return __int_as_float((int)0xff800000); }

// Monotone map float -> uint32 (larger float <=> larger key); -0.0 is canonicalised to +0.0.
__device__ __forceinline__ unsigned KeyOf(float s) {
  const unsigned u = __float_as_uint(__fadd_rn(s, 0.0f));
  return (u & 0x80000000u) ? ~u : (u | 0x80000000u);
}
__device__ __forceinline__ float UnKey(unsigned k) {
  return __uint_as_float((k & 0x80000000u) ? (k & 0x7fffffffu) : ~k);
}
constexpr unsigned kKeyNegInf = 0x007fffffu;  // KeyOf(-inf)

__device__ __forceinline__ unsigned long long HashChild(unsigned long long h, int label) {
  unsigned long long z = (h ^ (unsigned long long)(unsigned)(label + 1)) * 0x9E3779B97F4A7C15ull;
  z ^= z >> 29;
  z *= 0xBF58476D1CE4E5B9ull;
  z ^= z >> 32;
  return z;
}

// Streamed float64 decodes (see StreamHdrT): the double block of utterance b, or null where the double
// kernel starts from the root -- it resumes only a block that a double kernel wrote after the reset of a
// float64 stream, so that a stream stepped with both score types never feeds it foreign bytes.
__device__ __forceinline__ StreamViewT<double> StreamBlock64(unsigned char* state, int B, int W, int b) {
  return StreamViewT<double>(StreamState64(state, B, W) + (size_t)b * StreamStateBytes<double>(W), W);
}
// the block of utterance b that the kernels with R scores carry their beam in
template <typename R>
__device__ __forceinline__ StreamViewT<R> StreamBlock(unsigned char* state, int B, int W, int b) {
  if constexpr (sizeof(R) == 4) return StreamViewT<R>(state + (size_t)b * StreamStateBytes(W), W);
  else return StreamBlock64(state, B, W, b);
}
__device__ __forceinline__ bool StreamResumable64(unsigned char* state, int B, int W, int b) {
  const StreamView fv(state + (size_t)b * StreamStateBytes(W), W);
  return __ldcg(&fv.hdr->type) == 8 && __ldcg(&StreamBlock64(state, B, W, b).hdr->type) == 8;
}
// after a double kernel saved block b: a float stream gets the mark that ctcx_stream_top_paths reports
__device__ __forceinline__ void StreamMarkF64Step(unsigned char* state, int W, int b) {
  const StreamView fv(state + (size_t)b * StreamStateBytes(W), W);
  if (fv.hdr->type != 8) fv.hdr->type |= kStreamF64Stepped;
}

// element i of the caller's logits tensor as the decoder's score type (exact: float16 / bfloat16 ->
// float32 is a widening). The loads bypass L1: the narrow fast kernel may run while a host->device
// copy of later frames is still in flight (BeamParamsT::ready).
template <typename IN>
__device__ __forceinline__ float LoadLogit(const void* base, size_t i);
template <>
__device__ __forceinline__ float LoadLogit<float>(const void* base, size_t i) {
  return __ldcg(reinterpret_cast<const float*>(base) + i);
}
template <>
__device__ __forceinline__ float LoadLogit<__half>(const void* base, size_t i) {
  return __half2float(__ldcg(reinterpret_cast<const __half*>(base) + i));
}
template <>
__device__ __forceinline__ float LoadLogit<__nv_bfloat16>(const void* base, size_t i) {
  return __bfloat162float(__ldcg(reinterpret_cast<const __nv_bfloat16*>(base) + i));
}

// two packed half-precision elements -> two floats
template <typename IN>
__device__ __forceinline__ float2 Unpack2(unsigned v);
template <>
__device__ __forceinline__ float2 Unpack2<__half>(unsigned v) {
  return __half22float2(*reinterpret_cast<const __half2*>(&v));
}
template <>
__device__ __forceinline__ float2 Unpack2<__nv_bfloat16>(unsigned v) {
  return __bfloat1622float2(*reinterpret_cast<const __nv_bfloat162*>(&v));
}
template <>
__device__ __forceinline__ float2 Unpack2<float>(unsigned v) {  // (never used: float rows take the cp.async path)
  return make_float2(__uint_as_float(v), 0.0f);
}

// 4-byte back-pointer record (beam_width <= 256 and num_classes <= 256): [0,8) prev_self slot |
// [8,16) an_src slot | [16] ab_kind | [17,19) an_kind | [24,32) label. A fresh child has no previous
// self (0xff, never followed).
__device__ __forceinline__ unsigned PackRec32(unsigned prev_self, unsigned an_src, unsigned ab_kind,
                                              unsigned an_kind, unsigned label) {
  return (prev_self & 0xffu) | ((an_src & 0xffu) << 8) | (ab_kind << 16) | (an_kind << 17) | (label << 24);
}
// 8-byte form (PackRec word + label) -> 4-byte form
__device__ __forceinline__ unsigned Rec64To32(unsigned rec, unsigned label) {
  return PackRec32(rec & 0x7ffu, (rec >> 11) & 0x7ffu, (rec >> 22) & 1u, (rec >> 23) & 3u, label & 0xffu);
}

#ifdef CTCX_WITH_NORM
// ---------------------------------------------------------------------------------------------
// Kernel 1: per-row softmax normaliser off[t,b] = max_j x_j + logf(sum_{j in index order} expf(x_j - max))
// (decoder.h:71-80). One warp per row; lanes evaluate expf in parallel into a per-warp shared-memory
// chunk, then every lane accumulates the chunk in index order (the reference's order, so the float
// sum is bit-identical) with 16-byte broadcast loads -- 4x fewer issue slots than passing the terms
// around with shuffles, which is what bounded the first version of this kernel.
// ---------------------------------------------------------------------------------------------
// element offset of logits row `row` = t * B + b in a tensor whose time stride is `tstride` elements
__device__ __forceinline__ long long RowOffset(long long row, int B, int C, long long tstride) {
  const long long t = row / B;
  return t * tstride + (row - t * B) * C;
}

constexpr int kLogNormChunk = 1024;  // floats per warp per pass
static __global__ void __launch_bounds__(256) LogNormKernel(const float* __restrict__ logits,
                                                     float* __restrict__ off, long long rows, int C,
                                                     int B, long long tstride) {
  __shared__ unsigned long long s_tab[32];
  __shared__ __align__(16) float s_e[8][kLogNormChunk];
  LoadExpTable(s_tab, threadIdx.x, blockDim.x);
  __syncthreads();
  const int lane = threadIdx.x & 31;
  float* e = s_e[threadIdx.x >> 5];
  const long long warp_global = ((long long)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
  const long long nwarps = ((long long)gridDim.x * blockDim.x) >> 5;
  for (long long row = warp_global; row < rows; row += nwarps) {
    const float* x = logits + RowOffset(row, B, C, tstride);
    float mx = NegInf();
    for (int j = lane; j < C; j += 32) mx = fmaxf(mx, x[j]);
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) mx = fmaxf(mx, __shfl_xor_sync(kFull, mx, o));
    float sum = 0.0f;
    for (int base = 0; base < C; base += kLogNormChunk) {
      const int m = min(kLogNormChunk, C - base);
      const int m4 = (m + 3) & ~3;
      __syncwarp();  // the previous chunk has been summed by every lane
      for (int i = lane; i < m4; i += 32)
        e[i] = (i < m) ? ExpfExact(__fsub_rn(x[base + i], mx), s_tab) : 0.0f;
      __syncwarp();
      // adding the +0.0f padding of the last group leaves the (non-negative) sum unchanged
      for (int i = 0; i < m4; i += 4) {
        const float4 v = *reinterpret_cast<const float4*>(e + i);
        sum = __fadd_rn(__fadd_rn(__fadd_rn(__fadd_rn(sum, v.x), v.y), v.z), v.w);
      }
    }
    if (lane == 0) off[row] = __fadd_rn(mx, LogfExact(sum));
  }
}

// T = double (kernels.cc:275): the same normaliser through the double-precision exp()/log().
static __global__ void __launch_bounds__(256) LogNormKernelF64(const double* __restrict__ logits,
                                                        double* __restrict__ off, long long rows, int C,
                                                        int B, long long tstride) {
  __shared__ unsigned long long s_tab[256];
  for (int i = threadIdx.x; i < 256; i += blockDim.x) s_tab[i] = kCtcxExpTab[i];
  __syncthreads();
  const int lane = threadIdx.x & 31;
  const long long warp_global = ((long long)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
  const long long nwarps = ((long long)gridDim.x * blockDim.x) >> 5;
  for (long long row = warp_global; row < rows; row += nwarps) {
    const double* x = logits + RowOffset(row, B, C, tstride);
    double mx = __longlong_as_double((long long)0xfff0000000000000ull);
    for (int j = lane; j < C; j += 32) mx = fmax(mx, x[j]);
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) mx = fmax(mx, __shfl_xor_sync(kFull, mx, o));
    double sum = 0.0;
    for (int base = 0; base < C; base += 32) {
      const int j = base + lane;
      const double e = (j < C) ? ExpExactD(__dsub_rn(x[j], mx), s_tab) : 0.0;
      const int m = min(32, C - base);
      for (int k = 0; k < m; ++k) sum = __dadd_rn(sum, __shfl_sync(kFull, e, k));
    }
    if (lane == 0) off[row] = __dadd_rn(mx, LogExactD(sum));
  }
}

// Narrow-vocabulary variant (C <= 64): one THREAD per row. A CTA stages 256 consecutive rows (one
// contiguous, coalesced chunk of 256*C floats) in shared memory with an odd row stride (no bank
// conflicts), then every thread walks its own row: max, then the exp-sum in index order. 4x fewer
// issued instructions per row than the warp-per-row form, which is what keeps this kernel off the
// HBM roofline (the exact expf is ~25 instructions, half of them fp64).
constexpr int kLogNormRows = 256;
static __global__ void __launch_bounds__(kLogNormRows) LogNormRowKernel(const float* __restrict__ logits,
                                                                  float* __restrict__ off, long long rows,
                                                                  int C, int B, long long tstride) {
  extern __shared__ __align__(16) float lsm[];
  __shared__ unsigned long long s_tab[32];
  LoadExpTable(s_tab, threadIdx.x, blockDim.x);
  const int stride = C | 1;
  for (long long row0 = (long long)blockIdx.x * kLogNormRows; row0 < rows;
       row0 += (long long)gridDim.x * kLogNormRows) {
    const int nrow = (int)min((long long)kLogNormRows, rows - row0);
    const int total = nrow * C;
    const bool dense = (tstride == (long long)B * C);
    __syncthreads();  // previous tile fully consumed (and the table is loaded)
    for (int i = threadIdx.x; i < total; i += kLogNormRows) {
      const int r = i / C, c = i - r * C;
      lsm[r * stride + c] = dense ? logits[row0 * C + i] : logits[RowOffset(row0 + r, B, C, tstride) + c];
    }
    __syncthreads();
    if ((int)threadIdx.x < nrow) {
      const float* x = lsm + threadIdx.x * stride;
      float mx = x[0];
      for (int j = 1; j < C; ++j) mx = fmaxf(mx, x[j]);
      float sum = 0.0f;
      for (int j = 0; j < C; ++j) sum = __fadd_rn(sum, ExpfExact(__fsub_rn(x[j], mx), s_tab));
      off[row0 + threadIdx.x] = __fadd_rn(mx, LogfExact(sum));
    }
  }
}

// Pre-pass for wide vocabularies (32 < C <= 2048): the FUSED log-softmax normaliser and per-frame
// candidate-class top-k of the north star. One warp per (t,b) row reads the row once into registers
// (coalesced), computes off = max + log(sum exp) exactly as LogNormKernel does, and emits the `Ke` best
// non-blank classes ordered by (log-prob x_l - off descending, class ascending). The children of a
// beam entry above ANY threshold are a prefix of this order (fp addition is monotone), so the beam
// kernel finds them by binary search instead of scoring all C classes; and no entry can place more
// than beam_width children in the next beam, so the first Kc = 2*beam_width+2 classes (+1 sentinel,
// Ke = Kc+1) are all it ever needs (ctcx_beam_wide.cuh has the argument and the exact handling of the
// one tie case that reaches past the cut). Selection: keys in registers (NI per lane), the Ke-th
// largest key by a bitwise search with warp-wide counts, compaction by ballots, final order by rank
// counting.
template <typename IN, int NI>
__global__ void __launch_bounds__(256, 3) NormTopClassesKernel(const IN* __restrict__ logits,
                                                            float* __restrict__ off, long long rows, int C,
                                                            int blank, int Ke, int Ks,
                                                            float* __restrict__ srt_pl,
                                                            unsigned short* __restrict__ srt_cls, int B,
                                                            long long tstride) {
  // dynamic shared memory: [8 warps][NI*32] floats (the exp terms of a row), then [8 warps][Ke] u64
  extern __shared__ __align__(16) unsigned char nsm[];
  __shared__ unsigned long long s_tab[32];
  LoadExpTable(s_tab, threadIdx.x, blockDim.x);
  __syncthreads();
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  float* e = reinterpret_cast<float*>(nsm) + (size_t)warp * NI * 32;
  unsigned long long* buf = reinterpret_cast<unsigned long long*>(nsm + (size_t)8 * NI * 32 * sizeof(float)) + (size_t)warp * Ke;
  const unsigned lt = (1u << lane) - 1u;
  const int C4 = (C + 3) & ~3;
  const long long warp_global = ((long long)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
  const long long nwarps = ((long long)gridDim.x * blockDim.x) >> 5;
  for (long long row = warp_global; row < rows; row += nwarps) {
    const size_t x0 = (size_t)RowOffset(row, B, C, tstride);
    // the row, once, into registers (lane = class mod 32: coalesced)
    float v[NI];
    float mx = NegInf();
#pragma unroll
    for (int i = 0; i < NI; ++i) {
      const int j = i * 32 + lane;
      v[i] = (j < C) ? LoadLogit<IN>(logits, x0 + j) : NegInf();
      mx = fmaxf(mx, v[i]);
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) mx = fmaxf(mx, __shfl_xor_sync(kFull, mx, o));
    // log-softmax normaliser (decoder.h:71-80): exp terms to shared memory, summed in index order
    __syncwarp();  // the previous row is done with e and buf
#pragma unroll
    for (int i = 0; i < NI; ++i) {
      const int j = i * 32 + lane;
      if (j < C4) e[j] = (j < C) ? ExpfExact(__fsub_rn(v[i], mx), s_tab) : 0.0f;
    }
    __syncwarp();
    float sum = 0.0f;
    for (int i = 0; i < C4; i += 4) {
      const float4 q = *reinterpret_cast<const float4*>(e + i);
      sum = __fadd_rn(__fadd_rn(__fadd_rn(__fadd_rn(sum, q.x), q.y), q.z), q.w);
    }
    const float o = __fadd_rn(mx, LogfExact(sum));
    if (lane == 0) off[row] = o;
    // per-frame candidate classes: keys of the log-probs, 0 = blank / padding (every real key is > 0)
    unsigned k[NI];
#pragma unroll
    for (int i = 0; i < NI; ++i) {
      const int j = i * 32 + lane;
      k[i] = (j < C && j != blank) ? KeyOf(__fsub_rn(v[i], o)) : 0u;
    }
    // the Ke-th largest key, most significant bit first; stop early once some threshold separates
    // exactly Ke keys (the usual case long before bit 0)
    unsigned kth = 0u;
    bool exact = false;
    for (int bit = 31; bit >= 0; --bit) {
      const unsigned trial = kth | (1u << bit);
      int cnt = 0;
#pragma unroll
      for (int i = 0; i < NI; ++i) cnt += (k[i] >= trial) ? 1 : 0;
      cnt = __reduce_add_sync(kFull, cnt);
      if (cnt >= Ke) {
        kth = trial;
        if (cnt == Ke) { exact = true; break; }
      }
    }
    int ties_left = 0;  // keys equal to kth to take, lowest classes first (only if !exact)
    if (!exact) {
      int g = 0;
#pragma unroll
      for (int i = 0; i < NI; ++i) g += (k[i] > kth) ? 1 : 0;
      ties_left = Ke - __reduce_add_sync(kFull, g);
    }
    int base = 0;
#pragma unroll
    for (int i = 0; i < NI; ++i) {
      bool take = exact ? (k[i] >= kth) : (k[i] > kth);
      if (!exact) {
        const unsigned tm = __ballot_sync(kFull, k[i] == kth);
        if (k[i] == kth && __popc(tm & lt) < ties_left) take = true;
        ties_left -= min(ties_left, __popc(tm));
      }
      const unsigned sm = __ballot_sync(kFull, take);
      if (take)
        buf[base + __popc(sm & lt)] = ((unsigned long long)k[i] << 16) | (unsigned long long)(0xffff - (i * 32 + lane));
      base += __popc(sm);
    }
    __syncwarp();
    for (int q0 = lane; q0 < Ks; q0 += 32) {
      if (q0 < Ke) {
        const unsigned long long mine = buf[q0];
        int rank = 0;
        for (int q = 0; q < Ke; ++q) rank += (buf[q] > mine) ? 1 : 0;
        srt_pl[row * Ks + rank] = UnKey((unsigned)(mine >> 16));
        srt_cls[row * Ks + rank] = (unsigned short)(0xffff - (unsigned)(mine & 0xffffull));
      } else {
        srt_pl[row * Ks + q0] = NegInf();
        srt_cls[row * Ks + q0] = (unsigned short)0xffff;
      }
    }
  }
}

#endif  // CTCX_WITH_NORM

// Arithmetic of the score type R (float, or double for the reference's T = double registration,
// kernels.cc:275): explicit round-to-nearest operations, the monotone score -> integer key map and
// the (key, ~tie order) composite the survivors are ranked by.
template <typename R>
struct RealOps;
template <>
struct RealOps<float> {
  using Key = unsigned;
  using Comp = unsigned long long;  // key << 32 | ~order
  static constexpr int kKeyBits = 32;
  static constexpr Key kKeyMax = 0xffffffffu;
  static constexpr Key kKeyNegInf = 0x007fffffu;
  __device__ static __forceinline__ float NegInf() { return __int_as_float((int)0xff800000); }
  __device__ static __forceinline__ float Add(float a, float b) { return __fadd_rn(a, b); }
  __device__ static __forceinline__ float Sub(float a, float b) { return __fsub_rn(a, b); }
  __device__ static __forceinline__ Key KeyOf(float s) { return ctcx::KeyOf(s); }
  __device__ static __forceinline__ float UnKey(Key k) { return ctcx::UnKey(k); }
  __device__ static __forceinline__ int Bits(Key range) { return range == 0u ? 0 : 32 - __clz(range); }
  __device__ static __forceinline__ Comp MakeComp(Key k, unsigned not_order) {
    return ((unsigned long long)k << 32) | (unsigned long long)not_order;
  }
  __device__ static __forceinline__ bool Greater(Comp a, Comp b) { return a > b; }
  __device__ static __forceinline__ Key CompKey(Comp c) { return (unsigned)(c >> 32); }
  __device__ static __forceinline__ unsigned CompNotOrder(Comp c) { return (unsigned)(c & 0xffffffffull); }
};
template <>
struct RealOps<double> {
  using Key = unsigned long long;
  using Comp = ulonglong2;  // {key, ~order}
  static constexpr int kKeyBits = 64;
  static constexpr Key kKeyMax = 0xffffffffffffffffull;
  static constexpr Key kKeyNegInf = 0x000fffffffffffffull;
  __device__ static __forceinline__ double NegInf() { return __longlong_as_double((long long)0xfff0000000000000ull); }
  __device__ static __forceinline__ double Add(double a, double b) { return __dadd_rn(a, b); }
  __device__ static __forceinline__ double Sub(double a, double b) { return __dsub_rn(a, b); }
  __device__ static __forceinline__ Key KeyOf(double s) {  // -0.0 canonicalised to +0.0
    const unsigned long long u = (unsigned long long)__double_as_longlong(__dadd_rn(s, 0.0));
    return (u >> 63) ? ~u : (u | 0x8000000000000000ull);
  }
  __device__ static __forceinline__ double UnKey(Key k) {
    return __longlong_as_double((long long)((k >> 63) ? (k & 0x7fffffffffffffffull) : ~k));
  }
  __device__ static __forceinline__ int Bits(Key range) { return range == 0ull ? 0 : 64 - __clzll((long long)range); }
  __device__ static __forceinline__ Comp MakeComp(Key k, unsigned not_order) {
    return make_ulonglong2(k, (unsigned long long)not_order);
  }
  __device__ static __forceinline__ bool Greater(Comp a, Comp b) { return a.x > b.x || (a.x == b.x && a.y > b.y); }
  __device__ static __forceinline__ Key CompKey(Comp c) { return c.x; }
  __device__ static __forceinline__ unsigned CompNotOrder(Comp c) { return (unsigned)c.y; }
};

#ifdef CTCX_WITH_GENERIC
// ---------------------------------------------------------------------------------------------
// Kernel 2: the beam kernel.
// ---------------------------------------------------------------------------------------------


// Shared-memory carve-up, computed identically on host and device.
struct BeamSmem {
  // byte offsets
  size_t hash, phash;          // u64 [2][WMAX]
  size_t surv;                 // Comp [WMAX]
  size_t exptab;               // u64 [32]
  size_t total, blk, lab, ab, an;  // R [2][WMAX]
  size_t label;                // i32 [2][WMAX]
  size_t m_nt, m_nb, m_nl, m_nab, m_nan;  // R [WMAX]
  size_t m_key;                // Key [WMAX]
  size_t m_rec;                // u32 [WMAX]
  size_t m_pslot;              // i32 [WMAX]
  size_t risk, risk_new;       // i32 [WMAX]
  size_t wiped;                // u32 [WMAX] (0/1)
  size_t part;                 // i32 [NT]
  size_t htab;                 // i32 [2*WMAX]
  size_t hist;                 // u32 [256]
  size_t x;                    // R [2][Cpad]
  size_t kid;                  // u32 [kid_rows*kid_words], kid_rows = beam_width rounded up to 32
  size_t c_key;                // Key [cand_cap]
  size_t c_id;                 // u32 [cand_cap]
  size_t offv;                 // R [2]   this / the next frame's normaliser
  size_t keys;                 // Key [4] min key, max key, radix prefix
  size_t scal;                 // i32/u32 [32] scalars
  size_t bytes;

  __host__ __device__ static size_t Align(size_t v, size_t a) { return (v + a - 1) / a * a; }
  // rs = sizeof(R): 4 (float) or 8 (double); every 8-byte array precedes the 4-byte ones
  __host__ __device__ static int KidRows(int W) { return (W + 31) / 32 * 32; }
  __host__ __device__ void Init(int wmax, int nt, int C, int kid_words, int cand_cap, int rs, int W) {
    size_t o = 0;
    const size_t w = (size_t)wmax, r = (size_t)rs;
    const size_t cpad = Align((size_t)C, 4);
    hash = o; o += 2 * w * 8;
    phash = o; o += 2 * w * 8;
    surv = o; o += w * (rs == 4 ? 8 : 16);
    exptab = o; o += 32 * 8;
    keys = o; o += 4 * 8;
    offv = o; o += 2 * 8;
    total = o; o += 2 * w * r;
    blk = o; o += 2 * w * r;
    lab = o; o += 2 * w * r;
    ab = o; o += 2 * w * r;
    an = o; o += 2 * w * r;
    m_nt = o; o += w * r;
    m_nb = o; o += w * r;
    m_nl = o; o += w * r;
    m_nab = o; o += w * r;
    m_nan = o; o += w * r;
    m_key = o; o += w * r;
    x = o; o += 2 * cpad * r;
    c_key = o; o += Align((size_t)cand_cap * r, 8);
    label = o; o += 2 * w * 4;
    m_rec = o; o += w * 4;
    m_pslot = o; o += w * 4;
    risk = o; o += w * 4;
    risk_new = o; o += w * 4;
    wiped = o; o += w * 4;
    part = o; o += (size_t)nt * 4;
    htab = o; o += 2 * w * 4;
    hist = o; o += 256 * 4;
    kid = o; o += (size_t)KidRows(W) * (size_t)kid_words * 4;  // sized by the beam width, not the tier
    c_id = o; o += (size_t)cand_cap * 4;
    scal = o; o += 32 * 4;
    bytes = Align(o, 16);
  }
};

// indices into the scalar block
enum {
  kScNCand = 0, kScNRisk, kScChanged, kScK, kScE, kScNSurv, kScTotalItems, kScAnomaly
};
enum { kKeyMin = 0, kKeyMaxSlot = 1, kKeyPrefix = 2 };  // slots of the Key-typed scalar block

template <typename R, int WMAX, int NT>
__global__ void __launch_bounds__(NT) BeamKernelT(BeamParamsT<R> p) {
  using Ops = RealOps<R>;
  using Key = typename Ops::Key;
  using Comp = typename Ops::Comp;
  constexpr bool kIsF32 = (sizeof(R) == 4);
  extern __shared__ __align__(16) unsigned char smem[];
  constexpr int NWARP = NT / 32;
  constexpr int TS = 2 * WMAX;  // hash-table slots (power of two)
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const int b = blockIdx.x;
  const int W = p.W, C = p.C, T = p.T, B = p.B, KW = p.kid_words, blank = p.blank_index;
  const bool list_mode = p.cand_cap > 0;
  // streaming: frames already consumed by earlier chunks; this chunk contributes L more
  const int t_done = (p.t_done != nullptr) ? p.t_done[b] : 0;
  const int L = max(0, min(p.seq_len[b], p.Tcap - t_done));
  bool resume = (p.state != nullptr) && t_done > 0;
  if constexpr (!kIsF32) resume = resume && StreamResumable64(p.state, B, W, b);

  BeamSmem lay;
  lay.Init(WMAX, NT, C, KW, p.cand_cap, (int)sizeof(R), W);
  unsigned long long* s_hash = (unsigned long long*)(smem + lay.hash);
  unsigned long long* s_phash = (unsigned long long*)(smem + lay.phash);
  Comp* s_surv = (Comp*)(smem + lay.surv);
  unsigned long long* s_exptab = (unsigned long long*)(smem + lay.exptab);
  R* s_total = (R*)(smem + lay.total);
  R* s_blk = (R*)(smem + lay.blk);
  R* s_lab = (R*)(smem + lay.lab);
  R* s_ab = (R*)(smem + lay.ab);
  R* s_an = (R*)(smem + lay.an);
  int* s_label = (int*)(smem + lay.label);
  R* m_nt = (R*)(smem + lay.m_nt);
  R* m_nb = (R*)(smem + lay.m_nb);
  R* m_nl = (R*)(smem + lay.m_nl);
  R* m_nab = (R*)(smem + lay.m_nab);
  R* m_nan = (R*)(smem + lay.m_nan);
  Key* m_key = (Key*)(smem + lay.m_key);
  unsigned* m_rec = (unsigned*)(smem + lay.m_rec);
  int* m_pslot = (int*)(smem + lay.m_pslot);
  int* s_risk = (int*)(smem + lay.risk);
  int* s_risk_new = (int*)(smem + lay.risk_new);
  unsigned* s_wiped = (unsigned*)(smem + lay.wiped);
  int* s_part = (int*)(smem + lay.part);
  int* s_htab = (int*)(smem + lay.htab);
  unsigned* s_hist = (unsigned*)(smem + lay.hist);
  R* s_x = (R*)(smem + lay.x);
  unsigned* s_kid = (unsigned*)(smem + lay.kid);
  Key* c_key = (Key*)(smem + lay.c_key);
  unsigned* c_id = (unsigned*)(smem + lay.c_id);
  volatile int* sc = (volatile int*)(smem + lay.scal);
  int* sci = (int*)(smem + lay.scal);
  Key* s_keys = (Key*)(smem + lay.keys);
  R* s_offv = (R*)(smem + lay.offv);
  const int cpad = (int)BeamSmem::Align((size_t)C, 4);

  // ---- initial state: the root (decoder.h:212-227) ----
  LoadExpTable(s_exptab, tid, NT);
  for (int i = tid; i < TS; i += NT) s_htab[i] = -1;
  for (int i = tid; i < BeamSmem::KidRows(W) * KW; i += NT) s_kid[i] = 0u;
  for (int i = tid; i < WMAX; i += NT) s_wiped[i] = 0u;
  if (tid == 0 && !resume) {
    s_total[0] = (R)0;
    s_blk[0] = (R)0;
    s_lab[0] = Ops::NegInf();
    s_ab[0] = (R)0;  // empty alignment with probability 1 (entry.h:204-209)
    s_an[0] = Ops::NegInf();
    s_label[0] = -1;
    s_hash[0] = kRootHash;
    s_phash[0] = 0ull;
    sci[kScAnomaly] = 0;
  }
  int n = 1;  // members in the beam (uniform across the CTA)
  if (resume) {  // beam as the previous chunk left it (buffer 0: local frame 0 reads buffer 0)
    const StreamViewT<R> sv = StreamBlock<R>(p.state, B, W, b);
    n = sv.hdr->n;
    for (int i = tid; i < n; i += NT) {
      s_total[i] = sv.total[i]; s_blk[i] = sv.blk[i]; s_lab[i] = sv.lab[i];
      s_ab[i] = sv.ab[i]; s_an[i] = sv.an[i]; s_label[i] = sv.label[i];
      s_hash[i] = sv.hash[i]; s_phash[i] = sv.phash[i];
    }
    if (tid == 0) sci[kScAnomaly] = sv.hdr->flags & 1;
  }
  // row 0 of the logits
  if (L > 0) {
    const R* g = p.logits + (size_t)b * C;
    for (int l = tid; l < C; l += NT) s_x[l] = g[l];
    if (tid == 0) s_offv[0] = p.off[b];
  }
  __syncthreads();
  for (int i = tid; i < n; i += NT) {  // parent look-up table of the initial beam (the root, or the resumed one)
    unsigned h = (unsigned)s_hash[i] & (TS - 1);
    while (atomicCAS(&s_htab[h], -1, i) != -1) h = (h + 1) & (TS - 1);
  }
  __syncthreads();

  for (int t = 0; t < L; ++t) {
    const int cur = t & 1, nxt = cur ^ 1;
    const R* x = s_x + cur * cpad;
    const R off = s_offv[cur];
    const R* o_total = s_total + cur * WMAX;
    const R* o_blk = s_blk + cur * WMAX;
    const R* o_lab = s_lab + cur * WMAX;
    const R* o_ab = s_ab + cur * WMAX;
    const R* o_an = s_an + cur * WMAX;
    const int* o_label = s_label + cur * WMAX;
    const unsigned long long* o_hash = s_hash + cur * WMAX;
    const unsigned long long* o_phash = s_phash + cur * WMAX;

    // prefetch the next frame's row (consumed after the barrier that ends this frame)
    if (t + 1 < L) {
      const R* g = p.logits + (size_t)(t + 1) * (size_t)p.tstride + (size_t)b * C;
      R* dst = s_x + nxt * cpad;
      for (int l = tid; l < C; l += NT) {
        const unsigned sa = (unsigned)__cvta_generic_to_shared(dst + l);
        asm volatile("cp.async.ca.shared.global [%0], [%1], %2;\n" ::"r"(sa), "l"(g + l), "n"(sizeof(R)));
      }
      if (tid == 0) {
        const unsigned sa = (unsigned)__cvta_generic_to_shared(s_offv + nxt);
        asm volatile("cp.async.ca.shared.global [%0], [%1], %2;\n" ::"r"(sa),
                     "l"(p.off + (size_t)(t + 1) * B + b), "n"(sizeof(R)));
      }
      asm volatile("cp.async.commit_group;\n" ::);
    }
    if (tid == 0) {
      sci[kScNCand] = 0;
      sci[kScNRisk] = 0;
      s_keys[kKeyMin] = Ops::kKeyMax;
      s_keys[kKeyMaxSlot] = (Key)0;
      sci[kScNSurv] = 0;
    }
    __syncthreads();

    // ---- (A) update the existing members (decoder.h:95-143) ----
    const R xb = x[blank];
    const R pb = Ops::Sub(xb, off);
    Key my_key = (Key)0;
    bool suspect = false;
    if (tid < n) {
      const int i = tid;
      const int lbl = o_label[i];
      int pslot = -1;
      R v_nl = o_lab[i], v_an = Ops::NegInf();
      R rescore = Ops::NegInf();  // what the parent's re-score of this member would be (decoder.h:172-182)
      unsigned an_kind = kAnNone, an_src = kInvalidSlot;
      if (lbl >= 0) {
        const unsigned long long ph = o_phash[i];
        unsigned h = (unsigned)ph & (TS - 1);
        for (;;) {  // parent->Active() <=> the parent prefix is in the beam (decoder.h:97)
          const int s = s_htab[h];
          if (s < 0) break;
          if (o_hash[s] == ph) { pslot = s; break; }
          h = (h + 1) & (TS - 1);
        }
        const R xl = x[lbl];
        const R pl = Ops::Sub(xl, off);
        const R self_an = Ops::Add(o_an[i], pl);
        if (pslot >= 0) {
          const bool same = (lbl == o_label[pslot]);
          R base = same ? o_blk[pslot] : o_total[pslot];
          if (p.lm != nullptr)  // GetStateExpansionScore(b->state, .), decoder.h:103,114
            base = Ops::Add(base, p.lm[(size_t)(o_label[pslot] + 1) * C + lbl]);
          v_nl = Ops::Sub(Ops::Add(LogSumExp(o_lab[i], base, s_exptab), xl), off);  // :102-104,:113-115
          rescore = Ops::Add(pl, base);
          v_an = Ops::Add(o_ab[pslot], pl);
          an_kind = kAnParAb;
          an_src = (unsigned)pslot;
          if (!same) {
            const R c2 = Ops::Add(o_an[pslot], pl);
            if (c2 > v_an) { v_an = c2; an_kind = kAnParAn; }
          }
          if (self_an > v_an) { v_an = self_an; an_kind = kAnSelfAn; an_src = (unsigned)i; }
        } else {
          v_nl = Ops::Add(o_lab[i], pl);  // :125
          v_an = self_an;
          an_kind = kAnSelfAn;
          an_src = (unsigned)i;
        }
      }
      const R v_nb = Ops::Sub(Ops::Add(o_total[i], xb), off);  // :132
      const R c1 = Ops::Add(o_ab[i], pb), c2 = Ops::Add(o_an[i], pb);
      const unsigned ab_kind = (c2 > c1) ? kAbFromAn : kAbFromAb;
      const R v_nt = LogSumExp(v_nb, v_nl, s_exptab);  // :139
      m_nt[i] = v_nt;
      m_nb[i] = v_nb;
      m_nl[i] = v_nl;
      m_nab[i] = (c2 > c1) ? c2 : c1;
      m_nan[i] = v_an;
      my_key = Ops::KeyOf(v_nt);
      m_key[i] = my_key;
      m_rec[i] = PackRec((unsigned)i, an_src, ab_kind, an_kind);
      m_pslot[i] = pslot;
      // Precondition of the one event that is reported instead of modelled (DESIGN.md "Known deviation"):
      // were this member evicted and then re-scored by its parent, rounding would put the re-score ABOVE
      // the member's own total, so the reference could accept it again (decoder.h:189-199; it does so only
      // when the beam bottom ties with that total). Mathematically total >= re-score always. The utterance
      // is flagged if such a member then drops out of the beam (survivor collection, below).
      suspect = Ops::KeyOf(rescore) > my_key;
      if (pslot >= 0) {
        atomicOr(&s_kid[pslot * KW + (lbl >> 5)], 1u << (lbl & 31));
        if (pslot < i) {  // the parent's turn comes first: candidate for the revisit-wipe
          const int q = atomicAdd(&sci[kScNRisk], 1);
          s_risk[q] = i;
        }
      }
    }
    // min / max member key
    {
      Key kmin = (tid < n) ? my_key : Ops::kKeyMax, kmax = (tid < n) ? my_key : (Key)0;
#pragma unroll
      for (int o = 16; o > 0; o >>= 1) {
        kmin = min(kmin, __shfl_xor_sync(kFull, kmin, o));
        kmax = max(kmax, __shfl_xor_sync(kFull, kmax, o));
      }
      if (lane == 0 && warp * 32 < n) {
        atomicMin(&s_keys[kKeyMin], kmin);
        atomicMax(&s_keys[kKeyMaxSlot], kmax);
      }
    }
    __syncthreads();
    // the hash table has served this frame's look-ups: clear it for the next beam
    for (int i = tid; i < TS; i += NT) s_htab[i] = -1;

    // weakest a-priori threshold: with a full beam nothing at or below the W-th member total can
    // ever be admitted (decoder.h:151-155); keys are compared instead of floats from here on
    const Key th0 = (n == W) ? max(s_keys[kKeyMin], Ops::kKeyNegInf) : Ops::kKeyNegInf;

    // ---- (C) fresh children above the threshold (decoder.h:161-187) ----
    // evaluates (row, label) -> score key; used to build the list or, in streaming mode, directly
    auto eval_child = [&](int row, int l, Key& skey) -> bool {
      if (l == blank) return false;
      if ((s_kid[row * KW + (l >> 5)] >> (l & 31)) & 1u) return false;  // c.Active(): merged in (A)
      const R pl = Ops::Sub(x[l], off);
      R base = (l == o_label[row]) ? o_blk[row] : o_total[row];
      if (p.lm != nullptr) base = Ops::Add(base, p.lm[(size_t)(o_label[row] + 1) * C + l]);  // :171,:176,:182
      skey = Ops::KeyOf(Ops::Add(pl, base));  // :172-182
      return skey > th0;
    };
    {
      Key kmax = (Key)0, kmin = Ops::kKeyMax;
      int cnt_stream = 0;
      for (int row = warp; row < n; row += NWARP) {
        for (int l0 = 0; l0 < C; l0 += 32) {
          const int l = l0 + lane;
          Key skey = (Key)0;
          const bool ok = (l < C) && eval_child(row, l, skey);
          if (ok) { kmax = max(kmax, skey); kmin = min(kmin, skey); }
          if (list_mode) {
            const unsigned m = __ballot_sync(kFull, ok);
            if (m) {
              int base = 0;
              if (lane == 0) base = atomicAdd(&sci[kScNCand], __popc(m));
              base = __shfl_sync(kFull, base, 0);
              if (ok) {
                const int pos = base + __popc(m & ((1u << lane) - 1u));
                c_key[pos] = skey;
                c_id[pos] = ((unsigned)row << 16) | (unsigned)l;
              }
            }
          } else {
            cnt_stream += ok ? 1 : 0;
          }
        }
      }
#pragma unroll
      for (int o = 16; o > 0; o >>= 1) {
        kmin = min(kmin, __shfl_xor_sync(kFull, kmin, o));
        kmax = max(kmax, __shfl_xor_sync(kFull, kmax, o));
        cnt_stream += __shfl_xor_sync(kFull, cnt_stream, o);
      }
      if (lane == 0) {
        if (kmax != (Key)0) {
          atomicMin(&s_keys[kKeyMin], kmin);
          atomicMax(&s_keys[kKeyMaxSlot], kmax);
        }
        if (!list_mode && cnt_stream) atomicAdd(&sci[kScNCand], cnt_stream);
      }
    }
    __syncthreads();
    const int n_cand = sci[kScNCand];
    const int n_risk = sci[kScNRisk];

    // ---- (D) revisit-wipe fixed point (SURVEY A.4; DESIGN.md "Parallel formulation") ----
    bool any_wiped = false;
    if (n_risk > 0) {
      for (;;) {
        if (tid == 0) sci[kScChanged] = 0;
        for (int q = warp; q < n_risk; q += NWARP) {  // one warp per at-risk member
          const int m = s_risk[q];
          const int pb_slot = m_pslot[m];
          int verdict = 0;
          if (!s_wiped[pb_slot]) {
            const Key vkey = m_key[m];
            const unsigned idm = ((unsigned)pb_slot << 16) | (unsigned)o_label[m];
            int cnt = 0;
            for (int j = lane; j < n; j += 32) {
              const Key kj = m_key[j];
              cnt += (kj > vkey || (kj == vkey && j < m)) ? 1 : 0;
            }
            if (list_mode) {
              for (int c = lane; c < n_cand; c += 32) {
                const unsigned id = c_id[c];
                cnt += (c_key[c] > vkey && id < idm && !s_wiped[id >> 16]) ? 1 : 0;
              }
            } else {
              for (int row = 0; row <= pb_slot; ++row) {
                if (s_wiped[row]) continue;
                const int lend = (row == pb_slot) ? o_label[m] : C;
                for (int l = lane; l < lend; l += 32) {
                  Key skey;
                  cnt += (eval_child(row, l, skey) && skey > vkey) ? 1 : 0;
                }
              }
            }
#pragma unroll
            for (int o = 16; o > 0; o >>= 1) cnt += __shfl_xor_sync(kFull, cnt, o);
            verdict = (cnt >= W) ? 1 : 0;
          }
          if (lane == 0) s_risk_new[q] = verdict;
        }
        __syncthreads();
        for (int q = tid; q < n_risk; q += NT) {
          const int m = s_risk[q];
          const unsigned v = (unsigned)s_risk_new[q];
          if (s_wiped[m] != v) {
            s_wiped[m] = v;
            sci[kScChanged] = 1;
          }
        }
        __syncthreads();
        const int changed = sc[kScChanged];
        __syncthreads();  // everyone has read the flag before it is written again
        if (!changed) break;
      }
      for (int q = tid; q < n_risk; q += NT) {
        const int m = s_risk[q];
        if (s_wiped[m]) {
          sci[kScChanged] = 2;  // "some member is wiped"
        }
      }
      __syncthreads();
      any_wiped = (sc[kScChanged] == 2);
    }

    // ---- (E) next beam = first W items in (score desc, members before children, visiting order) ----
    // Items are the members (key m_key, tie order = slot) and the live candidates (tie order =
    // (row,label)). Radix select on the score key finds the W-th key; exact ties at that key are cut
    // by a second select on the tie order.
    auto live = [&](unsigned id) -> bool { return !any_wiped || !s_wiped[id >> 16]; };
    // for_each_item(f): f(score_key, order_key) for every item, each handled by exactly one thread
    auto for_each_item = [&](auto&& f) {
      for (int i = tid; i < n; i += NT) f(m_key[i], (unsigned)i);
      if (list_mode) {
        for (int c = tid; c < n_cand; c += NT) {
          const unsigned id = c_id[c];
          if (live(id)) f(c_key[c], 0x80000000u | id);
        }
      } else {
        for (int row = warp; row < n; row += NWARP) {
          if (any_wiped && s_wiped[row]) continue;
          for (int l = lane; l < C; l += 32) {
            Key skey;
            if (eval_child(row, l, skey)) f(skey, 0x80000000u | ((unsigned)row << 16) | (unsigned)l);
          }
        }
      }
    };
    // one radix-select level: among items with pred(), find the K-th largest of key(); returns the
    // selected key in sc[kScPrefix] (+lo), the number still to take at that key in sc[kScK] and the
    // number of items equal to it in sc[kScE]; sc[kScTotalItems] = number of items seen.
    auto radix_select = [&](Key lo, Key range, int K, auto&& keyfn) {
      const int nbits = Ops::Bits(range);
      int npass = (nbits + 7) / 8;
      if (npass == 0) npass = 1;
      if (tid == 0) { s_keys[kKeyPrefix] = (Key)0; sci[kScK] = K; }
      for (int pass = npass - 1; pass >= 0; --pass) {
        const int shift = pass * 8;
        for (int i = tid; i < 256; i += NT) s_hist[i] = 0u;
        __syncthreads();
        const Key prefix = s_keys[kKeyPrefix];
        for_each_item([&](Key skey, unsigned okey) {
          Key key;
          if (!keyfn(skey, okey, key)) return;
          const Key d = key - lo;
          const Key hi = (shift + 8 >= Ops::kKeyBits) ? (Key)0 : (d >> (shift + 8));
          if (hi == prefix) atomicAdd(&s_hist[(unsigned)(d >> shift) & 255u], 1u);
        });
        __syncthreads();
        if (warp == 0) {
          const int k = sci[kScK];
          unsigned h[8];
          unsigned loc = 0;
#pragma unroll
          for (int q = 0; q < 8; ++q) { h[q] = s_hist[lane * 8 + q]; loc += h[q]; }
          unsigned suf = loc;  // inclusive suffix sum over lanes >= lane
#pragma unroll
          for (int o = 1; o < 32; o <<= 1) {
            const unsigned v = __shfl_down_sync(kFull, suf, o);
            if (lane + o < 32) suf += v;
          }
          const unsigned above = suf - loc;  // items in higher lanes' bins
          if (pass == npass - 1 && lane == 0) sci[kScTotalItems] = (int)suf;
          if ((int)suf >= k && (int)above < k) {
            unsigned acc = above;
#pragma unroll
            for (int q = 7; q >= 0; --q) {
              if ((int)(acc + h[q]) >= k && (int)acc < k) {
                s_keys[kKeyPrefix] = (prefix << 8) | (Key)(lane * 8 + q);
                sci[kScK] = k - (int)acc;
                sci[kScE] = (int)h[q];
              }
              acc += h[q];
            }
          }
        }
        __syncthreads();
      }
    };

    const int n_items_upper = n + n_cand;  // before removing wiped rows
    Key cut_d = (Key)0;  // survivors: d > cut_d || (d == cut_d && ~okey >= cut_o)
    unsigned cut_o = 0u;
    const Key lo = s_keys[kKeyMin];
    bool take_all = (!any_wiped && n_items_upper <= W);
    if (!take_all) {
      const Key range = s_keys[kKeyMaxSlot] - lo;
      radix_select(lo, range, W, [&](Key skey, unsigned, Key& key) { key = skey; return true; });
      const int total_items = sc[kScTotalItems];
      if (total_items <= W) {
        take_all = true;
      } else {
        cut_d = s_keys[kKeyPrefix];
        const int k_rem = sc[kScK], e = sc[kScE];
        __syncthreads();
        if (e != k_rem) {  // exact ties straddle the beam boundary: cut them by tie order
          const Key want = cut_d + lo;
          radix_select((Key)0, (Key)0xffffffffu, k_rem, [&](Key skey, unsigned okey, Key& key) {
            key = (Key)(~okey);
            return skey == want;
          });
          cut_o = (unsigned)s_keys[kKeyPrefix];
          __syncthreads();
        }
      }
    }
    // collect survivors as 64-bit composites (score key, ~tie order): larger = earlier in the beam
    for_each_item([&](Key skey, unsigned okey) {
      const Key d = skey - lo;
      if (take_all || d > cut_d || (d == cut_d && ~okey >= cut_o)) {
        const int pos = atomicAdd(&sci[kScNSurv], 1);
        if (pos < WMAX) s_surv[pos] = Ops::MakeComp(skey, ~okey);
      } else if (okey == (unsigned)tid && suspect) {
        sci[kScAnomaly] = 1;  // a suspect member (see (A)) drops out of the beam: report the utterance
      }
    });
    __syncthreads();
    const int n_new = min(sci[kScNSurv], WMAX);

    // ---- (F) rank the survivors and write the next beam + back-pointers ----
    {
      static_assert(NT >= WMAX && NT % WMAX == 0, "one thread per beam slot is assumed");
      constexpr int PARTS = NT / WMAX;
      const int k = (PARTS > 1) ? (tid % WMAX) : tid;
      const int part = (PARTS > 1) ? (tid / WMAX) : 0;
      int cnt = 0;
      if (k < n_new && part < PARTS) {
        const Comp mine = s_surv[k];
        const int j0 = (int)((long long)n_new * part / PARTS), j1 = (int)((long long)n_new * (part + 1) / PARTS);
        for (int j = j0; j < j1; ++j) cnt += Ops::Greater(s_surv[j], mine) ? 1 : 0;
      }
      if (PARTS > 1) {
        s_part[tid] = cnt;
        __syncthreads();
        if (part == 0 && k < n_new) {
          for (int q = 1; q < PARTS; ++q) cnt += s_part[q * WMAX + k];
        }
      }
      R* w_total = s_total + nxt * WMAX;
      R* w_blk = s_blk + nxt * WMAX;
      R* w_lab = s_lab + nxt * WMAX;
      R* w_ab = s_ab + nxt * WMAX;
      R* w_an = s_an + nxt * WMAX;
      int* w_label = s_label + nxt * WMAX;
      unsigned long long* w_hash = s_hash + nxt * WMAX;
      unsigned long long* w_phash = s_phash + nxt * WMAX;
      if (part == 0 && k < n_new) {
        const int r = cnt;  // new slot
        const Comp comp = s_surv[k];
        const unsigned okey = ~Ops::CompNotOrder(comp);
        unsigned rec;
        int lbl;
        unsigned long long hsh;
        if (!(okey & 0x80000000u)) {  // surviving member
          const int i = (int)okey;
          w_total[r] = m_nt[i];
          w_blk[r] = m_nb[i];
          w_lab[r] = m_nl[i];
          w_ab[r] = m_nab[i];
          w_an[r] = m_nan[i];
          lbl = o_label[i];
          hsh = o_hash[i];
          w_phash[r] = o_phash[i];
          rec = m_rec[i];
        } else {  // fresh child (decoder.h:170-187)
          const int row = (int)((okey & 0x7fffffffu) >> 16);
          lbl = (int)(okey & 0xffffu);
          const R s = Ops::UnKey(Ops::CompKey(comp));
          const R pl = Ops::Sub(x[lbl], off);
          R v_an = Ops::Add(o_ab[row], pl);
          unsigned an_kind = kAnParAb;
          if (lbl != o_label[row]) {
            const R c2 = Ops::Add(o_an[row], pl);
            if (c2 > v_an) { v_an = c2; an_kind = kAnParAn; }
          }
          w_total[r] = s;
          w_blk[r] = Ops::NegInf();
          w_lab[r] = s;
          w_ab[r] = Ops::NegInf();
          w_an[r] = v_an;
          hsh = HashChild(o_hash[row], lbl);
          w_phash[r] = o_hash[row];
          rec = PackRec(kInvalidSlot, (unsigned)row, kAbFromAb, an_kind);
        }
        w_label[r] = lbl;
        w_hash[r] = hsh;
        if (p.bp32 != nullptr)
          p.bp32[((size_t)b * p.Tcap + (t_done + t)) * W + r] = Rec64To32(rec, (unsigned)lbl);
        else
          p.bp[((size_t)b * p.Tcap + (t_done + t)) * W + r] = make_uint2(rec, (unsigned)lbl);
        if (p.dbg_totals) p.dbg_totals[((size_t)b * T + t) * W + r] = w_total[r];
        // next frame's parent look-up table
        unsigned h = (unsigned)hsh & (TS - 1);
        while (atomicCAS(&s_htab[h], -1, r) != -1) h = (h + 1) & (TS - 1);
      }
      // un-mark this frame's member children and wipes
      if (tid < n) {
        const int ps = m_pslot[tid];
        if (ps >= 0) s_kid[ps * KW + (o_label[tid] >> 5)] = 0u;
        s_wiped[tid] = 0u;
      }
      if (p.dbg_n && tid == 0) p.dbg_n[(size_t)b * T + t] = n_new;
    }
    asm volatile("cp.async.wait_all;\n" ::);
    __syncthreads();
    n = n_new;
  }

  // ---- final beam (decoder.h:229-261): already sorted, the first P slots are the top paths ----
  {
    const int cur = L & 1;
    if (tid < p.P) {
      if (tid < n) {
        p.fin_total[(size_t)b * p.P + tid] = s_total[cur * WMAX + tid];
        p.fin_kind[(size_t)b * p.P + tid] = (s_ab[cur * WMAX + tid] > s_an[cur * WMAX + tid]) ? 1 : 0;
      } else {
        p.fin_total[(size_t)b * p.P + tid] = (R)0;
        p.fin_kind[(size_t)b * p.P + tid] = 0;
      }
    }
    const int overflow = (p.seq_len[b] > p.Tcap - t_done) ? 4 : 0;
    if (tid == 0) {
      p.fin_n[b] = n;
      p.flags[b] = (sci[kScAnomaly] ? 1 : 0) | ((p.P > n) ? 2 : 0) | overflow;
    }
    if (p.state != nullptr) {  // carry the beam to the next chunk
      const StreamViewT<R> sv = StreamBlock<R>(p.state, B, W, b);
      for (int i = tid; i < n; i += NT) {
        sv.total[i] = s_total[cur * WMAX + i]; sv.blk[i] = s_blk[cur * WMAX + i];
        sv.lab[i] = s_lab[cur * WMAX + i]; sv.ab[i] = s_ab[cur * WMAX + i];
        sv.an[i] = s_an[cur * WMAX + i]; sv.label[i] = s_label[cur * WMAX + i];
        sv.hash[i] = s_hash[cur * WMAX + i]; sv.phash[i] = s_phash[cur * WMAX + i];
      }
      if (tid == 0) {
        sv.hdr->n = n;
        sv.hdr->gap = 0u;
        sv.hdr->flags = (sci[kScAnomaly] ? 1 : 0) | overflow | (resume ? (sv.hdr->flags & 4) : 0);
        if constexpr (!kIsF32) {
          sv.hdr->type = 8;
          StreamMarkF64Step(p.state, W, b);
        }
      }
    }
    if (p.t_done != nullptr && tid == 0) p.t_done[b] = t_done + L;
  }
}

#endif  // CTCX_WITH_GENERIC

#ifdef CTCX_WITH_POST
// ---------------------------------------------------------------------------------------------
// Kernel 3: trace-back. One thread per (utterance, path) walks the back-pointer records from the
// last frame to the first, emitting the alignment (entry.h:137-152) and the decoded labels
// (entry.h:123-136, with optional repeat merging).
// ---------------------------------------------------------------------------------------------
// Back-pointer record formats: the generic / wide kernels write 8-byte records {packed word, label}
// (PackRec), the narrow fast kernel 4-byte ones (PackRec32, ctcx_beam_v4.cuh).
struct RecFields {
  unsigned prev_self, an_src, ab_kind, an_kind;
  int label;
};
__device__ __forceinline__ RecFields UnpackRec(const uint2 r) {
  return {r.x & 0x7ffu, (r.x >> 11) & 0x7ffu, (r.x >> 22) & 1u, (r.x >> 23) & 3u, (int)r.y};
}
__device__ __forceinline__ RecFields UnpackRec(const unsigned r) {
  return {r & 0xffu, (r >> 8) & 0xffu, (r >> 16) & 1u, (r >> 17) & 3u, (int)(r >> 24)};
}


template <typename REC>
__global__ void __launch_bounds__(128) TraceKernel(TraceParams p) {
  const int idx = blockIdx.x * blockDim.x + threadIdx.x;
  if (idx >= p.B * p.P) return;
  const int b = idx / p.P, path = idx - b * p.P;
  const int L = max(0, min(p.seq_len[b], p.T));  // out-of-range lengths are reported by the host, not walked
  int* ali = p.ali + (size_t)idx * p.T;
  int* dec = p.dec + (size_t)idx * p.T;
  if (path >= p.fin_n[b] || L <= 0) {
    p.dec_len[idx] = 0;
    p.ali_len[idx] = 0;
    return;
  }
  int slot = path;
  int kind_ab = p.fin_kind[idx];
  const REC* bp = reinterpret_cast<const REC*>(p.bp) + (size_t)b * p.T * p.W;
  for (int t = L - 1; t >= 0; --t) {
    const RecFields r = UnpackRec(bp[(size_t)t * p.W + min(slot, p.W - 1)]);
    if (kind_ab) {
      ali[t] = p.blank_label;
      dec[t] = -1;
      kind_ab = (r.ab_kind == kAbFromAb) ? 1 : 0;
      slot = (int)r.prev_self;
    } else {
      ali[t] = r.label;
      if (r.an_kind == kAnSelfAn) {
        dec[t] = -1;
        slot = (int)r.prev_self;
      } else {
        dec[t] = r.label;  // a new label was emitted at this frame
        slot = (int)r.an_src;
        kind_ab = (r.an_kind == kAnParAb) ? 1 : 0;
      }
    }
  }
  int pos = 0, prev = -1;
  for (int t = 0; t < L; ++t) {
    const int v = dec[t];
    if (v >= 0) {
      if (!p.merge_repeated || v != prev) dec[pos++] = v;
      prev = v;
    }
  }
  p.dec_len[idx] = pos;
  p.ali_len[idx] = L;
}

// Warp-cooperative trace-back (used when there are too few walks to hide latency by themselves;
// TraceKernel above is the simple form). One warp per (utterance, path). The walk is a dependent
// chain (the slot at frame t-1 comes out of the record at frame t), but WHICH ROWS are needed next is
// known in advance: the warp streams blocks of `rows` consecutive back-pointer rows [rows x W x 8 B,
// contiguous in memory] into a double buffer in shared memory with cp.async, one block ahead of the
// walk, so a step is one shared-memory broadcast read plus a few ALU operations instead of a
// dependent trip to L2/HBM. Symbols are collected 32 frames at a time in registers and written as
// coalesced rows; the decoded labels are compacted with warp ballots.
// When a row of records is a multiple of 16 bytes (beam 100 with 4-byte records: 400 B) a block of rows is
// ONE contiguous, 16-byte aligned span of HBM: it is fetched by a single bulk-copy instruction
// (cp.async.bulk, the TMA unit's 1-D form) issued by one lane and signalled on an mbarrier, instead
// of one 4-byte cp.async per record (3 200 per block).
template <typename REC, int WARPS>
__global__ void __launch_bounds__(WARPS * 32) TraceWarpKernel(TraceParams p, int rows_log2, int use_bulk) {
  extern __shared__ __align__(16) unsigned char tsm[];
  __shared__ __align__(8) unsigned long long s_mbar[WARPS][2];
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const int idx = blockIdx.x * WARPS + warp;
  if (idx >= p.B * p.P) return;
  const int b = idx / p.P, path = idx - b * p.P;
  const int L = max(0, min(p.seq_len[b], p.T));  // out-of-range lengths are reported by the host, not walked
  int* ali = p.ali + (size_t)idx * p.T;
  int* dec = p.dec + (size_t)idx * p.T;
  if (path >= p.fin_n[b] || L <= 0) {
    if (lane == 0) {
      p.dec_len[idx] = 0;
      p.ali_len[idx] = 0;
    }
    return;
  }
  const int W = p.W;
  const int R = 1 << rows_log2;
  REC* buf = reinterpret_cast<REC*>(tsm) + (size_t)warp * 2 * R * W;
  const REC* bp = reinterpret_cast<const REC*>(p.bp) + (size_t)b * p.T * W;
  const unsigned mbar0 = (unsigned)__cvta_generic_to_shared(&s_mbar[warp][0]);
  if (use_bulk) {
    if (lane == 0) {
      asm volatile("mbarrier.init.shared::cta.b64 [%0], 1;\n" ::"r"(mbar0));
      asm volatile("mbarrier.init.shared::cta.b64 [%0], 1;\n" ::"r"(mbar0 + 8u));
      asm volatile("fence.mbarrier_init.release.cluster;\n" ::: "memory");
    }
    __syncwarp();
  }
  // block k holds frames [k*R, min(L, (k+1)*R)); blocks are walked from the last one down
  auto fetch_block = [&](int k) {
    if (k >= 0) {
      const int t0 = k << rows_log2;
      const int nrec = (min(L, t0 + R) - t0) * W;
      const REC* src = bp + (size_t)t0 * W;
      const unsigned dst = (unsigned)__cvta_generic_to_shared(buf + (size_t)(k & 1) * R * W);
      if (use_bulk) {
        if (lane == 0) {
          const unsigned bytes = (unsigned)nrec * (unsigned)sizeof(REC);
          const unsigned mbar = mbar0 + 8u * (unsigned)(k & 1);
          // the buffer was last read through ordinary loads (two blocks ago): order them before the
          // asynchronous-proxy write
          asm volatile("fence.proxy.async.shared::cta;\n" ::: "memory");
          asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;\n" ::"r"(mbar), "r"(bytes) : "memory");
          asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];\n" ::"r"(dst),
                       "l"(src), "r"(bytes), "r"(mbar)
                       : "memory");
        }
      } else {
        for (int i = lane; i < nrec; i += 32)
          asm volatile("cp.async.ca.shared.global [%0], [%1], %2;\n" ::"r"(dst + (unsigned)sizeof(REC) * (unsigned)i),
                       "l"(src + i), "n"(sizeof(REC)));
      }
    }
    if (!use_bulk) asm volatile("cp.async.commit_group;\n" ::);
  };
  // wait until block k has landed (bulk path: the k-th use of its buffer flips the barrier's phase)
  const int last_block = (L - 1) >> rows_log2;
  auto wait_block = [&](int k) {
    if (use_bulk) {
      const unsigned mbar = mbar0 + 8u * (unsigned)(k & 1);
      const unsigned parity = (unsigned)(((last_block - k) >> 1) & 1);
      unsigned done = 0;
      while (!done) {
        asm volatile(
            "{\n .reg .pred p;\n mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n selp.u32 %0, 1, 0, p;\n}\n"
            : "=r"(done)
            : "r"(mbar), "r"(parity)
            : "memory");
      }
    } else {
      asm volatile("cp.async.wait_group 1;\n" ::);
    }
  };
  fetch_block(last_block);
  int slot = path;
  int kind_ab = p.fin_kind[idx];
  int a_val = 0, d_val = -1;  // this lane's symbols of the current 32-frame store block
  for (int k = last_block; k >= 0; --k) {
    fetch_block(k - 1);  // next block in flight while this one is walked
    wait_block(k);       // block k has landed
    __syncwarp();
    const REC* blk = buf + (size_t)(k & 1) * R * W;
    const int t_lo = k << rows_log2;
    for (int t = min(L, t_lo + R) - 1; t >= t_lo; --t) {
      const RecFields r = UnpackRec(blk[(t - t_lo) * W + min(slot, W - 1)]);
      int sym_a, sym_d = -1;
      if (kind_ab) {  // entry.h:133-136: a blank frame
        sym_a = p.blank_label;
        kind_ab = (r.ab_kind == kAbFromAb) ? 1 : 0;
        slot = (int)r.prev_self;
      } else {
        sym_a = r.label;
        if (r.an_kind == kAnSelfAn) {
          slot = (int)r.prev_self;
        } else {
          sym_d = r.label;  // a new label was emitted at this frame
          slot = (int)r.an_src;
          kind_ab = (r.an_kind == kAnParAb) ? 1 : 0;
        }
      }
      if (lane == (t & 31)) {
        a_val = sym_a;
        d_val = sym_d;
      }
      if ((t & 31) == 0) {  // frames [t, t+32) complete: coalesced store
        const int tt = t + lane;
        if (tt < L) {
          ali[tt] = a_val;
          dec[tt] = d_val;
        }
      }
    }
    __syncwarp();  // buffer (k & 1) is refilled two iterations from now
  }
  __syncwarp();
  // forward compaction of the new labels (entry.h:123-136, optional repeat merging)
  int base = 0, carry = -1;
  for (int t0 = 0; t0 < L; t0 += 32) {
    const int tt = t0 + lane;
    const int v = (tt < L) ? dec[tt] : -1;
    const unsigned mask = __ballot_sync(kFull, v >= 0);
    const unsigned pm = mask & ((1u << lane) - 1u);
    const int prev_lane = pm ? (31 - __clz(pm)) : 0;
    int prev_val = __shfl_sync(kFull, v, prev_lane);
    if (!pm) prev_val = carry;
    const bool keep = (v >= 0) && (!p.merge_repeated || v != prev_val);
    const unsigned kmask = __ballot_sync(kFull, keep);
    __syncwarp();
    if (keep) dec[base + __popc(kmask & ((1u << lane) - 1u))] = v;
    base += __popc(kmask);
    if (mask) carry = __shfl_sync(kFull, v, 31 - __clz(mask));
  }
  if (lane == 0) {
    p.dec_len[idx] = base;
    p.ali_len[idx] = L;
  }
}

// ---------------------------------------------------------------------------------------------
// Kernels 4/5: sparse packing (kernels.cc:163-257). ScanKernel: per path, exclusive prefix sums of
// the lengths over the batch + totals + maxima. PackKernel: indices [b,pos], values, shapes.
// ---------------------------------------------------------------------------------------------

static __global__ void __launch_bounds__(1024) ScanKernel(ScanParams p) {
  __shared__ long long s_sum[2][32];
  __shared__ int s_max[2][32];
  const int path = blockIdx.x;
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const int per = (p.B + 1023) / 1024;
  const int b0 = min(p.B, tid * per), b1 = min(p.B, b0 + per);
  long long sum[2] = {0, 0};
  int mx[2] = {0, 0};
  for (int b = b0; b < b1; ++b) {
    const int d = p.dec_len[(size_t)b * p.P + path], a = p.ali_len[(size_t)b * p.P + path];
    sum[0] += d; sum[1] += a;
    mx[0] = max(mx[0], d); mx[1] = max(mx[1], a);
  }
  long long incl[2];
#pragma unroll
  for (int w = 0; w < 2; ++w) {
    long long v = sum[w];
    int m = mx[w];
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
      const long long u = __shfl_up_sync(kFull, v, o);
      if (lane >= o) v += u;
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) m = max(m, __shfl_xor_sync(kFull, m, o));
    incl[w] = v;
    if (lane == 31) s_sum[w][warp] = v;
    if (lane == 0) s_max[w][warp] = m;
  }
  __syncthreads();
  if (warp == 0) {
#pragma unroll
    for (int w = 0; w < 2; ++w) {
      long long v = s_sum[w][lane];
      int m = s_max[w][lane];
#pragma unroll
      for (int o = 1; o < 32; o <<= 1) {
        const long long u = __shfl_up_sync(kFull, v, o);
        if (lane >= o) v += u;
      }
#pragma unroll
      for (int o = 16; o > 0; o >>= 1) m = max(m, __shfl_xor_sync(kFull, m, o));
      s_sum[w][lane] = v;  // inclusive over warps
      if (lane == 31) p.sizes[(w * 2) * p.P + path] = v;
      if (lane == 0) p.sizes[(w * 2 + 1) * p.P + path] = m;
    }
  }
  __syncthreads();
#pragma unroll
  for (int w = 0; w < 2; ++w) {
    long long base = incl[w] - sum[w] + (warp > 0 ? s_sum[w][warp - 1] : 0);
    long long* out = (w == 0 ? p.dec_off : p.ali_off) + (size_t)path * p.B;
    for (int b = b0; b < b1; ++b) {
      out[b] = base;
      base += (w == 0) ? p.dec_len[(size_t)b * p.P + path] : p.ali_len[(size_t)b * p.P + path];
    }
  }
}


// Pointer table of the COMPACT output layout: all outputs of a decode as consecutive slices of one
// int64 buffer -- per path: decoded indices [n,2], values [n], shape [2], alignment indices, values,
// shape; then log_probability [B,P] (float32 pairs or float64 in int64 slots) -- computed on the device
// from the sizes the scan left there, so that the pack can be enqueued before the host knows them.
static __global__ void PackTableKernel(const long long* sizes, int B, int P, int real_bytes, long long* buf,
                                       unsigned long long buf_elems, long long** ptrs, int* overflow) {
  if (threadIdx.x != 0 || blockIdx.x != 0) return;
  unsigned long long o = 0;
  for (int p = 0; p < P; ++p) {
    const unsigned long long nd = (unsigned long long)sizes[0 * P + p], na = (unsigned long long)sizes[2 * P + p];
    ptrs[0 * P + p] = buf + o; o += 2 * nd;
    ptrs[1 * P + p] = buf + o; o += nd;
    ptrs[2 * P + p] = buf + o; o += 2;
    ptrs[3 * P + p] = buf + o; o += 2 * na;
    ptrs[4 * P + p] = buf + o; o += na;
    ptrs[5 * P + p] = buf + o; o += 2;
  }
  ptrs[6 * P] = buf + o;
  o += (real_bytes == 8) ? (unsigned long long)B * P : ((unsigned long long)B * P + 1) / 2;
  if (o > buf_elems) *overflow = 1;
}

static __global__ void __launch_bounds__(128) PackKernel(PackParams p) {
  if (p.skip != nullptr && *p.skip != 0) return;
  const int b = blockIdx.x, path = blockIdx.y;
  const size_t row = (size_t)b * p.P + path;
  {
    const int n = p.dec_len[row];
    const long long o = p.dec_off[(size_t)path * p.B + b];
    long long* idx = p.ptrs[0 * p.P + path];
    long long* val = p.ptrs[1 * p.P + path];
    const int* src = p.dec + row * p.T;
    for (int i = threadIdx.x; i < n; i += blockDim.x) {
      idx[2 * (o + i)] = b;
      idx[2 * (o + i) + 1] = i;
      val[o + i] = src[i];
    }
  }
  {
    const int n = p.ali_len[row];
    const long long o = p.ali_off[(size_t)path * p.B + b];
    long long* idx = p.ptrs[3 * p.P + path];
    long long* val = p.ptrs[4 * p.P + path];
    const int* src = p.ali + row * p.T;
    for (int i = threadIdx.x; i < n; i += blockDim.x) {
      idx[2 * (o + i)] = b;
      idx[2 * (o + i) + 1] = i;
      val[o + i] = src[i];
    }
  }
  if (threadIdx.x == 0) {
    void* lp = (p.log_prob != nullptr) ? p.log_prob : (void*)p.ptrs[6 * p.P];
    if (p.real_bytes == 8)  // kernels.cc:87-89
      ((double*)lp)[row] = ((const double*)p.fin_total)[row];
    else
      ((float*)lp)[row] = ((const float*)p.fin_total)[row];
    if (b == 0) {
      long long* ds = p.ptrs[2 * p.P + path];
      long long* as = p.ptrs[5 * p.P + path];
      ds[0] = p.B; ds[1] = p.sizes[1 * p.P + path];  // kernels.cc:236-237
      as[0] = p.B; as[1] = p.sizes[3 * p.P + path];  // kernels.cc:253-254
    }
  }
}

// Test hook: element-wise evaluation of the exact math functions.
// op 0: expf, 1: log1pf, 2: logf, 3: LogSumExp(x, 0), 4: LogSumExp(0, x)
static __global__ void MathTestKernel(int op, const float* x, float* y, int n) {
  __shared__ unsigned long long s_tab[32];
  LoadExpTable(s_tab, threadIdx.x, blockDim.x);
  __syncthreads();
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  const float v = x[i];
  y[i] = (op == 0) ? ExpfExact(v, s_tab) : (op == 1) ? Log1pfExact(v) : (op == 2) ? LogfExact(v)
       : (op == 3) ? LogSumExp(v, 0.0f, s_tab) : LogSumExp(0.0f, v, s_tab);
}

// op 0: exp (x <= 0), 1: log (x >= 1), 2: LogSumExp(x, 0) of the double path
static __global__ void MathTestKernelF64(int op, const double* x, double* y, int n) {
  __shared__ unsigned long long s_tab[256];
  __shared__ unsigned long long s_tabf[32];
  for (int i = threadIdx.x; i < 256; i += blockDim.x) s_tab[i] = kCtcxExpTab[i];
  LoadExpTable(s_tabf, threadIdx.x, blockDim.x);
  __syncthreads();
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  const double v = x[i];
  y[i] = (op == 0) ? ExpExactD(v, s_tab) : (op == 1) ? LogExactD(v) : LogSumExp(v, 0.0, s_tabf);
}

#endif  // CTCX_WITH_POST

}  // namespace ctcx
