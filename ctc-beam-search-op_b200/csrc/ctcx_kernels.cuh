// Device helpers shared by the kernel families of the CTC "extended" beam-search decode (sm_100a):
// back-pointer record formats, score keys, prefix hashes, logit loads, the streamed-state blocks and
// the score-type arithmetic. Each family of kernels lives in the translation unit that launches it:
//   k_generic.cu  softmax normalisers (LogNorm*Kernel) and the generic beam kernel
//                 (BeamKernelT, ctcx_beam_generic.cuh)
//   k_narrow.cu   narrow-vocabulary fast beam kernel (BeamKernelV4, ctcx_beam_v4.cuh)
//   k_wide.cu     wide-vocabulary pre-pass (NormTopClassesKernel) and fast beam kernel
//                 (BeamKernelWide, ctcx_beam_wide.cuh)
//   k_post.cu     trace-back, scan, pack and the math test hooks
//
// What each kernel replaces in the reference (paths relative to
// tensorflow_ctc_ext_beam_search_decoder/cc/):
//   LogNormKernel   util/ctc_ext_beam_search_decoder.h:71-80   softmax normaliser of Step()
//   BeamKernel*     util/ctc_ext_beam_search_decoder.h:84-209  Step(): extract/sort, member update,
//                   grow + prune; util/ctc_beam_entry.h (BeamEntry trie, BeamProbability,
//                   AddAlignmentCandidate); gtl::TopN; util/ctc_loss_util.h LogSumExp
//   TraceKernel     util/ctc_ext_beam_search_decoder.h:229-261 TopPaths +
//                   util/ctc_beam_entry.h:123-152 LabelSeq / AlignmentLabelSeq
//   ScanKernel/PackKernel  kernels/ctc_ext_beam_search_decoder_kernels.cc:163-257
//                   StoreAllDecodedSequences
//
// The beam kernels do NOT translate the reference's sequential trie walk. They implement the
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

// element offset of logits row `row` = t * B + b in a tensor whose time stride is `tstride` elements
__device__ __forceinline__ long long RowOffset(long long row, int B, int C, long long tstride) {
  const long long t = row / B;
  return t * tstride + (row - t * B) * C;
}

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

}  // namespace ctcx
