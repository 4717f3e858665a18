// Translation unit of the wide-vocabulary fast path: the fused normaliser + per-frame class
// selection pre-pass (NormTopClassesKernel) and the wide beam kernel (ctcx_beam_wide.cuh).
#include "ctcx_beam_wide.cuh"
#include "ctcx_launch.h"

#include <algorithm>

namespace ctcx {

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

namespace {
constexpr size_t kWideSmemMax = 200 * 1024;  // the most WideFastShape admits
constexpr int kKeMax = 2 * 256 + 3;          // WideKe at beam_width 256, the widest WideFastShape admits

// exp terms + selection buffer per warp
constexpr size_t TopClassesSmem(int NI, int Ke) { return (size_t)8 * NI * 32 * sizeof(float) + (size_t)8 * Ke * 8; }

template <typename IN, int NI>
LaunchStatus TopClassesNI(const void* logits, float* off, long long rows, int C, int blank, int Ke, int Ks,
                          float* srt_pl, unsigned short* srt_cls, int B, long long tstride, cudaStream_t stream) {
  auto kern = NormTopClassesKernel<IN, NI>;
  static KernelSetup setup;
  cudaError_t e = setup.RaiseSmemLimit((const void*)kern, TopClassesSmem(NI, kKeMax));
  if (e != cudaSuccess) return LaunchFrom(e, "shared-memory limit of NormTopClassesKernel");
  const size_t smem = TopClassesSmem(NI, Ke);
  const long long blocks = std::min<long long>((rows + 7) / 8, (long long)SmCount() * 16);
  kern<<<(unsigned)blocks, 256, smem, stream>>>(reinterpret_cast<const IN*>(logits), off, rows, C, blank, Ke, Ks,
                                                srt_pl, srt_cls, B, tstride);
  return LaunchFrom(cudaGetLastError(), "NormTopClassesKernel launch");
}

template <typename IN>
LaunchStatus TopClassesTyped(const void* logits, float* off, long long rows, int C, int blank, int W, float* srt_pl,
                             unsigned short* srt_cls, int B, long long tstride, cudaStream_t stream) {
  const int Ke = WideKe(W, C), Ks = WideKs(W, C), ni = (C + 31) / 32;
#define CTCX_TOPC(N) TopClassesNI<IN, N>(logits, off, rows, C, blank, Ke, Ks, srt_pl, srt_cls, B, tstride, stream)
  if (ni <= 2) return CTCX_TOPC(2);
  if (ni <= 4) return CTCX_TOPC(4);
  if (ni <= 8) return CTCX_TOPC(8);
  if (ni <= 16) return CTCX_TOPC(16);
  if (ni <= 32) return CTCX_TOPC(32);
  return CTCX_TOPC(64);
#undef CTCX_TOPC
}

template <typename IN, int WMAX, bool TIMING>
LaunchStatus LaunchOne(const BeamParams& p, size_t smem, cudaStream_t stream) {
  auto kern = BeamKernelWide<IN, WMAX, 256, TIMING>;
  static KernelSetup setup;
  const cudaError_t e = setup.RaiseSmemLimit((const void*)kern, kWideSmemMax);
  if (e != cudaSuccess) return LaunchFrom(e, "shared-memory limit of BeamKernelWide");
  kern<<<p.B, 256, smem, stream>>>(p);
  return LaunchFrom(cudaGetLastError(), "BeamKernelWide launch");
}

template <typename IN>
LaunchStatus LaunchTyped(const BeamParams& p, int wmax, size_t smem, cudaStream_t stream) {
  if constexpr (sizeof(IN) == 4) {
    if (p.dbg_cycles != nullptr) {  // timing build: float32 inputs only
      switch (wmax) {
        case 32: return LaunchOne<IN, 32, true>(p, smem, stream);
        case 128: return LaunchOne<IN, 128, true>(p, smem, stream);
        default: return LaunchOne<IN, 256, true>(p, smem, stream);
      }
    }
  }
  switch (wmax) {
    case 32: return LaunchOne<IN, 32, false>(p, smem, stream);
    case 128: return LaunchOne<IN, 128, false>(p, smem, stream);
    default: return LaunchOne<IN, 256, false>(p, smem, stream);
  }
}
}  // namespace

// WideKc = sorted classes the beam kernel uses, WideKs = row stride of the sorted arrays (Kc + one
// sentinel when classes are left out, rounded up to 8).
int WideKc(int W, int C) { return std::min(C - 1, 2 * W + 2); }
int WideKe(int W, int C) { return std::min(C - 1, WideKc(W, C) + 1); }
int WideKs(int W, int C) { return (WideKe(W, C) + 7) / 8 * 8; }
bool WideFastShape(int W, int C) {
  if (C <= 32 || C > 2048 || W > 256) return false;
  BeamSmemWide lay;
  lay.Init(TierOf(W), W * WideKc(W, C), C, WideKs(W, C));
  return lay.bytes <= kWideSmemMax;
}

LaunchStatus LaunchNormTopClasses(const void* logits, int in_dtype, float* off, long long rows, int C, int blank,
                                  int W, float* srt_pl, unsigned short* srt_cls, int B, long long tstride,
                                  cudaStream_t stream) {
  switch (in_dtype) {
    case kInF32: return TopClassesTyped<float>(logits, off, rows, C, blank, W, srt_pl, srt_cls, B, tstride, stream);
    case kInF16: return TopClassesTyped<__half>(logits, off, rows, C, blank, W, srt_pl, srt_cls, B, tstride, stream);
    case kInBF16: return TopClassesTyped<__nv_bfloat16>(logits, off, rows, C, blank, W, srt_pl, srt_cls, B, tstride, stream);
    default: return {kLaunchUnsupported, cudaSuccess, ""};
  }
}

LaunchStatus LaunchBeamWide(BeamParams& p, int in_dtype, cudaStream_t stream) {
  if (!WideFastShape(p.W, p.C) || p.srt_pl == nullptr) return {kLaunchUnsupported, cudaSuccess, ""};
  p.kid_words = (p.C + 31) / 32;
  p.Kc = WideKc(p.W, p.C);
  p.Cs = WideKs(p.W, p.C);
  p.cand_cap = p.W * p.Kc;
  const int wmax = TierOf(p.W);
  BeamSmemWide lay;
  lay.Init(wmax, p.cand_cap, p.C, p.Cs);
  switch (in_dtype) {
    case kInF32: return LaunchTyped<float>(p, wmax, lay.bytes, stream);
    case kInF16: return LaunchTyped<__half>(p, wmax, lay.bytes, stream);
    case kInBF16: return LaunchTyped<__nv_bfloat16>(p, wmax, lay.bytes, stream);
    default: return {kLaunchUnsupported, cudaSuccess, ""};
  }
}

}  // namespace ctcx
