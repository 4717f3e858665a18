// Translation unit of the wide-vocabulary fast path: the fused normaliser + per-frame class
// selection pre-pass (NormTopClassesKernel) and the wide beam kernel (ctcx_beam_wide.cuh).
#define CTCX_WITH_NORM
#include "ctcx_beam_wide.cuh"
#include "ctcx_launch.h"

#include <algorithm>

namespace ctcx {

namespace {
template <typename IN, int NI>
LaunchStatus TopClassesNI(const void* logits, float* off, long long rows, int C, int blank, int Ke, int Ks,
                          float* srt_pl, unsigned short* srt_cls, int B, long long tstride, cudaStream_t stream) {
  auto kern = NormTopClassesKernel<IN, NI>;
  const size_t smem = (size_t)8 * NI * 32 * sizeof(float) + (size_t)8 * Ke * 8;  // exp terms + selection buffer per warp
  cudaError_t e = cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
  if (e != cudaSuccess) return LaunchFrom(e, "cudaFuncSetAttribute(NormTopClassesKernel)");
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
  cudaError_t e = cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
  if (e != cudaSuccess) return LaunchFrom(e, "cudaFuncSetAttribute(BeamKernelWide)");
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
  return lay.bytes <= 200 * 1024;
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
