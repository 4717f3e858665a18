// Translation unit of the generic path: the stand-alone softmax-normaliser kernels and the generic
// beam kernel (any vocabulary width, beam widths up to 1024, float32 and float64 scores, scorer table).
#define CTCX_WITH_NORM
#define CTCX_WITH_GENERIC
#include "ctcx_kernels.cuh"
#include "ctcx_launch.h"

#include <algorithm>

namespace ctcx {

namespace {
struct Tier {
  int wmax, nt;
};
Tier PickTier(int W) {
  if (W <= 32) return {32, 128};
  if (W <= 128) return {128, 256};
  if (W <= 256) return {256, 256};
  return {1024, 1024};
}

template <typename R, int WMAX, int NT>
LaunchStatus LaunchOne(const BeamParamsT<R>& p, size_t smem, cudaStream_t stream) {
  auto kern = BeamKernelT<R, WMAX, NT>;
  cudaError_t e = cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
  if (e != cudaSuccess) return LaunchFrom(e, "cudaFuncSetAttribute(BeamKernelT)");
  kern<<<p.B, NT, smem, stream>>>(p);
  return LaunchFrom(cudaGetLastError(), "BeamKernelT launch");
}

// Exact upcast of (possibly strided) half-precision logits to dense float32.
template <typename H>
__global__ void UpcastKernel(const H* __restrict__ in, float* __restrict__ out, long long rows, int C, int B,
                             long long tstride) {
  const long long n = rows * C;
  for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (long long)gridDim.x * blockDim.x) {
    const long long row = i / C;
    const int c = (int)(i - row * C);
    out[i] = LoadLogit<H>(in, (size_t)(RowOffset(row, B, C, tstride) + c));
  }
}
}  // namespace

// kernel 1: softmax normalisers of `rows` = T * B logit rows
LaunchStatus LaunchLogNorm(const float* logits, float* off, long long rows, int C, int B, long long tstride,
                           cudaStream_t stream) {
  const int sm_count = SmCount();
  if (C <= 64) {  // thread per row, rows staged through shared memory
    long long blocks = (rows + kLogNormRows - 1) / kLogNormRows;
    if (blocks > (long long)sm_count * 8) blocks = (long long)sm_count * 8;
    const size_t lsm = (size_t)kLogNormRows * (C | 1) * sizeof(float);
    cudaError_t e = cudaFuncSetAttribute(LogNormRowKernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)lsm);
    if (e != cudaSuccess) return LaunchFrom(e, "cudaFuncSetAttribute(LogNormRowKernel)");
    LogNormRowKernel<<<(unsigned)blocks, kLogNormRows, lsm, stream>>>(logits, off, rows, C, B, tstride);
  } else {  // warp per row
    long long blocks = (rows + 7) / 8;
    if (blocks > (long long)sm_count * 16) blocks = (long long)sm_count * 16;
    LogNormKernel<<<(unsigned)blocks, 256, 0, stream>>>(logits, off, rows, C, B, tstride);
  }
  return LaunchFrom(cudaGetLastError(), "LogNorm kernel launch");
}

LaunchStatus LaunchLogNorm(const double* logits, double* off, long long rows, int C, int B, long long tstride,
                           cudaStream_t stream) {
  long long blocks = (rows + 7) / 8;
  if (blocks > (long long)SmCount() * 16) blocks = (long long)SmCount() * 16;
  LogNormKernelF64<<<(unsigned)blocks, 256, 0, stream>>>(logits, off, rows, C, B, tstride);
  return LaunchFrom(cudaGetLastError(), "LogNormKernelF64 launch");
}

LaunchStatus LaunchUpcast(const void* in, int in_dtype, float* out, int T, int B, int C, long long tstride,
                          cudaStream_t stream) {
  const long long rows = (long long)T * B, n = rows * C;
  if (n <= 0) return LaunchOk();
  const unsigned blocks = (unsigned)std::min<long long>((n + 255) / 256, (long long)SmCount() * 32);
  if (in_dtype == kInF16)
    UpcastKernel<__half><<<blocks, 256, 0, stream>>>((const __half*)in, out, rows, C, B, tstride);
  else if (in_dtype == kInBF16)
    UpcastKernel<__nv_bfloat16><<<blocks, 256, 0, stream>>>((const __nv_bfloat16*)in, out, rows, C, B, tstride);
  else
    return {kLaunchUnsupported, cudaSuccess, ""};
  return LaunchFrom(cudaGetLastError(), "UpcastKernel launch");
}

// kernel 2, generic form
template <typename R>
LaunchStatus LaunchBeamGeneric(BeamParamsT<R>& bp, cudaStream_t stream) {
  constexpr bool kF64 = (sizeof(R) == 8);
  const int W = bp.W, C = bp.C;
  bp.kid_words = (C + 31) / 32;
  const long long full_list = (long long)W * C;
  bp.cand_cap = (full_list <= kListCapMax) ? (int)full_list : 0;
  // double state is twice as wide: the largest tier that fits in shared memory holds 512 slots
  Tier tier = PickTier(W);
  if (kF64 && tier.wmax > 256) tier = (W <= 512) ? Tier{512, 512} : Tier{1024, 1024};
  BeamSmem lay;
  lay.Init(tier.wmax, tier.nt, C, bp.kid_words, bp.cand_cap, (int)sizeof(R), W);
  // (double: beam_width > 512, or a very wide vocabulary)
  if (lay.bytes > 220 * 1024) return {kLaunchUnsupported, cudaSuccess, ""};
  switch (tier.wmax) {
    case 32: return LaunchOne<R, 32, 128>(bp, lay.bytes, stream);
    case 128: return LaunchOne<R, 128, 256>(bp, lay.bytes, stream);
    case 256: return LaunchOne<R, 256, 256>(bp, lay.bytes, stream);
  }
  if constexpr (kF64) {
    if (tier.wmax == 512) return LaunchOne<double, 512, 512>(bp, lay.bytes, stream);
    return {kLaunchUnsupported, cudaSuccess, ""};
  } else {
    return LaunchOne<float, 1024, 1024>(bp, lay.bytes, stream);
  }
}
template LaunchStatus LaunchBeamGeneric<float>(BeamParamsT<float>& bp, cudaStream_t stream);
template LaunchStatus LaunchBeamGeneric<double>(BeamParamsT<double>& bp, cudaStream_t stream);

}  // namespace ctcx
