// Translation unit of the generic path: the stand-alone softmax-normaliser kernels and the generic
// beam kernel (ctcx_beam_generic.cuh).
#include "ctcx_beam_generic.cuh"
#include "ctcx_launch.h"

#include <algorithm>

namespace ctcx {

// ---------------------------------------------------------------------------------------------
// Kernel 1: per-row softmax normaliser off[t,b] = max_j x_j + logf(sum_{j in index order} expf(x_j - max))
// (decoder.h:71-80). One warp per row; lanes evaluate expf in parallel into a per-warp shared-memory
// chunk, then every lane accumulates the chunk in index order (the reference's order, so the float
// sum is bit-identical) with 16-byte broadcast loads -- 4x fewer issue slots than passing the terms
// around with shuffles, which is what bounded the first version of this kernel.
// ---------------------------------------------------------------------------------------------
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

namespace {
constexpr size_t kGenericSmemMax = 220 * 1024;  // the most LaunchBeamGeneric admits

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
  static KernelSetup setup;
  const cudaError_t e = setup.RaiseSmemLimit((const void*)kern, kGenericSmemMax);
  if (e != cudaSuccess) return LaunchFrom(e, "shared-memory limit of BeamKernelT");
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
  constexpr int kRowMaxC = 64;
  if (C <= kRowMaxC) {  // thread per row, rows staged through shared memory
    long long blocks = (rows + kLogNormRows - 1) / kLogNormRows;
    if (blocks > (long long)sm_count * 8) blocks = (long long)sm_count * 8;
    const size_t lsm = (size_t)kLogNormRows * (C | 1) * sizeof(float);
    static KernelSetup setup;
    const cudaError_t e =
        setup.RaiseSmemLimit((const void*)LogNormRowKernel, (size_t)kLogNormRows * (kRowMaxC | 1) * sizeof(float));
    if (e != cudaSuccess) return LaunchFrom(e, "shared-memory limit of LogNormRowKernel");
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
  if (lay.bytes > kGenericSmemMax) return {kLaunchUnsupported, cudaSuccess, ""};
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
