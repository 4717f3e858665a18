// Host-side launch interface of the kernel translation units, each of which holds one family of
// kernels and their launchers: k_narrow.cu (BeamKernelV4), k_wide.cu (NormTopClassesKernel,
// BeamKernelWide), k_generic.cu (the LogNorm normalisers, BeamKernelT) and k_post.cu (trace-back, scan,
// pack). ctcx_api.cu -- validation, workspace carve-up, stream choreography -- sees the kernels only
// through these functions.
#pragma once
#include <cuda_runtime.h>

#include <atomic>

#include "ctcx_params.h"

namespace ctcx {

enum InDtype { kInF32 = 0, kInF16 = 1, kInBF16 = 2 };

// Launch results (a subset of the CTCX_* codes of include/ctcx.h, repeated here to keep this header
// independent of the public one).
enum { kLaunchOk = 0, kLaunchUnsupported = 9, kLaunchCuda = 11 };

struct LaunchStatus {
  int code;           // kLaunchOk / kLaunchUnsupported / kLaunchCuda
  cudaError_t cuda;   // the failing CUDA call's error when code == kLaunchCuda
  const char* what;
};
inline LaunchStatus LaunchOk() { return {kLaunchOk, cudaSuccess, ""}; }
inline LaunchStatus LaunchFrom(cudaError_t e, const char* what) {
  if (e == cudaSuccess) return LaunchOk();
  return {kLaunchCuda, e, what};
}

// ---- shape predicates: pure functions of the shape (the workspace layout depends on them) ----
// narrow fast kernel (ctcx_beam_v4.cuh): num_classes <= 32, beam_width <= 256, beam_width * num_classes
// candidates fit in shared memory
bool NarrowFastShape(int W, int C);
// wide fast kernel (ctcx_beam_wide.cuh): 32 < num_classes <= 2048, beam_width <= 256, and the worst
// frame's candidate list fits in shared memory
bool WideFastShape(int W, int C);
int WideKc(int W, int C);  // sorted classes per frame the beam kernel uses
int WideKe(int W, int C);  // ... plus the sentinel
int WideKs(int W, int C);  // row stride of the sorted arrays
// 4-byte back-pointer records when every slot and label fits in a byte
inline int RecBytes(int W, int C) { return (W <= 256 && C <= 256) ? 4 : 8; }

// ---- shared by the launchers ----
constexpr int kListCapMax = 4608;  // candidate-list entries kept in shared memory (8 B each)
// beam tier (slots per CTA) of the fast kernels' instantiations
inline int TierOf(int W) { return (W <= 32) ? 32 : (W <= 128) ? 128 : 256; }

// Facts about a device are cached for the first kMaxDevices device ordinals (queried anew on others).
// The attribute and occupancy queries cost tens of microseconds of host time that would otherwise sit
// between the kernels of every decode. Every cached fact is one atomic word, so concurrent callers
// never see a half-written entry; callers racing on a first query store the same value.
constexpr int kMaxDevices = 64;

// multiprocessors of the current device
inline int SmCount() {
  static std::atomic<int> cached[kMaxDevices];
  int dev = 0;
  cudaGetDevice(&dev);
  const bool keep = dev >= 0 && dev < kMaxDevices;
  int sms = keep ? cached[dev].load(std::memory_order_relaxed) : 0;
  if (sms > 0) return sms;
  sms = 148;
  cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev);
  if (keep) cached[dev].store(sms, std::memory_order_relaxed);
  return sms;
}

// Launch set-up of one kernel instantiation; its launcher keeps one as a function-local static.
class KernelSetup {
 public:
  // Raises the kernel's dynamic shared-memory limit to `max_smem`, once per device: the most that any
  // shape reaching the instantiation requests. The limit belongs to the function and the whole
  // process, so it is never set lower, and no launch depends on what another host thread set.
  cudaError_t RaiseSmemLimit(const void* kern, size_t max_smem) {
    int dev = 0;
    cudaGetDevice(&dev);
    const bool keep = dev >= 0 && dev < kMaxDevices;
    if (keep && raised_[dev].load(std::memory_order_acquire)) return cudaSuccess;
    const cudaError_t e = cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)max_smem);
    if (e == cudaSuccess && keep) raised_[dev].store(true, std::memory_order_release);
    return e;
  }
  // CTAs of the kernel (`threads` each, `smem` bytes of dynamic shared memory) that the current device
  // keeps resident, remembered for the last `smem` asked about
  cudaError_t Resident(const void* kern, int threads, size_t smem, long long* ctas) {
    int dev = 0;
    cudaGetDevice(&dev);
    const bool keep = dev >= 0 && dev < kMaxDevices;
    const unsigned long long seen = keep ? resident_[dev].load(std::memory_order_relaxed) : 0ull;
    if (seen != 0ull && (seen >> 32) == smem) {
      *ctas = (long long)(seen & 0xffffffffull);
      return cudaSuccess;
    }
    int per_sm = 1;
    const cudaError_t e = cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, kern, threads, smem);
    if (e != cudaSuccess) return e;
    *ctas = (long long)SmCount() * (per_sm > 0 ? per_sm : 1);
    if (keep) resident_[dev].store((unsigned long long)smem << 32 | (unsigned long long)*ctas, std::memory_order_relaxed);
    return cudaSuccess;
  }

 private:
  std::atomic<bool> raised_[kMaxDevices] = {};
  std::atomic<unsigned long long> resident_[kMaxDevices] = {};  // smem << 32 | CTAs, 0 = not known yet
};

// ---- kernel 1 ----
LaunchStatus LaunchLogNorm(const float* logits, float* off, long long rows, int C, int B, long long tstride,
                           cudaStream_t stream);
LaunchStatus LaunchLogNorm(const double* logits, double* off, long long rows, int C, int B, long long tstride,
                           cudaStream_t stream);
LaunchStatus LaunchNormTopClasses(const void* logits, int in_dtype, float* off, long long rows, int C, int blank,
                                  int W, float* srt_pl, unsigned short* srt_cls, int B, long long tstride,
                                  cudaStream_t stream);
// exact upcast of a (possibly strided) half-precision [T,B,C] tensor into a dense float32 one
LaunchStatus LaunchUpcast(const void* in, int in_dtype, float* out, int T, int B, int C, long long tstride,
                          cudaStream_t stream);

// ---- kernel 2 ----
LaunchStatus LaunchBeamNarrow(BeamParams& p, int in_dtype, cudaStream_t stream);
LaunchStatus LaunchBeamNarrow(BeamParamsT<double>& p, cudaStream_t stream);  // float64 logits, double scores
LaunchStatus LaunchBeamWide(BeamParams& p, int in_dtype, cudaStream_t stream);
template <typename R>  // float or double scores
LaunchStatus LaunchBeamGeneric(BeamParamsT<R>& p, cudaStream_t stream);

// ---- kernels 3-5 ----
// trace-back of the top paths, then per-path offsets / sizes and the reduction of the per-utterance
// flags into `stats` (see FlagsKernel in k_post.cu); with tp.mask set, over the selected utterances only
LaunchStatus LaunchTraceScanFlags(const TraceParams& tp, int rec_bytes, const ScanParams& sp, const int* flags,
                                  int* stats, cudaStream_t stream, cudaEvent_t after_trace);
LaunchStatus LaunchFlagsOnly(const int* seq_len, int B, int T, int* stats, cudaStream_t stream);
LaunchStatus LaunchPack(const PackParams& pp, cudaStream_t stream);
// pointer table of the compact one-buffer output layout, from the sizes on the device (PackTableKernel)
LaunchStatus LaunchPackTable(const long long* sizes, int B, int P, int real_bytes, long long* buf,
                             unsigned long long buf_elems, long long** ptrs, int* overflow, cudaStream_t stream);
LaunchStatus LaunchPositive(const float* v, long long n, int* flag, cudaStream_t stream);
// streamed decodes (StreamHdrT): the state blocks of a reset stream with score_bytes (4 or 8) scores, and
// the check before TopPaths -- stats[3] = 0 (a bad argument) if *table_flag is set or score types were mixed
// (mask: optional [B], non-zero = utterance checked; null = all)
LaunchStatus LaunchStreamReset(unsigned char* state, int B, int W, int score_bytes, cudaStream_t stream);
// the reset of the utterances selected by p.mask only, entirely on the device
LaunchStatus LaunchStreamResetSlots(const StreamSlotsParams& p, cudaStream_t stream);
LaunchStatus LaunchStreamCheck(unsigned char* state, int B, int W, const int* table_flag, int* stats,
                               const int* mask, cudaStream_t stream);
// out[b] = frames of utterance b inside the time chunk [t0, t0 + len) (lengths clamped to [0, T])
LaunchStatus LaunchChunkLen(const int* seq_len, int B, int T, int t0, int len, int* out, cudaStream_t stream);
LaunchStatus LaunchMathTest(int op, const float* x, float* y, int n, cudaStream_t stream);
LaunchStatus LaunchMathTest(int op, const double* x, double* y, int n, cudaStream_t stream);

}  // namespace ctcx
