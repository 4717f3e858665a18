// Host-side launch interface of the kernel translation units (k_narrow.cu, k_wide.cu, k_generic.cu,
// k_post.cu). ctcx_api.cu -- validation, workspace carve-up, stream choreography -- sees the kernels
// only through these functions, so each family of kernels compiles in its own translation unit.
#pragma once
#include <cuda_runtime.h>

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
int SmCount();  // multiprocessors of the current device (cached per device)

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
// flags into `stats` (see FlagsKernel in k_post.cu)
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
LaunchStatus LaunchStreamReset(unsigned char* state, int B, int W, int score_bytes, cudaStream_t stream);
LaunchStatus LaunchStreamCheck(unsigned char* state, int B, int W, const int* table_flag, int* stats,
                               cudaStream_t stream);
// out[b] = frames of utterance b inside the time chunk [t0, t0 + len) (lengths clamped to [0, T])
LaunchStatus LaunchChunkLen(const int* seq_len, int B, int T, int t0, int len, int* out, cudaStream_t stream);
LaunchStatus LaunchMathTest(int op, const float* x, float* y, int n, cudaStream_t stream);
LaunchStatus LaunchMathTest(int op, const double* x, double* y, int n, cudaStream_t stream);

}  // namespace ctcx
