// Translation unit of the kernels after the beam search: trace-back of the top paths, prefix sums of
// the sparse sizes, reduction of the per-utterance flags, sparse packing; plus the math test hooks.
#define CTCX_WITH_POST
#include "ctcx_kernels.cuh"
#include "ctcx_launch.h"

#include <algorithm>
#include <cstdint>

namespace ctcx {

namespace {
// Reduces the per-utterance flags to stats[0..5] = {OR of anomaly bits, first b with too few leaves (or
// B), first b with sequence_length > T (or B), first b with negative sequence_length (or B), first b fed
// more frames than a stream holds (or B), first b whose input frames never arrived (or B)}.
__global__ void FlagsKernel(const int* flags, const int* seq_len, int B, int T, int* out) {
  for (int b = blockIdx.x * blockDim.x + threadIdx.x; b < B; b += gridDim.x * blockDim.x) {
    const int f = flags ? flags[b] : 0;
    if (f & 1) atomicOr(&out[0], 1);
    if (f & 2) atomicMin(&out[1], b);
    if (seq_len[b] > T) atomicMin(&out[2], b);
    if (seq_len[b] < 0) atomicMin(&out[3], b);
    if (f & 4) atomicMin(&out[4], b);
    if (f & 8) atomicMin(&out[5], b);
  }
}

// flag = 1 if any entry is positive or NaN (scorer tables hold log-probabilities)
__global__ void PositiveKernel(const float* v, long long n, int* flag) {
  for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (long long)gridDim.x * blockDim.x)
    if (!(v[i] <= 0.0f)) *flag = 1;
}

// Every float block holds the root (what a float kernel resumes if a float64 step advanced the frame
// count: a valid beam, never foreign bytes), marked "no float step yet" and tagged with the stream's
// score type; the double blocks of a float64 stream are marked unwritten.
__global__ void StreamResetKernel(unsigned char* state, int B, int W, int score_bytes) {
  for (int b = blockIdx.x * blockDim.x + threadIdx.x; b < B; b += gridDim.x * blockDim.x) {
    const StreamView fv(state + (size_t)b * StreamStateBytes(W), W);
    fv.hdr->n = 1;
    fv.hdr->gap = 0u;
    fv.hdr->flags = kStreamNoF32Step;
    fv.hdr->type = score_bytes;
    fv.total[0] = 0.0f; fv.blk[0] = 0.0f; fv.lab[0] = NegInf(); fv.ab[0] = 0.0f; fv.an[0] = NegInf();
    fv.label[0] = -1; fv.hash[0] = kRootHash; fv.phash[0] = 0ull;
    if (score_bytes == 8) {
      const StreamViewT<double> dv = StreamBlock64(state, B, W, b);
      dv.hdr->n = 0;
      dv.hdr->type = 0;
    }
  }
}

// A float64 step on a float stream marks the float header's type; a float step on a float64 stream drops
// the "no float step yet" flag (float kernels rewrite the flags of every block they step).
__global__ void StreamCheckKernel(const unsigned char* state, int B, int W, const int* table_flag, int* stats) {
  for (int b = blockIdx.x * blockDim.x + threadIdx.x; b < B; b += gridDim.x * blockDim.x) {
    const StreamHdr* h = reinterpret_cast<const StreamHdr*>(state + (size_t)b * StreamStateBytes(W));
    const bool mixed = (h->type & kStreamF64Stepped) || (h->type == 8 && !(h->flags & kStreamNoF32Step));
    if (mixed || (b == 0 && *table_flag != 0)) atomicMin(&stats[3], 0);
  }
}

// frames of utterance b inside the time chunk [t0, t0 + len) of a decode that is run chunk by chunk
__global__ void ChunkLenKernel(const int* seq_len, int B, int T, int t0, int len, int* out) {
  const int b = blockIdx.x * blockDim.x + threadIdx.x;
  if (b < B) out[b] = min(max(min(max(seq_len[b], 0), T) - t0, 0), len);
}

template <typename REC>
LaunchStatus LaunchTrace(const TraceParams& tp, cudaStream_t stream) {
  const int W = tp.W;
  const long long walks = (long long)tp.B * tp.P;
  if (walks >= 4096) {
    // thousands of independent walks hide the latency of the dependent loads by themselves, and
    // touch one record per frame instead of whole rows
    TraceKernel<REC><<<(unsigned)((walks + 127) / 128), 128, 0, stream>>>(tp);
  } else {
    // one warp per (utterance, path); two blocks of 2^rows_log2 back-pointer rows per warp in
    // shared memory (about 26 KB per block)
    constexpr int kTraceWarps = 2;
    int rows_log2 = 5;
    while (rows_log2 > 0 && ((size_t)W << rows_log2) * sizeof(REC) > 26 * 1024) --rows_log2;
    const size_t tsm = (size_t)kTraceWarps * 2 * ((size_t)W << rows_log2) * sizeof(REC);
    auto tk = TraceWarpKernel<REC, kTraceWarps>;
    cudaError_t e = cudaFuncSetAttribute(tk, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)tsm);
    if (e != cudaSuccess) return LaunchFrom(e, "cudaFuncSetAttribute(TraceWarpKernel)");
    // a row of records that is a multiple of 16 bytes makes every block of rows one aligned span: bulk copies
    const int use_bulk = (((size_t)W * sizeof(REC)) % 16 == 0 && (reinterpret_cast<uintptr_t>(tp.bp) & 15u) == 0) ? 1 : 0;
    tk<<<(unsigned)((walks + kTraceWarps - 1) / kTraceWarps), kTraceWarps * 32, tsm, stream>>>(tp, rows_log2, use_bulk);
  }
  return LaunchFrom(cudaGetLastError(), "trace kernel launch");
}
}  // namespace

LaunchStatus LaunchTraceScanFlags(const TraceParams& tp, int rec_bytes, const ScanParams& sp, const int* flags,
                                  int* stats, cudaStream_t stream, cudaEvent_t after_trace) {
  LaunchStatus st = (rec_bytes == 4) ? LaunchTrace<unsigned>(tp, stream) : LaunchTrace<uint2>(tp, stream);
  if (st.code != kLaunchOk) return st;
  if (after_trace != nullptr) cudaEventRecord(after_trace, stream);
  ScanKernel<<<tp.P, 1024, 0, stream>>>(sp);
  cudaError_t e = cudaGetLastError();
  if (e != cudaSuccess) return LaunchFrom(e, "ScanKernel launch");
  FlagsKernel<<<(tp.B + 255) / 256, 256, 0, stream>>>(flags, tp.seq_len, tp.B, tp.T, stats);
  return LaunchFrom(cudaGetLastError(), "FlagsKernel launch");
}

LaunchStatus LaunchFlagsOnly(const int* seq_len, int B, int T, int* stats, cudaStream_t stream) {
  FlagsKernel<<<(B + 255) / 256, 256, 0, stream>>>(nullptr, seq_len, B, T, stats);
  return LaunchFrom(cudaGetLastError(), "FlagsKernel launch");
}

LaunchStatus LaunchPack(const PackParams& pp, cudaStream_t stream) {
  dim3 grid((unsigned)pp.B, (unsigned)pp.P);
  PackKernel<<<grid, 128, 0, stream>>>(pp);
  return LaunchFrom(cudaGetLastError(), "PackKernel launch");
}

LaunchStatus LaunchPackTable(const long long* sizes, int B, int P, int real_bytes, long long* buf,
                             unsigned long long buf_elems, long long** ptrs, int* overflow, cudaStream_t stream) {
  PackTableKernel<<<1, 32, 0, stream>>>(sizes, B, P, real_bytes, buf, buf_elems, ptrs, overflow);
  return LaunchFrom(cudaGetLastError(), "PackTableKernel launch");
}

LaunchStatus LaunchChunkLen(const int* seq_len, int B, int T, int t0, int len, int* out, cudaStream_t stream) {
  ChunkLenKernel<<<(unsigned)((B + 255) / 256), 256, 0, stream>>>(seq_len, B, T, t0, len, out);
  return LaunchFrom(cudaGetLastError(), "ChunkLenKernel launch");
}

LaunchStatus LaunchPositive(const float* v, long long n, int* flag, cudaStream_t stream) {
  PositiveKernel<<<(unsigned)std::min<long long>((n + 255) / 256, 1024), 256, 0, stream>>>(v, n, flag);
  return LaunchFrom(cudaGetLastError(), "PositiveKernel launch");
}

LaunchStatus LaunchStreamReset(unsigned char* state, int B, int W, int score_bytes, cudaStream_t stream) {
  StreamResetKernel<<<(unsigned)((B + 127) / 128), 128, 0, stream>>>(state, B, W, score_bytes);
  return LaunchFrom(cudaGetLastError(), "StreamResetKernel launch");
}

LaunchStatus LaunchStreamCheck(unsigned char* state, int B, int W, const int* table_flag, int* stats,
                               cudaStream_t stream) {
  StreamCheckKernel<<<(unsigned)((B + 127) / 128), 128, 0, stream>>>(state, B, W, table_flag, stats);
  return LaunchFrom(cudaGetLastError(), "StreamCheckKernel launch");
}

LaunchStatus LaunchMathTest(int op, const float* x, float* y, int n, cudaStream_t stream) {
  MathTestKernel<<<(n + 255) / 256, 256, 0, stream>>>(op, x, y, n);
  return LaunchFrom(cudaGetLastError(), "MathTestKernel launch");
}

LaunchStatus LaunchMathTest(int op, const double* x, double* y, int n, cudaStream_t stream) {
  MathTestKernelF64<<<(n + 255) / 256, 256, 0, stream>>>(op, x, y, n);
  return LaunchFrom(cudaGetLastError(), "MathTestKernelF64 launch");
}

}  // namespace ctcx
