// Translation unit of the narrow-vocabulary fast beam kernel (ctcx_beam_v4.cuh).
#include "ctcx_beam_v4.cuh"
#include "ctcx_launch.h"

namespace ctcx {

int SmCount() {
  static int cached[64] = {0};
  int dev = 0, sms = 148;
  cudaGetDevice(&dev);
  if (dev >= 0 && dev < 64 && cached[dev] > 0) return cached[dev];
  cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev);
  if (dev >= 0 && dev < 64) cached[dev] = sms;
  return sms;
}

namespace {
// Launch configuration of one kernel instantiation on one device, computed once: the attribute and
// occupancy queries cost tens of microseconds of host time that would otherwise sit between the
// kernels of every decode. (A cache of immutable facts about the device, not decoder state.)
struct LaunchCfg {
  size_t smem = 0;   // dynamic shared memory the attribute was raised to
  int resident = 0;  // CTAs the device keeps resident at that size
};
constexpr int kMaxDevices = 64;
constexpr int kMinSliceFrames = 32;  // shorter slices would not amortise the hand-over

template <typename IN, int WMAX, bool TIMING, int MINB, bool LM = false>
LaunchStatus LaunchOne(BeamParamsT<typename ScoreOf<IN>::type>& p, size_t smem, cudaStream_t stream) {
  auto kern = BeamKernelV4<IN, WMAX, 256, TIMING, MINB, LM>;
  static LaunchCfg cfgs[kMaxDevices];
  int dev = 0;
  cudaGetDevice(&dev);
  LaunchCfg local;
  LaunchCfg& cfg = (dev >= 0 && dev < kMaxDevices) ? cfgs[dev] : local;
  if (cfg.resident == 0 || cfg.smem != smem) {
    cudaError_t e = cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
    if (e != cudaSuccess) return LaunchFrom(e, "cudaFuncSetAttribute(BeamKernelV4)");
    // persistent CTAs: as many as the device keeps resident, each pulls utterances from p.queue
    int per_sm = 1, sms = 148;
    cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev);
    e = cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, kern, 256, smem);
    if (e != cudaSuccess) return LaunchFrom(e, "cudaOccupancyMaxActiveBlocksPerMultiprocessor(BeamKernelV4)");
    cfg.smem = smem;
    cfg.resident = sms * (per_sm > 0 ? per_sm : 1);
  }
  const long long resident = cfg.resident;
  const unsigned grid = (unsigned)(p.B < resident ? p.B : resident);
  // Batches beyond the resident CTAs: cut every utterance into time slices so that the queue keeps all
  // CTAs busy to the end (the beam travels between slices through the state block in HBM, ~4 KB).
  p.n_slices = 1;
  p.slice_frames = p.T > 0 ? p.T : 1;
  if (p.B > resident && p.t_done == nullptr && p.state != nullptr && p.progress != nullptr && p.T >= 2 * kMinSliceFrames) {
    // enough tasks that the last round of the queue is a small part of the whole: ~12 per CTA
    long long want = (12 * resident + p.B - 1) / p.B;
    want = want < 2 ? 2 : (want > 16 ? 16 : want);
    const long long most = p.T / kMinSliceFrames;
    p.n_slices = (int)(want < most ? want : most);
    p.slice_frames = (p.T + p.n_slices - 1) / p.n_slices;
  }
  kern<<<grid, 256, smem, stream>>>(p);
  return LaunchFrom(cudaGetLastError(), "BeamKernelV4 launch");
}

template <typename IN>
LaunchStatus LaunchTyped(BeamParams& p, int wmax, size_t smem, cudaStream_t stream) {
  if constexpr (sizeof(IN) == 4) {
    if (p.lm != nullptr && p.dbg_cycles != nullptr && wmax == 128) return LaunchOne<IN, 128, true, 1, true>(p, smem, stream);
    if (p.lm != nullptr) {  // scorer table plugged in: float32 inputs only
      const bool latency = p.B <= 2 * SmCount();
      switch (wmax) {
        case 32: return latency ? LaunchOne<IN, 32, false, 2, true>(p, smem, stream) : LaunchOne<IN, 32, false, 4, true>(p, smem, stream);
        case 128: return latency ? LaunchOne<IN, 128, false, 2, true>(p, smem, stream) : LaunchOne<IN, 128, false, 4, true>(p, smem, stream);
        default: return latency ? LaunchOne<IN, 256, false, 2, true>(p, smem, stream) : LaunchOne<IN, 256, false, 4, true>(p, smem, stream);
      }
    }
    if (p.dbg_cycles != nullptr) {  // timing build: float32 inputs only
      switch (wmax) {
        case 32: return LaunchOne<IN, 32, true, 1>(p, smem, stream);
        case 128: return LaunchOne<IN, 128, true, 1>(p, smem, stream);
        default: return LaunchOne<IN, 256, true, 1>(p, smem, stream);
      }
    }
  }
  if (p.B <= 2 * SmCount()) {  // latency regime: at most two utterances per SM, 128 registers per thread
    switch (wmax) {
      case 32: return LaunchOne<IN, 32, false, 2>(p, smem, stream);
      case 128: return LaunchOne<IN, 128, false, 2>(p, smem, stream);
      default: return LaunchOne<IN, 256, false, 2>(p, smem, stream);
    }
  }
  switch (wmax) {
    case 32: return LaunchOne<IN, 32, false, 4>(p, smem, stream);
    case 128: return LaunchOne<IN, 128, false, 4>(p, smem, stream);
    default: return LaunchOne<IN, 256, false, 4>(p, smem, stream);
  }
}

size_t SmemBytes(int wmax, int cand_cap, bool lm, bool f64 = false) {  // (the scorer table adds a constant)
  const size_t extra = lm ? (BeamSmemV4<32, true>::list - BeamSmemV4<32, false>::list) : 0;
  if (f64) {
    switch (wmax) {
      case 32: return BeamSmemV4<32, false, 8>::Bytes(cand_cap);
      case 128: return BeamSmemV4<128, false, 8>::Bytes(cand_cap);
      default: return BeamSmemV4<256, false, 8>::Bytes(cand_cap);
    }
  }
  switch (wmax) {
    case 32: return BeamSmemV4<32>::Bytes(cand_cap) + extra;
    case 128: return BeamSmemV4<128>::Bytes(cand_cap) + extra;
    default: return BeamSmemV4<256>::Bytes(cand_cap) + extra;
  }
}

// the preconditions both score types share, and the fields they derive; false = not this kernel's
template <typename R>
bool PrepareNarrow(BeamParamsT<R>& p) {
  if (!NarrowFastShape(p.W, p.C) || p.queue == nullptr || p.bp32 == nullptr) return false;
  p.cand_cap = p.W * p.C;
  p.kid_words = 1;
  return true;
}
}  // namespace

bool NarrowFastShape(int W, int C) {
  if (C > 32 || W > 256 || (long long)W * C > kListCapMax) return false;
  return SmemBytes(TierOf(W), W * C, true) <= 220 * 1024 && SmemBytes(TierOf(W), W * C, false, true) <= 220 * 1024;
}

LaunchStatus LaunchBeamNarrow(BeamParams& p, int in_dtype, cudaStream_t stream) {
  if (!PrepareNarrow(p) || (p.lm != nullptr && in_dtype != kInF32)) return {kLaunchUnsupported, cudaSuccess, ""};
  const int wmax = TierOf(p.W);
  const size_t smem = SmemBytes(wmax, p.cand_cap, p.lm != nullptr);
  switch (in_dtype) {
    case kInF32: return LaunchTyped<float>(p, wmax, smem, stream);
    case kInF16: return LaunchTyped<__half>(p, wmax, smem, stream);
    case kInBF16: return LaunchTyped<__nv_bfloat16>(p, wmax, smem, stream);
    default: return {kLaunchUnsupported, cudaSuccess, ""};
  }
}

// float64 logits (the op's T = double registration): the same kernel computing in double, 64-bit keys
LaunchStatus LaunchBeamNarrow(BeamParamsT<double>& p, cudaStream_t stream) {
  if (!PrepareNarrow(p) || p.lm != nullptr) return {kLaunchUnsupported, cudaSuccess, ""};
  // one-shot decodes take whole utterances from the queue (no time slices); a streamed step
  // (t_done set) carries the beam in the double blocks of the state
  if (p.t_done == nullptr) p.state = nullptr;
  const int wmax = TierOf(p.W);
  const size_t smem = SmemBytes(wmax, p.cand_cap, false, true);
  // (~90 KB of shared memory at beam 100: two CTAs per SM in either regime, 128 registers)
  switch (wmax) {
    case 32: return LaunchOne<double, 32, false, 2>(p, smem, stream);
    case 128: return LaunchOne<double, 128, false, 2>(p, smem, stream);
    default: return LaunchOne<double, 256, false, 2>(p, smem, stream);
  }
}

}  // namespace ctcx
