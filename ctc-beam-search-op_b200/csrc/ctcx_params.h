// Parameter blocks of the kernels (plain structs shared by the host-side launch code in ctcx_api.cu
// and the kernel translation units).
#pragma once
#include <cuda_runtime.h>

#include <cstddef>
#include <cstdint>

namespace ctcx {

template <typename R>
struct BeamParamsT {
  const R* logits;  // [T,B,C] time-major raw logits
  const R* off;     // [T,B]   normaliser from LogNormKernel
  const int* seq_len;   // [B]
  int T, B, C, W, P;
  int blank_index;
  int cand_cap;   // capacity of the shared-memory candidate list; 0 = streaming mode
  int kid_words;  // ceil(C/32)
  uint2* bp;      // [B,T,W] back-pointer records {packed, label}
  R* fin_total;      // [B,P]
  int* fin_kind;     // [B,P] 1 = best alignment ends in blank
  int* fin_n;        // [B]   members in the final beam
  int* flags;        // [B]   bit0 rounding anomaly, bit1 fewer leaves than top_paths
  R* dbg_totals;      // optional [B,T,W]
  int* dbg_n;         // optional [B,T]
  long long* dbg_cycles;  // optional [B,24]: clock64 cycles per phase (thread 0), summed over frames
  // streaming (Step / TopPaths / Reset, decoder.h:39-53); all null / T for a one-shot decode
  int Tcap;               // frames per utterance the back-pointer array can hold (its row stride)
  int* t_done;            // [B] frames already consumed per utterance (updated by the kernel), or null
  unsigned char* state;   // [B] x StreamStateBytes(W): beam state carried between chunks, or null
  // wide-vocabulary fast path (ctcx_beam_wide.cuh): per frame, the classes sorted by log-prob
  const R* srt_pl;               // [T,B,Cs] x_l - off of the best classes, descending (padding = -inf)
  const unsigned short* srt_cls; // [T,B,Cs] class index at each sorted position
  int Cs;                        // row stride of the two arrays (a multiple of 8)
  int Kc;                        // sorted classes per frame the kernel may use (entry Kc, if < C-1
                                 // classes are listed, is a sentinel: the best class left out)
  // scorer extension point (util/ctc_beam_scorer.h:31-65), generic kernel and the narrow kernel's LM variant: null = the default
  // scorer; otherwise a [C+1, C] table of expansion scores (<= 0), row = label of the expanded
  // entry + 1 (row 0: the root), column = new label: GetStateExpansionScore(state, s) = s + entry
  const R* lm;
  // input layout: row (t, b) of `logits` starts at element t * tstride + b * C (tstride = B * C for a
  // contiguous tensor; larger when the batch is a shard [:, b0:b1, :] of a wider tensor, decoded in place)
  long long tstride;
  // fast narrow kernel (ctcx_beam_v4.cuh) only:
  const int* ready;    // device word: number of leading frames of `logits` that have landed (an H2D copy
                       // in time slabs may still be in flight); null = everything is there
  int* queue;          // device word, zero at launch: next utterance for the persistent CTAs
  unsigned* bp32;      // [B,Tcap,W] 4-byte back-pointer records (instead of `bp`)
  // time slicing of the narrow kernel's work queue (set by its launcher): an utterance is cut into
  // n_slices tasks of slice_frames frames; progress[b] = slices of utterance b finished so far
  int n_slices, slice_frames;
  int* progress;       // [B] device words, zero at launch (needed when n_slices > 1)
};
using BeamParams = BeamParamsT<float>;

// Beam state of one utterance between two chunks of a streamed decode, for R scores. A streamed
// workspace holds [B] float blocks, and for a float64 stream [B] double blocks after them
// (StreamState64): the float kernels always find a valid beam in their own blocks, whichever score
// type stepped the stream, and the two header words below tell the type of every step since the reset.
template <typename R>
struct StreamHdrT;
template <>
struct StreamHdrT<float> {
  int n;         // members in the beam
  unsigned gap;  // score-range prediction of the fast kernel
  int flags;     // bit0 rounding anomaly, bit2 more frames than the stream was sized for, kStreamNoF32Step
  int type;      // score bytes of the stream, set by the reset (the float kernels leave it alone);
                 // kStreamF64Stepped is or-ed in by a float64 step
};
template <>
struct StreamHdrT<double> {
  int n;
  int flags;
  int type;  // 8 once a double kernel has written the block (0 after a reset)
  int pad;
  unsigned long long gap;  // the fast kernel's 64-bit key
};
using StreamHdr = StreamHdrT<float>;
// float header flag set by the reset and dropped by every float step (each one rewrites the flags)
constexpr int kStreamNoF32Step = 1 << 30;
// float header type bit: a float64 step ran on a stream reset for float scores
constexpr int kStreamF64Stepped = 1 << 8;

template <typename R = float>
__host__ __device__ inline size_t StreamStateBytes(int W) {
  // 5 scores + label + 2 x u64 per slot: 16 + 40 W bytes for float, 24 + 60 W for double
  return (sizeof(StreamHdrT<R>) + (size_t)W * (5 * sizeof(R) + 20) + 15) / 16 * 16;
}
// the double blocks of a float64 stream: right after the [B] float blocks (256-byte aligned)
__host__ __device__ inline unsigned char* StreamState64(unsigned char* state, int B, int W) {
  return state + ((size_t)B * StreamStateBytes<float>(W) + 255) / 256 * 256;
}
template <typename R>
struct StreamViewT {
  StreamHdrT<R>* hdr;
  R *total, *blk, *lab, *ab, *an;
  int* label;
  unsigned long long *hash, *phash;
  __host__ __device__ StreamViewT(unsigned char* base, int W) {
    hdr = reinterpret_cast<StreamHdrT<R>*>(base);
    total = reinterpret_cast<R*>(base + sizeof(StreamHdrT<R>));
    blk = total + W; lab = blk + W; ab = lab + W; an = ab + W;
    if constexpr (sizeof(R) == 4) {
      label = reinterpret_cast<int*>(an + W);
      hash = reinterpret_cast<unsigned long long*>(label + W);
      phash = hash + W;
    } else {  // the 8-byte arrays first: aligned for any W
      hash = reinterpret_cast<unsigned long long*>(an + W);
      phash = hash + W;
      label = reinterpret_cast<int*>(phash + W);
    }
  }
};
using StreamView = StreamViewT<float>;


// Kernel 3: trace-back
struct TraceParams {
  const void* bp;  // [B,T,W] records, uint2 or unsigned (the kernels are templated on the type)
  const int* seq_len;
  const int* fin_kind;
  const int* fin_n;
  int T, B, W, P;
  int merge_repeated, blank_label;
  int* dec_len;  // [B,P]
  int* dec;      // [B,P,T]
  int* ali_len;  // [B,P]
  int* ali;      // [B,P,T]
};

// Kernels 4/5: sparse packing
struct ScanParams {
  const int* dec_len;  // [B,P]
  const int* ali_len;  // [B,P]
  int B, P;
  long long* dec_off;  // [P,B]
  long long* ali_off;  // [P,B]
  long long* sizes;    // [4,P]: n_dec, max_dec, n_ali, max_ali
};

struct PackParams {
  const int* dec_len; const int* dec; const int* ali_len; const int* ali;  // dense rows
  const long long* dec_off; const long long* ali_off;                      // [P,B]
  const long long* sizes;                                                   // [4,P]
  const void* fin_total;                                                    // [B,P] float or double
  long long* const* ptrs;  // device table [6,P]: dec_idx, dec_val, dec_shape, ali_idx, ali_val, ali_shape
                           // (+ entry 6*P: log_probability, used when log_prob is null -- compact pack)
  void* log_prob;          // [B,P] float or double
  const int* skip;         // optional device word: non-zero = the table is invalid, write nothing
  int real_bytes;          // 4 or 8
  int T, B, P;
};

}  // namespace ctcx
