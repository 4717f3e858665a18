// C-ABI shim (include/ctcx.h): validation, workspace carve-up, stream choreography and the host-buffer
// entries. The kernels live in their own translation units behind ctcx_launch.h. No CPU fallback.
//
// Reference counterparts (tensorflow_ctc_ext_beam_search_decoder/cc/kernels/
// ctc_ext_beam_search_decoder_kernels.cc): ValidateInputsGenerateOutputs :97-160, Compute :20-95,
// StoreAllDecodedSequences :163-257.
// the library is built with -fvisibility=hidden: only what include/ctcx.h declares is exported
#pragma GCC visibility push(default)
#include "../../include/ctcx.h"
#pragma GCC visibility pop

#include <cuda_runtime.h>

#include <algorithm>
#include <atomic>
#include <climits>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <vector>

#include "ctcx_launch.h"

namespace {

thread_local char g_cuda_err[256] = "";

bool Check(cudaError_t e, const char* what) {
  if (e == cudaSuccess) return true;
  std::snprintf(g_cuda_err, sizeof(g_cuda_err), "%s: %s", what, cudaGetErrorString(e));
  return false;
}
#define CTCX_CUDA(call)                                 \
  do {                                                  \
    if (!Check((call), #call)) return CTCX_ERR_CUDA;    \
  } while (0)

// result of a kernel launcher -> CTCX_* code
int FromLaunch(const ctcx::LaunchStatus& st) {
  if (st.code == ctcx::kLaunchCuda) Check(st.cuda, st.what);
  return st.code;
}
#define CTCX_RC(call)                           \
  do {                                          \
    const int rc_ = (call);                     \
    if (rc_ != CTCX_OK) return rc_;             \
  } while (0)
#define CTCX_LAUNCH(call) CTCX_RC(FromLaunch(call))

constexpr int kMaxBeamWidth = 1024;
constexpr int kMaxClasses = 65535;
constexpr uint32_t kMagic = 0x43544359u;  // "CTCY": workspace layout of this build
constexpr int kNStats = 16;
// control word (Workspace::ctrl) set when a scorer table with a positive entry was passed
constexpr int kCtrlTablePositive = 8;

size_t Align256(size_t v) { return (v + 255) / 256 * 256; }

// The result block, ONE copy to the host: sizes [4,P] int64, then the kNStats status words (stats[0..5]
// as FlagsKernel reduces them; stats[6] = the compact pack's overflow word).
size_t StatsOffset(int P) { return 4 * (size_t)P * 8; }
size_t ResultBytes(int P) { return StatsOffset(P) + kNStats * 4; }
// status words before the kernels run: no flags, and B (= none) as every "first failing utterance"
void InitStats(int* stats, int B) {
  stats[0] = 0;
  for (int k = 1; k < 6; ++k) stats[k] = B;
}

// test hook (ctcx_debug_set_beam_impl): 1 = route every decode to the generic beam kernel
std::atomic<int> g_force_generic{0};
// measurement hook (ctcx_debug_set_cycles_buffer)
thread_local long long* g_dbg_cycles = nullptr;
thread_local int g_dbg_slots = 24;

enum Path { kPathNarrow, kPathWide, kPathGeneric };
// which beam kernel (and with it which pre-pass) decodes this shape with R scores
template <typename R>
Path PathOf(int W, int C, bool scorer) {
  if (g_force_generic.load(std::memory_order_relaxed)) return kPathGeneric;
  if (ctcx::NarrowFastShape(W, C)) return kPathNarrow;  // (has a scorer variant: all 32 classes tested per row)
  // a scorer table breaks the wide kernel's monotone-prefix argument, and the wide kernel has no
  // float64 form: generic kernel
  if (scorer || sizeof(R) == 8) return kPathGeneric;
  if (ctcx::WideFastShape(W, C)) return kPathWide;
  return kPathGeneric;
}

// Everything a decode leaves behind for pack, at fixed offsets inside the caller's workspace. The
// layout is a pure function of the shape; the first group (up to `ali`) depends on (T, B, P) only, so
// ctcx_pack_* needs neither the class count nor the beam width, and no look at the device header.
struct Workspace {
  struct Header {
    uint32_t magic;
    int T, B, C, W, P;
    int real_bytes;  // 4: float32 decode, 8: float64 decode
  };
  size_t header, result, stats, ctrl, dec_len, ali_len, dec_off, ali_off, ptrs, fin_total, fin_kind, dec, ali,
      seq, chunk_len, fin_n, flags, t_done, state, off, bp, srt_pl, srt_cls, scratch, bytes;
  int Cs;         // row stride of the sorted-class arrays (0 when the wide fast path does not apply)
  int rec_bytes;  // back-pointer record size
  size_t InitPack(int T, int B, int P) {
    size_t o = 0;
    const size_t b = (size_t)B, t = (size_t)T, pp = (size_t)P;
    header = o; o += Align256(sizeof(Header));
    result = o; o += Align256(ResultBytes(P));
    stats = result + StatsOffset(P);
    ctrl = o; o += 256;                                          // [0] utterance queue, [1] frames landed
    dec_len = o; o += Align256(b * pp * 4);
    ali_len = o; o += Align256(b * pp * 4);
    dec_off = o; o += Align256(pp * b * 8);
    ali_off = o; o += Align256(pp * b * 8);
    ptrs = o; o += Align256((6 * pp + 1) * 8);                  // output pointer table (+ log_probability for the compact pack)
    fin_total = o; o += Align256(b * pp * 8);                    // float or double
    fin_kind = o; o += Align256(b * pp * 4);
    dec = o; o += Align256(b * pp * t * 4);
    ali = o; o += Align256(b * pp * t * 4);
    return o;
  }
  // score_bytes: 8 = room for a float64 stream (the double state blocks after the float ones)
  void Init(int T, int B, int C, int W, int P, int score_bytes = 4) {
    size_t o = InitPack(T, B, P);
    const size_t b = (size_t)B, t = (size_t)T, w = (size_t)W;
    seq = o; o += Align256(b * 4);                               // sequence_length of host-input decodes
    chunk_len = o; o += Align256(b * 4);                         // frames per utterance of the time chunk being decoded
    fin_n = o; o += Align256(b * 4);
    flags = o; o += Align256(b * 4);
    t_done = o; o += Align256(b * 4);                            // streaming: frames consumed so far
    const bool narrow = ctcx::NarrowFastShape(W, C), wide = ctcx::WideFastShape(W, C);
    off = o; o += Align256(t * b * 8);                           // float or double (unused by the narrow kernel, which normalises itself)
    rec_bytes = ctcx::RecBytes(W, C);
    bp = o; o += Align256(b * t * w * (size_t)rec_bytes);
    Cs = wide ? ctcx::WideKs(W, C) : 0;                          // wide fast path: best classes per frame, sorted
    srt_pl = o; o += Align256(t * b * (size_t)Cs * 4);
    srt_cls = o; o += Align256(t * b * (size_t)Cs * 2);
    // shapes served by the generic kernel only: room to upcast half-precision logits (the fast kernels
    // read them directly)
    scratch = o; o += (narrow || wide) ? 0 : Align256(t * b * (size_t)C * 4);
    // streaming: the beam between chunks (last, so that no other offset depends on the score type)
    state = o; o += Align256(b * ctcx::StreamStateBytes(W));
    if (score_bytes == 8) o += Align256(b * ctcx::StreamStateBytes<double>(W));  // at ctcx::StreamState64
    bytes = o;
  }
  // the upcast room, or null where a fast kernel takes the shape (even with the generic kernel forced:
  // the layout does not depend on the test hook)
  float* Scratch(unsigned char* base) const { return state > scratch ? (float*)(base + scratch) : nullptr; }
};

thread_local int g_err_batch = -1;
thread_local int g_err_max_time = 0;
thread_local char g_msg[160];

// optional per-kernel timing (ctcx_profile_enable): CUDA events on the launching stream
thread_local int g_profile = 0;
thread_local cudaEvent_t g_ev[6];
thread_local bool g_ev_ready = false;
thread_local float g_ms[5] = {0, 0, 0, 0, 0};  // pre-pass, beam, trace, scan+flags, total
void ProfRecord(int i, cudaStream_t s) {
  if (!g_profile) return;
  if (!g_ev_ready) {
    for (int k = 0; k < 6; ++k) cudaEventCreate(&g_ev[k]);
    g_ev_ready = true;
  }
  cudaEventRecord(g_ev[i], s);
}

struct DecodeOpts {
  int in_dtype = ctcx::kInF32;     // float32 decodes: element type of the logits
  long long tstride = 0;           // elements between frames; 0 = batch * num_classes
  const int* ready = nullptr;      // device word "frames landed" (narrow path only), or null
  const void* lm = nullptr;        // scorer table (float32 decodes)
  // wide path, host feed: the logits arrive in n_slabs time slabs, slab k = frames [slab_end[k-1], slab_end[k]),
  // complete once slab_event[k] has fired; the decode then runs slab by slab behind the copies
  int n_slabs = 0;
  const int* slab_end = nullptr;
  const cudaEvent_t* slab_event = nullptr;
};

// header + zeroed sizes + initial stats + control words, staged in one host block -> one H2D copy
struct InitBlock {
  std::vector<unsigned char> bytes;
  InitBlock(const Workspace& ws, const Workspace::Header& hdr, int B) : bytes(ws.dec_len, 0) {
    std::memcpy(bytes.data() + ws.header, &hdr, sizeof(hdr));
    InitStats(reinterpret_cast<int*>(bytes.data() + ws.stats), B);
  }
};

// per-kernel times of the LAST decode this thread enqueued (ctcx_profile_enable), once it has completed
void CollectProfile(int B) {
  if (!g_profile || B <= 0 || !g_ev_ready || cudaEventQuery(g_ev[4]) != cudaSuccess) return;
  for (int k = 0; k < 4; ++k) cudaEventElapsedTime(&g_ms[k], g_ev[k], g_ev[k + 1]);
  cudaEventElapsedTime(&g_ms[4], g_ev[0], g_ev[4]);
}

// the result block as it arrived on the host -> sizes, flags, return code
int ParseResult(const unsigned char* h_res, int T, int B, int P, ctcx_sizes* sizes, int32_t* flags_out) {
  const long long* h_sizes = (const long long*)h_res;
  const int* h_stats = (const int*)(h_res + StatsOffset(P));
  if (h_stats[6] != 0) return CTCX_ERR_WORKSPACE;  // ctcx_pack_compact: the caller's buffer was too small
  if (h_stats[5] < B) {
    std::snprintf(g_cuda_err, sizeof(g_cuda_err), "the host->device copy of the logits never delivered the frames of utterance %d",
                  h_stats[5]);
    return CTCX_ERR_CUDA;
  }
  if (h_stats[2] < B) {  // kernels.cc:134-138
    g_err_batch = h_stats[2];
    g_err_max_time = T;
    return CTCX_ERR_SEQ_LEN_RANGE;
  }
  if (h_stats[3] < B) return CTCX_ERR_BAD_ARGUMENT;  // negative sequence_length
  if (h_stats[4] < B) {  // streaming: an utterance was fed more frames than the stream holds
    g_err_batch = h_stats[4];
    g_err_max_time = T;
    return CTCX_ERR_SEQ_LEN_RANGE;
  }
  if (h_stats[1] < B) return CTCX_ERR_TOO_FEW_LEAVES;
  for (int p = 0; p < P; ++p) {
    if (sizes->n_decoded) sizes->n_decoded[p] = h_sizes[0 * (size_t)P + p];
    if (sizes->max_decoded) sizes->max_decoded[p] = h_sizes[1 * (size_t)P + p];
    if (sizes->n_alignment) sizes->n_alignment[p] = h_sizes[2 * (size_t)P + p];
    if (sizes->max_alignment) sizes->max_alignment[p] = h_sizes[3 * (size_t)P + p];
  }
  if (flags_out) *flags_out = h_stats[0];
  return CTCX_OK;
}

// ONE copy brings the sparse sizes and the status words to the host; the only synchronisation of a decode
int FinishImpl(const unsigned char* d_result, int T, int B, int P, cudaStream_t stream, ctcx_sizes* sizes,
               int32_t* flags_out) {
  std::vector<unsigned char> h_res(ResultBytes(P));
  CTCX_CUDA(cudaMemcpyAsync(h_res.data(), d_result, h_res.size(), cudaMemcpyDeviceToHost, stream));
  CTCX_CUDA(cudaStreamSynchronize(stream));
  CollectProfile(B);
  return ParseResult(h_res.data(), T, B, P, sizes, flags_out);
}

// Logits as the kernels read them: [T,B,C] of element type in_dtype (float64 decodes: kInF32, unused),
// row (t, b) at element t * tstride + b * C.
struct Logits {
  const void* p;
  int in_dtype;
  long long tstride;
};

// Enqueues the normaliser pre-pass the beam kernel of `path` needs, over the T*B rows of `x`: nothing
// for the narrow kernel, which normalises inside; the normaliser and every row's best classes, sorted,
// for the wide kernel; the normaliser alone for the generic kernel, half-precision logits first widened
// exactly into `scratch` ([T,B,C] float32; null = no room), which then stands in for `x`.
template <typename R>
int PrePass(Path path, Logits& x, int T, int B, int C, int blank_index, int W, R* off, float* srt_pl,
            unsigned short* srt_cls, float* scratch, cudaStream_t stream) {
  const long long rows = (long long)T * B;
  if (path == kPathNarrow) return CTCX_OK;
  if constexpr (sizeof(R) == 8) {
    CTCX_LAUNCH(ctcx::LaunchLogNorm((const double*)x.p, off, rows, C, B, x.tstride, stream));
  } else if (path == kPathWide) {
    CTCX_LAUNCH(ctcx::LaunchNormTopClasses(x.p, x.in_dtype, off, rows, C, blank_index, W, srt_pl, srt_cls, B,
                                           x.tstride, stream));
  } else {
    if (x.in_dtype != ctcx::kInF32) {
      if (scratch == nullptr) return CTCX_ERR_UNSUPPORTED;
      CTCX_LAUNCH(ctcx::LaunchUpcast(x.p, x.in_dtype, scratch, T, B, C, x.tstride, stream));
      x = {scratch, ctcx::kInF32, (long long)B * C};
    }
    CTCX_LAUNCH(ctcx::LaunchLogNorm((const float*)x.p, off, rows, C, B, x.tstride, stream));
  }
  return CTCX_OK;
}

// The beam kernels' parameters over a workspace laid out for Tcap frames: a pass over all of them that
// carries no beam in or out. Streamed passes add state and t_done.
template <typename R>
ctcx::BeamParamsT<R> BeamParamsOf(const Workspace& ws, unsigned char* base, int Tcap, int B, int C, int W, int P,
                                  int blank_index, const int* seq_len) {
  ctcx::BeamParamsT<R> bp;
  std::memset(&bp, 0, sizeof(bp));
  bp.off = (const R*)(base + ws.off);
  bp.seq_len = seq_len;
  bp.T = Tcap; bp.B = B; bp.C = C; bp.W = W; bp.P = P;
  bp.blank_index = blank_index;
  if (ws.rec_bytes == 4) bp.bp32 = (unsigned*)(base + ws.bp); else bp.bp = (uint2*)(base + ws.bp);
  bp.fin_total = (R*)(base + ws.fin_total);
  bp.fin_kind = (int*)(base + ws.fin_kind);
  bp.fin_n = (int*)(base + ws.fin_n);
  bp.flags = (int*)(base + ws.flags);
  bp.Tcap = Tcap;
  if (ws.Cs > 0) {  // the wide kernel's sorted classes
    bp.srt_pl = (const R*)(base + ws.srt_pl);
    bp.srt_cls = (const unsigned short*)(base + ws.srt_cls);
  }
  bp.queue = (int*)(base + ws.ctrl);
  bp.n_slices = 1;
  bp.slice_frames = Tcap;
  return bp;
}

// One beam pass over the frames [0, bp.T) of `x`: the pre-pass of `path` into the workspace, then the
// beam kernel of `path`. `after_prepass`, if set, is recorded between the two.
template <typename R>
int BeamPass(Path path, Logits x, ctcx::BeamParamsT<R>& bp, const Workspace& ws, unsigned char* base,
             cudaEvent_t after_prepass, cudaStream_t stream) {
  CTCX_RC(PrePass<R>(path, x, bp.T, bp.B, bp.C, bp.blank_index, bp.W, (R*)(base + ws.off), (float*)(base + ws.srt_pl),
                     (unsigned short*)(base + ws.srt_cls), ws.Scratch(base), stream));
  if (after_prepass != nullptr) cudaEventRecord(after_prepass, stream);
  bp.logits = (const R*)x.p;
  bp.tstride = x.tstride;
  if (path == kPathGeneric) CTCX_LAUNCH(ctcx::LaunchBeamGeneric(bp, stream));
  else if constexpr (sizeof(R) == 8) CTCX_LAUNCH(ctcx::LaunchBeamNarrow(bp, stream));  // (no float64 wide kernel)
  else if (path == kPathNarrow) CTCX_LAUNCH(ctcx::LaunchBeamNarrow(bp, x.in_dtype, stream));
  else CTCX_LAUNCH(ctcx::LaunchBeamWide(bp, x.in_dtype, stream));
  return CTCX_OK;
}

// One Step() of a streamed decode with R scores: up to chunk_len[b] frames of the chunk `x` for every
// utterance, the beam carried in from and out to the state blocks. `lm`: scorer table (float), or null.
template <typename R>
int StreamStep(const Workspace& ws, unsigned char* base, int T_total, int B, int C, int W, int P, const Logits& x,
               int chunk_time, const int32_t* chunk_len_dev, int blank_index, const float* lm, cudaStream_t stream) {
  ctcx::BeamParamsT<R> bp = BeamParamsOf<R>(ws, base, T_total, B, C, W, P, blank_index,
                                            chunk_len_dev);  // frames of THIS chunk to consume, per utterance
  bp.T = chunk_time;
  bp.t_done = (int*)(base + ws.t_done);
  bp.state = base + ws.state;
  bp.lm = (const R*)lm;
  const Path path = PathOf<R>(W, C, lm != nullptr);
  if (path == kPathNarrow) CTCX_CUDA(cudaMemsetAsync(bp.queue, 0, 4, stream));  // the queue word, zero at launch
  return BeamPass(path, x, bp, ws, base, nullptr, stream);
}

// Trace-back of the top paths over the first seq_len[b] frames, then the sparse offsets and sizes and the
// status words into the result block. `mask`: optional [B] device words, non-zero = utterance traced and
// checked; the others contribute lengths 0.
int TraceScanFlags(const Workspace& ws, unsigned char* base, const int* seq_len, int T, int B, int W, int P,
                   int merge_repeated, int blank_label, cudaEvent_t after_trace, cudaStream_t stream,
                   const int* mask = nullptr) {
  ctcx::TraceParams tp;
  tp.bp = base + ws.bp; tp.seq_len = seq_len;
  tp.fin_kind = (const int*)(base + ws.fin_kind); tp.fin_n = (const int*)(base + ws.fin_n);
  tp.T = T; tp.B = B; tp.W = W; tp.P = P;
  tp.merge_repeated = merge_repeated ? 1 : 0; tp.blank_label = blank_label;
  tp.dec_len = (int*)(base + ws.dec_len); tp.dec = (int*)(base + ws.dec);
  tp.ali_len = (int*)(base + ws.ali_len); tp.ali = (int*)(base + ws.ali);
  tp.mask = mask;
  ctcx::ScanParams sp;
  sp.dec_len = tp.dec_len; sp.ali_len = tp.ali_len; sp.B = B; sp.P = P;
  sp.dec_off = (long long*)(base + ws.dec_off); sp.ali_off = (long long*)(base + ws.ali_off);
  sp.sizes = (long long*)(base + ws.result);
  return FromLaunch(ctcx::LaunchTraceScanFlags(tp, ws.rec_bytes, sp, (const int*)(base + ws.flags),
                                               (int*)(base + ws.stats), stream, after_trace));
}

// The sparse outputs from the dense rows a decode left in the workspace, through the pointer table at
// ws.ptrs. `skip`: optional device word, non-zero = write nothing.
int Pack(const Workspace& ws, const unsigned char* base, int T, int B, int P, void* log_prob, const int* skip,
         int real_bytes, cudaStream_t stream) {
  ctcx::PackParams pp;
  pp.dec_len = (const int*)(base + ws.dec_len); pp.dec = (const int*)(base + ws.dec);
  pp.ali_len = (const int*)(base + ws.ali_len); pp.ali = (const int*)(base + ws.ali);
  pp.dec_off = (const long long*)(base + ws.dec_off); pp.ali_off = (const long long*)(base + ws.ali_off);
  pp.sizes = (const long long*)(base + ws.result);
  pp.fin_total = (const void*)(base + ws.fin_total);
  pp.ptrs = (long long* const*)(base + ws.ptrs);
  pp.log_prob = log_prob;
  pp.skip = skip;
  pp.real_bytes = real_bytes;
  pp.T = T; pp.B = B; pp.P = P;
  return FromLaunch(ctcx::LaunchPack(pp, stream));
}

template <typename R>
int DecodeImpl(const void* logits_dev, int T, int B, int C, const int32_t* seq_len_dev, int W,
               int P, int merge_repeated, int blank_index, int blank_label, void* workspace,
               size_t workspace_bytes, void* stream_v, ctcx_sizes* sizes, int32_t* flags_out,
               const DecodeOpts& opt) {
  cudaStream_t stream = (cudaStream_t)stream_v;
  // --- validation, in the reference's order (kernels.cc:111-138), then TopPaths' (decoder.h:237) ---
  if (T == 0) return CTCX_ERR_MAX_TIME_ZERO;
  if (T < 0 || B < 0 || C <= 0 || W < 1 || P < 1 || blank_index < 0 || blank_index >= C)
    return CTCX_ERR_BAD_ARGUMENT;
  if (W > kMaxBeamWidth || C > kMaxClasses) return CTCX_ERR_UNSUPPORTED;
  const bool defer = (sizes == nullptr);  // enqueue only: ctcx_finish() brings the sizes and the status later
  const long long tstride = opt.tstride ? opt.tstride : (long long)B * C;
  if (tstride < (long long)B * C) return CTCX_ERR_BAD_ARGUMENT;
  Workspace ws;
  ws.Init(T, B, C, W, P);
  if (workspace == nullptr || workspace_bytes < ws.bytes || ((uintptr_t)workspace & 255u))
    return CTCX_ERR_WORKSPACE;
  unsigned char* base = (unsigned char*)workspace;
  int* d_stats = (int*)(base + ws.stats);
  int* d_ctrl = (int*)(base + ws.ctrl);

  // sequence_length lives on the device: its range check (kernels.cc:134-138) is folded into the
  // flags reduction at the end -- every kernel clamps the lengths it walks -- so that a decode has
  // ONE host round trip. Only when top_paths > beam_width (an error either way) is it evaluated
  // first, because the reference reports a bad length before TopPaths' own error (decoder.h:237).
  Workspace::Header hdr = {kMagic, T, B, C, W, P, (int)sizeof(R)};
  {
    // the control words are not part of this copy when a host->device feed owns them (opt.ready)
    InitBlock init(ws, hdr, B);
    const size_t n = (opt.ready != nullptr) ? ws.ctrl : ws.dec_len;
    CTCX_CUDA(cudaMemcpyAsync(base, init.bytes.data(), n, cudaMemcpyHostToDevice, stream));
    if (opt.ready != nullptr) CTCX_CUDA(cudaMemsetAsync(d_ctrl, 0, 4, stream));  // the queue word only
  }
  if (B > 0 && P > W) {
    CTCX_LAUNCH(ctcx::LaunchFlagsOnly(seq_len_dev, B, T, d_stats, stream));
    int h[kNStats];
    CTCX_CUDA(cudaMemcpyAsync(h, d_stats, sizeof(h), cudaMemcpyDeviceToHost, stream));
    CTCX_CUDA(cudaStreamSynchronize(stream));
    if (h[2] < B) {
      g_err_batch = h[2];
      g_err_max_time = T;
      return CTCX_ERR_SEQ_LEN_RANGE;
    }
    if (h[3] < B) return CTCX_ERR_BAD_ARGUMENT;
    // TopPaths is reached for utterance 0 only after its frames; for B == 0 it is never reached
    return CTCX_ERR_TOO_MANY_PATHS;
  }

  if (B > 0) {
    ProfRecord(0, stream);
    const Path path = PathOf<R>(W, C, opt.lm != nullptr);
    ctcx::BeamParamsT<R> bp = BeamParamsOf<R>(ws, base, T, B, C, W, P, blank_index, seq_len_dev);
    bp.lm = (const R*)opt.lm;
    bp.ready = opt.ready;
    bp.dbg_cycles = g_dbg_cycles;
    bp.dbg_slots = g_dbg_slots;
    const Logits x = {logits_dev, opt.in_dtype, tstride};
    if (path == kPathWide && opt.n_slabs > 0) {
      // Host feed of a wide-vocabulary batch: the copy (hundreds of MB) takes longer than the decode, so
      // the decode runs time chunk by time chunk behind it -- plain stream order, one event per slab. The
      // beam crosses chunks through the per-utterance state block, exactly as in a streamed decode
      // (ctcx_stream_step_f32); the class-selection arrays are chunk-relative and stay in L2.
      const size_t es = (x.in_dtype == ctcx::kInF32) ? 4 : 2;
      int* d_chunk_len = (int*)(base + ws.chunk_len);
      bp.seq_len = d_chunk_len;
      bp.t_done = (int*)(base + ws.t_done);
      bp.state = base + ws.state;
      CTCX_CUDA(cudaMemsetAsync(bp.t_done, 0, (size_t)B * 4, stream));
      ProfRecord(1, stream);
      int t0 = 0;
      for (int k = 0; k < opt.n_slabs; ++k) {
        const int len = opt.slab_end[k] - t0;
        CTCX_CUDA(cudaStreamWaitEvent(stream, opt.slab_event[k], 0));
        CTCX_LAUNCH(ctcx::LaunchChunkLen(seq_len_dev, B, T, t0, len, d_chunk_len, stream));
        bp.T = len;
        const Logits chunk = {(const unsigned char*)x.p + (size_t)t0 * (size_t)tstride * es, x.in_dtype, tstride};
        CTCX_RC(BeamPass(path, chunk, bp, ws, base, nullptr, stream));
        t0 = opt.slab_end[k];
      }
    } else {
      if constexpr (sizeof(R) == 4) {
        if (path == kPathNarrow) {
          // time-sliced work queue (large batches): per-utterance state block + progress words (the regions
          // the streaming entries use for the same purpose between calls); the float64 kernel takes whole
          // utterances
          bp.state = base + ws.state;
          bp.progress = (int*)(base + ws.t_done);
          CTCX_CUDA(cudaMemsetAsync(bp.progress, 0, (size_t)B * 4, stream));
        }
      }
      CTCX_RC(BeamPass(path, x, bp, ws, base, g_profile ? g_ev[1] : nullptr, stream));
    }
    ProfRecord(2, stream);
    CTCX_RC(TraceScanFlags(ws, base, seq_len_dev, T, B, W, P, merge_repeated, blank_label,
                           g_profile ? g_ev[3] : nullptr, stream));
    ProfRecord(4, stream);
  }

  if (defer) return CTCX_OK;
  return FinishImpl(base + ws.result, T, B, P, stream, sizes, flags_out);
}

int PackImpl(const void* workspace, int T, int B, int P, int64_t* const* decoded_indices,
             int64_t* const* decoded_values, int64_t* const* decoded_shape,
             int64_t* const* alignment_indices, int64_t* const* alignment_values,
             int64_t* const* alignment_shape, void* log_probability, int real_bytes, void* stream_v) {
  cudaStream_t stream = (cudaStream_t)stream_v;
  if (workspace == nullptr || T <= 0 || B < 0 || P < 1 || ((uintptr_t)workspace & 255u)) return CTCX_ERR_WORKSPACE;
  const unsigned char* base = (const unsigned char*)workspace;
  Workspace ws;
  ws.InitPack(T, B, P);  // everything pack touches is laid out by (T, B, P) alone: no look at the device
  // device copy of the 6*P output pointers
  std::vector<long long*> table(6 * (size_t)P);
  for (int p = 0; p < P; ++p) {
    table[0 * (size_t)P + p] = (long long*)decoded_indices[p];
    table[1 * (size_t)P + p] = (long long*)decoded_values[p];
    table[2 * (size_t)P + p] = (long long*)decoded_shape[p];
    table[3 * (size_t)P + p] = (long long*)alignment_indices[p];
    table[4 * (size_t)P + p] = (long long*)alignment_values[p];
    table[5 * (size_t)P + p] = (long long*)alignment_shape[p];
  }
  unsigned char* wbase = (unsigned char*)workspace;
  // (a cudaMemcpyAsync from pageable memory returns only after the source has been staged)
  CTCX_CUDA(cudaMemcpyAsync(wbase + ws.ptrs, table.data(), table.size() * sizeof(void*),
                            cudaMemcpyHostToDevice, stream));
  if (B > 0) {
    CTCX_RC(Pack(ws, base, T, B, P, log_probability, nullptr, real_bytes, stream));
  } else {
    // empty batch: shapes [0, 0]
    const long long zeros[2] = {0, 0};
    for (int p = 0; p < P; ++p) {
      CTCX_CUDA(cudaMemcpyAsync(decoded_shape[p], zeros, 16, cudaMemcpyHostToDevice, stream));
      CTCX_CUDA(cudaMemcpyAsync(alignment_shape[p], zeros, 16, cudaMemcpyHostToDevice, stream));
    }
  }
  return CTCX_OK;
}

// Stream-ordered 32-bit store (the driver's cuStreamWriteValue32, resolved at run time so that the
// library does not link against libcuda): how the copy stream publishes "frames landed". Unlike a
// 4-byte cudaMemcpyAsync from pageable memory it never synchronises with anything.
typedef int (*StreamWriteValue32Fn)(cudaStream_t, unsigned long long, unsigned, unsigned);
StreamWriteValue32Fn StreamWriteValue32() {
  static StreamWriteValue32Fn fn = []() -> StreamWriteValue32Fn {
    void* p = nullptr;
    cudaDriverEntryPointQueryResult q;
    if (cudaGetDriverEntryPoint("cuStreamWriteValue32", &p, cudaEnableDefault, &q) != cudaSuccess ||
        q != cudaDriverEntryPointSuccess)
      return nullptr;
    return (StreamWriteValue32Fn)p;
  }();
  return fn;
}

// true if `p` is page-locked host memory (cudaHostAlloc / cudaHostRegister): only then is a
// cudaMemcpyAsync truly asynchronous
bool IsPinned(const void* p) {
  cudaPointerAttributes a;
  if (cudaPointerGetAttributes(&a, p) != cudaSuccess) {
    cudaGetLastError();
    return false;
  }
  return a.type == cudaMemoryTypeHost;
}

// ---- host -> device feed of the logits in time slabs (ctcx_decode_hostin_*) ----
struct Feed {
  const unsigned char* src;   // host logits
  unsigned char* dst;         // device staging [T, B, C]
  size_t row_bytes;           // B * C * element size
  size_t src_pitch;           // host bytes between frames
  int T;
  int* d_ready;               // device word: frames landed
  bool flags;                 // publish progress per slab (the narrow kernel consumes it)
  cudaStream_t copy_stream;
  // explicit slab schedule (wide path): n_slabs slabs ending at frame slab_end[k], an event after each
  int n_slabs = 0;
  const int* slab_end = nullptr;
  const cudaEvent_t* slab_event = nullptr;
};
int RunFeed(void* arg) {
  Feed& f = *(Feed*)arg;
  // Slabs grow geometrically (6, 12, 24, ... 192 frames): the first frames land after a few microseconds so
  // the beam kernel can start, the bulk moves in large copies.
  int t0 = 0, n = f.flags ? 6 : f.T, k = 0;
  while (t0 < f.T) {
    const int t1 = (f.n_slabs > 0) ? f.slab_end[k] : std::min(f.T, t0 + n);
    cudaError_t e;
    if (f.src_pitch == f.row_bytes)
      e = cudaMemcpyAsync(f.dst + (size_t)t0 * f.row_bytes, f.src + (size_t)t0 * f.src_pitch,
                          (size_t)(t1 - t0) * f.row_bytes, cudaMemcpyHostToDevice, f.copy_stream);
    else
      e = cudaMemcpy2DAsync(f.dst + (size_t)t0 * f.row_bytes, f.row_bytes, f.src + (size_t)t0 * f.src_pitch,
                            f.src_pitch, f.row_bytes, (size_t)(t1 - t0), cudaMemcpyHostToDevice, f.copy_stream);
    bool ok = Check(e, "host->device copy of the logits");
    if (ok && f.flags && StreamWriteValue32()(f.copy_stream, (unsigned long long)(uintptr_t)f.d_ready, (unsigned)t1, 0) != 0) {
      std::snprintf(g_cuda_err, sizeof(g_cuda_err), "cuStreamWriteValue32 failed");
      ok = false;
    }
    if (ok && f.n_slabs > 0) ok = Check(cudaEventRecord(f.slab_event[k], f.copy_stream), "cudaEventRecord");
    if (!ok) {
      // release the kernel: it must not wait for frames that will never come
      if (f.flags) StreamWriteValue32()(f.copy_stream, (unsigned long long)(uintptr_t)f.d_ready, (unsigned)INT_MAX, 0);
      return CTCX_ERR_CUDA;
    }
    t0 = t1;
    ++k;
    n = std::min(192, n * 2);  // doubling: a slab lands before the previous one is consumed at any copy rate >= 2x the kernel's
  }
  return CTCX_OK;
}

size_t ElemBytes(int dtype) {
  switch (dtype) {
    case CTCX_F32: return 4;
    case CTCX_F16: case CTCX_BF16: return 2;
    case CTCX_F64: return 8;
    default: return 0;
  }
}
int InDtypeOf(int dtype) {
  return dtype == CTCX_F16 ? ctcx::kInF16 : dtype == CTCX_BF16 ? ctcx::kInBF16 : ctcx::kInF32;
}

// argument checks of a stream reset (full or per slot), before any CUDA call; lays out *ws
int CheckStreamReset(const void* workspace, size_t workspace_bytes, int score_dtype, int T_total, int B, int C, int W,
                     int P, Workspace* ws) {
  if (score_dtype != CTCX_F32 && score_dtype != CTCX_F64) return CTCX_ERR_BAD_ARGUMENT;
  if (T_total <= 0 || B < 0 || C <= 0 || W < 1 || P < 1) return CTCX_ERR_BAD_ARGUMENT;
  if (W > kMaxBeamWidth || C > kMaxClasses) return CTCX_ERR_UNSUPPORTED;
  if (P > W) return CTCX_ERR_TOO_MANY_PATHS;
  ws->Init(T_total, B, C, W, P, (int)ElemBytes(score_dtype));
  if (workspace == nullptr || workspace_bytes < ws->bytes || ((uintptr_t)workspace & 255u))
    return CTCX_ERR_WORKSPACE;
  return CTCX_OK;
}

// TopPaths() of a stream for the utterances `mask` selects (null = all), after the checks of its entry:
// trace-back, sparse sizes and status words into the result block. sizes == NULL: only enqueued, completed
// like a deferred decode; otherwise one synchronisation and the reference's checks.
int StreamTopPaths(void* workspace, int T_total, int B, int C, int W, int P, int merge_repeated, int blank_label,
                   const int* mask, cudaStream_t stream, ctcx_sizes* sizes, int32_t* flags_out) {
  Workspace ws;
  ws.Init(T_total, B, C, W, P);
  unsigned char* base = (unsigned char*)workspace;
  std::vector<unsigned char> h_res(ResultBytes(P), 0);
  InitStats((int*)(h_res.data() + StatsOffset(P)), B);
  const bool defer = (sizes == nullptr);
  if (B > 0 || defer)  // (a deferred result is read from the device: it must hold the empty batch's too)
    CTCX_CUDA(cudaMemcpyAsync(base + ws.result, h_res.data(), h_res.size(), cudaMemcpyHostToDevice, stream));
  if (B > 0) {
    CTCX_RC(TraceScanFlags(ws, base, (const int*)(base + ws.t_done) /* frames consumed so far */, T_total, B, W, P,
                           merge_repeated, blank_label, nullptr, stream, mask));
    // score types mixed since the reset, or a table with a positive entry: CTCX_ERR_BAD_ARGUMENT
    CTCX_LAUNCH(ctcx::LaunchStreamCheck(base + ws.state, B, W, (const int*)(base + ws.ctrl) + kCtrlTablePositive,
                                        (int*)(base + ws.stats), mask, stream));
  }
  if (defer) return CTCX_OK;
  if (B > 0) {
    CTCX_CUDA(cudaMemcpyAsync(h_res.data(), base + ws.result, h_res.size(), cudaMemcpyDeviceToHost, stream));
    CTCX_CUDA(cudaStreamSynchronize(stream));
  }
  return ParseResult(h_res.data(), T_total, B, P, sizes, flags_out);
}

}  // namespace

extern "C" {

const char* ctcx_strerror(int code) {
  switch (code) {
    case CTCX_OK: return "ok";
    case CTCX_ERR_INPUTS_NOT_3D: return "inputs is not a 3-Tensor";
    case CTCX_ERR_MAX_TIME_ZERO: return "max_time is 0";
    case CTCX_ERR_SEQ_LEN_NOT_VECTOR: return "sequence_length is not a vector";
    case CTCX_ERR_SEQ_LEN_BATCH: return "len(sequence_length) != batch_size.  ";
    case CTCX_ERR_SEQ_LEN_RANGE:
      std::snprintf(g_msg, sizeof(g_msg), "sequence_length(%d) <= %d", g_err_batch, g_err_max_time);
      return g_msg;
    case CTCX_ERR_TOO_MANY_PATHS: return "requested more paths than the beam width.";
    case CTCX_ERR_TOO_FEW_LEAVES: return "Less leaves in the beam search than requested.";
    case CTCX_ERR_BAD_ARGUMENT: return "bad argument (blank_index outside [0, num_classes), negative sequence_length, beam_width/top_paths < 1, or a time stride shorter than a frame)";
    case CTCX_ERR_UNSUPPORTED: return "shape not supported by this build (see ctcx_get_limits)";
    case CTCX_ERR_WORKSPACE: return "workspace missing, misaligned or too small";
    case CTCX_ERR_CUDA: return g_cuda_err;
    default: return "unknown error";
  }
}

const char* ctcx_last_cuda_error(void) { return g_cuda_err; }

int ctcx_error_batch_index(void) { return g_err_batch; }

int ctcx_get_limits(ctcx_limits* out) {
  if (out) {
    out->max_beam_width = kMaxBeamWidth;
    out->max_classes = kMaxClasses;
    out->max_top_paths = kMaxBeamWidth;
  }
  return 100;
}

size_t ctcx_workspace_bytes(int T, int B, int C, int W, int P) {
  if (T <= 0 || B < 0 || C <= 0 || W <= 0 || P <= 0) return 0;
  Workspace ws;
  ws.Init(T, B, C, W, P);
  return ws.bytes;
}

int ctcx_decode_f32(const float* logits_dev, int T, int B, int C, const int32_t* seq_len_dev, int W,
                    int P, int merge_repeated, int blank_index, int blank_label, void* workspace,
                    size_t workspace_bytes, void* stream_v, ctcx_sizes* sizes, int32_t* flags_out) {
  return DecodeImpl<float>(logits_dev, T, B, C, seq_len_dev, W, P, merge_repeated, blank_index, blank_label,
                           workspace, workspace_bytes, stream_v, sizes, flags_out, DecodeOpts());
}

/* A view into a larger tensor / any of the four element types, decoded in place. */
int ctcx_decode_view(const void* logits_dev, int dtype, int64_t time_stride, int T, int B, int C,
                     const int32_t* seq_len_dev, int W, int P, int merge_repeated, int blank_index,
                     int blank_label, void* workspace, size_t workspace_bytes, void* stream_v,
                     ctcx_sizes* sizes, int32_t* flags_out) {
  if (ElemBytes(dtype) == 0 || time_stride < 0) return CTCX_ERR_BAD_ARGUMENT;
  DecodeOpts opt;
  opt.tstride = time_stride;
  if (dtype == CTCX_F64)
    return DecodeImpl<double>(logits_dev, T, B, C, seq_len_dev, W, P, merge_repeated, blank_index, blank_label,
                              workspace, workspace_bytes, stream_v, sizes, flags_out, opt);
  opt.in_dtype = InDtypeOf(dtype);
  return DecodeImpl<float>(logits_dev, T, B, C, seq_len_dev, W, P, merge_repeated, blank_index, blank_label,
                           workspace, workspace_bytes, stream_v, sizes, flags_out, opt);
}

/* Decode with a scorer plugged into the reference's extension point (util/ctc_beam_scorer.h:31-65). */
int ctcx_decode_scorer_f32(const float* logits_dev, int T, int B, int C, const int32_t* seq_len_dev, int W,
                           int P, int merge_repeated, int blank_index, int blank_label,
                           const float* expansion_scores_dev, void* workspace, size_t workspace_bytes,
                           void* stream_v, ctcx_sizes* sizes, int32_t* flags_out) {
  DecodeOpts opt;
  if (expansion_scores_dev != nullptr && C > 0) {  // expansion scores are log-probabilities: <= 0
    cudaStream_t stream = (cudaStream_t)stream_v;
    if (workspace == nullptr || ((uintptr_t)workspace & 255u)) return CTCX_ERR_WORKSPACE;
    Workspace ws;
    ws.Init(T > 0 ? T : 1, B > 0 ? B : 0, C, W > 0 ? W : 1, P > 0 ? P : 1);
    if (workspace_bytes < ws.bytes) return CTCX_ERR_WORKSPACE;
    int* d_flag = (int*)((unsigned char*)workspace + ws.ctrl) + kCtrlTablePositive;
    CTCX_CUDA(cudaMemsetAsync(d_flag, 0, 4, stream));
    CTCX_LAUNCH(ctcx::LaunchPositive(expansion_scores_dev, (long long)(C + 1) * C, d_flag, stream));
    int h_flag = 0;
    CTCX_CUDA(cudaMemcpyAsync(&h_flag, d_flag, 4, cudaMemcpyDeviceToHost, stream));
    CTCX_CUDA(cudaStreamSynchronize(stream));
    if (h_flag) return CTCX_ERR_BAD_ARGUMENT;
    opt.lm = expansion_scores_dev;
  }
  return DecodeImpl<float>(logits_dev, T, B, C, seq_len_dev, W, P, merge_repeated, blank_index, blank_label,
                           workspace, workspace_bytes, stream_v, sizes, flags_out, opt);
}

int ctcx_decode_f64(const double* logits_dev, int T, int B, int C, const int32_t* seq_len_dev, int W,
                    int P, int merge_repeated, int blank_index, int blank_label, void* workspace,
                    size_t workspace_bytes, void* stream_v, ctcx_sizes* sizes, int32_t* flags_out) {
  return DecodeImpl<double>(logits_dev, T, B, C, seq_len_dev, W, P, merge_repeated, blank_index, blank_label,
                            workspace, workspace_bytes, stream_v, sizes, flags_out, DecodeOpts());
}

/* fp16 / bf16 logits (what an acoustic model's projection typically emits), read by the kernels as
 * they are. dtype: 0 = IEEE half, 1 = bfloat16. scratch_dev is ignored (kept for ABI stability). */
int ctcx_decode_half(const void* logits_dev, int dtype, float* scratch_dev, int T, int B, int C,
                     const int32_t* seq_len_dev, int W, int P, int merge_repeated, int blank_index,
                     int blank_label, void* workspace, size_t workspace_bytes, void* stream_v,
                     ctcx_sizes* sizes, int32_t* flags_out) {
  (void)scratch_dev;
  if (dtype != 0 && dtype != 1) return (T == 0) ? CTCX_ERR_MAX_TIME_ZERO : CTCX_ERR_BAD_ARGUMENT;
  DecodeOpts opt;
  opt.in_dtype = (dtype == 0) ? ctcx::kInF16 : ctcx::kInBF16;
  return DecodeImpl<float>(logits_dev, T, B, C, seq_len_dev, W, P, merge_repeated, blank_index, blank_label,
                           workspace, workspace_bytes, stream_v, sizes, flags_out, opt);
}

size_t ctcx_hostin_staging_bytes(int dtype, int T, int B, int C) {
  if (T <= 0 || B < 0 || C <= 0) return 0;
  return (size_t)T * B * C * ElemBytes(dtype);
}

/* Host logits in, decode result left in the workspace: the copy to the device runs in time slabs on
 * `copy_stream` WHILE the beam kernel already consumes the first frames (narrow fast path); other
 * shapes wait for the copy. */
int ctcx_decode_hostin(const void* logits_host, int dtype, int64_t host_time_stride, int T, int B, int C,
                       const int32_t* seq_len_host, int W, int P, int merge_repeated, int blank_index,
                       int blank_label, void* staging_dev, size_t staging_bytes, void* workspace,
                       size_t workspace_bytes, void* stream_v, void* copy_stream_v, ctcx_sizes* sizes,
                       int32_t* flags_out) {
  cudaStream_t stream = (cudaStream_t)stream_v, copy_stream = (cudaStream_t)copy_stream_v;
  const size_t es = ElemBytes(dtype);
  if (T == 0) return CTCX_ERR_MAX_TIME_ZERO;
  if (es == 0 || T < 0 || B < 0 || C <= 0 || W < 1 || P < 1 || blank_index < 0 || blank_index >= C)
    return CTCX_ERR_BAD_ARGUMENT;
  if (W > kMaxBeamWidth || C > kMaxClasses) return CTCX_ERR_UNSUPPORTED;
  const long long hstride = host_time_stride ? host_time_stride : (long long)B * C;
  if (hstride < (long long)B * C) return CTCX_ERR_BAD_ARGUMENT;
  Workspace ws;
  ws.Init(T, B, C, W, P);
  if (workspace == nullptr || workspace_bytes < ws.bytes || ((uintptr_t)workspace & 255u))
    return CTCX_ERR_WORKSPACE;
  if (B > 0 && (staging_dev == nullptr || staging_bytes < (size_t)T * B * C * es || logits_host == nullptr ||
                seq_len_host == nullptr))
    return CTCX_ERR_BAD_ARGUMENT;
  if (copy_stream == stream) return CTCX_ERR_BAD_ARGUMENT;  // the kernel would wait for a copy queued behind it
  unsigned char* base = (unsigned char*)workspace;
  int* d_ctrl = (int*)(base + ws.ctrl);
  int32_t* d_seq = (int32_t*)(base + ws.seq);

  // overlap needs a truly asynchronous copy (page-locked source) and the stream-ordered flag store;
  // pageable sources are staged by the driver, which may wait for the kernel that waits for them
  const bool overlap = (B > 0) && PathOf<float>(W, C, false) == kPathNarrow && P <= W &&
                       IsPinned(logits_host) && StreamWriteValue32() != nullptr;
  Feed feed = {(const unsigned char*)logits_host, (unsigned char*)staging_dev, (size_t)B * C * es,
               (size_t)hstride * es, T, d_ctrl + 1, overlap, copy_stream};
  cudaEvent_t ev = nullptr;
  int rc = CTCX_OK;
  DecodeOpts opt;
  opt.in_dtype = InDtypeOf(dtype);
  // wide vocabularies: the copy is the longer leg; the decode follows it slab by slab (events, no polling)
  constexpr int kMaxSlabs = 8, kMinSlabFrames = 16;
  int slab_end[kMaxSlabs];
  cudaEvent_t slab_event[kMaxSlabs] = {};
  int n_slabs = 0;
  if (B > 0 && dtype != CTCX_F64 && PathOf<float>(W, C, false) == kPathWide && P <= W && IsPinned(logits_host) &&
      T >= 2 * kMinSlabFrames) {
    n_slabs = std::min(kMaxSlabs, T / kMinSlabFrames);
    for (int k = 0; k < n_slabs; ++k) slab_end[k] = (int)(((long long)T * (k + 1)) / n_slabs);
    for (int k = 0; k < n_slabs && rc == CTCX_OK; ++k)
      if (!Check(cudaEventCreateWithFlags(&slab_event[k], cudaEventDisableTiming), "cudaEventCreate")) rc = CTCX_ERR_CUDA;
    if (rc != CTCX_OK) {
      for (int k = 0; k < n_slabs; ++k)
        if (slab_event[k]) cudaEventDestroy(slab_event[k]);
      return rc;
    }
    feed.n_slabs = opt.n_slabs = n_slabs;
    feed.slab_end = opt.slab_end = slab_end;
    feed.slab_event = opt.slab_event = slab_event;
  }
  if (B > 0) {
    CTCX_CUDA(cudaMemcpyAsync(d_seq, seq_len_host, (size_t)B * 4, cudaMemcpyHostToDevice, stream));
    CTCX_CUDA(cudaEventCreateWithFlags(&ev, cudaEventDisableTiming));
    if (overlap) {
      // frames landed = 0, then the copy stream may start once everything queued on `stream` so far
      // (earlier users of the staging memory included) is done
      CTCX_CUDA(cudaMemsetAsync(d_ctrl + 1, 0, 4, stream));
      CTCX_CUDA(cudaEventRecord(ev, stream));
      CTCX_CUDA(cudaStreamWaitEvent(copy_stream, ev, 0));
      opt.ready = d_ctrl + 1;
      // The slab copies (page-locked source: the calls only enqueue) go out BEFORE the kernels: whatever
      // serialises launches -- a profiler, CUDA_LAUNCH_BLOCKING -- then finds the data already landed
      // instead of a kernel waiting for copies its own launch is holding back.
      rc = RunFeed(&feed);
    } else {
      // copy first (on the copy stream, so that it can still overlap other work of the caller), then decode
      // (wide path: slab by slab -- the decode waits for each slab's own event as well)
      CTCX_CUDA(cudaEventRecord(ev, stream));
      CTCX_CUDA(cudaStreamWaitEvent(copy_stream, ev, 0));
      rc = RunFeed(&feed);
      if (rc == CTCX_OK && n_slabs == 0) {
        if (!Check(cudaEventRecord(ev, copy_stream), "cudaEventRecord") ||
            !Check(cudaStreamWaitEvent(stream, ev, 0), "cudaStreamWaitEvent"))
          rc = CTCX_ERR_CUDA;
      }
    }
  }
  if (rc == CTCX_OK) {
    if (dtype == CTCX_F64)
      rc = DecodeImpl<double>(staging_dev, T, B, C, d_seq, W, P, merge_repeated, blank_index, blank_label, workspace,
                              workspace_bytes, stream_v, sizes, flags_out, opt);
    else
      rc = DecodeImpl<float>(staging_dev, T, B, C, d_seq, W, P, merge_repeated, blank_index, blank_label, workspace,
                             workspace_bytes, stream_v, sizes, flags_out, opt);
  }
  if (ev != nullptr) {
    if (rc != CTCX_OK) cudaStreamSynchronize(copy_stream);  // nothing of this call stays in flight after an error
    cudaEventDestroy(ev);
  }
  for (int k = 0; k < n_slabs; ++k) cudaEventDestroy(slab_event[k]);  // (deferred by the runtime until they have fired)
  return rc;
}

int ctcx_pack_f32(const void* workspace, int T, int B, int P, int64_t* const* decoded_indices,
                  int64_t* const* decoded_values, int64_t* const* decoded_shape,
                  int64_t* const* alignment_indices, int64_t* const* alignment_values,
                  int64_t* const* alignment_shape, float* log_probability, void* stream_v) {
  return PackImpl(workspace, T, B, P, decoded_indices, decoded_values, decoded_shape, alignment_indices,
                  alignment_values, alignment_shape, log_probability, 4, stream_v);
}

/* Compact pack: every output of the decode into ONE caller buffer, laid out on the device (see
 * PackTableKernel), enqueued without knowing the sizes on the host. */
int ctcx_pack_compact(void* workspace, int T, int B, int P, int real_bytes, int64_t* packed_dev,
                      size_t packed_elems, void* stream_v) {
  cudaStream_t stream = (cudaStream_t)stream_v;
  if (workspace == nullptr || T <= 0 || B < 1 || P < 1 || ((uintptr_t)workspace & 255u)) return CTCX_ERR_WORKSPACE;
  if (packed_dev == nullptr || (real_bytes != 4 && real_bytes != 8)) return CTCX_ERR_BAD_ARGUMENT;
  unsigned char* base = (unsigned char*)workspace;
  Workspace ws;
  ws.InitPack(T, B, P);
  int* overflow = (int*)(base + ws.stats) + 6;
  CTCX_LAUNCH(ctcx::LaunchPackTable((const long long*)(base + ws.result), B, P, real_bytes, (long long*)packed_dev,
                                    (unsigned long long)packed_elems, (long long**)(base + ws.ptrs), overflow, stream));
  return Pack(ws, base, T, B, P, nullptr, overflow, real_bytes, stream);
}

/* Completes a decode that was enqueued with sizes == NULL: one device->host copy of the sizes and the
 * status words, one synchronisation of `stream`, the reference's error checks. */
int ctcx_finish(const void* workspace, int T, int B, int P, void* stream_v, ctcx_sizes* sizes, int32_t* flags_out) {
  if (workspace == nullptr || sizes == nullptr || T <= 0 || B < 0 || P < 1 || ((uintptr_t)workspace & 255u))
    return CTCX_ERR_WORKSPACE;
  Workspace ws;
  ws.InitPack(T, B, P);
  return FinishImpl((const unsigned char*)workspace + ws.result, T, B, P, (cudaStream_t)stream_v, sizes, flags_out);
}

/* The two halves of ctcx_finish for callers that keep several decodes in flight on one stream: enqueue the
 * copy of the result block into (page-locked) host memory right behind the decode, wait for an event of
 * their own recorded there, then parse the block on the host. */
size_t ctcx_result_bytes(int top_paths) { return top_paths > 0 ? ResultBytes(top_paths) : 0; }

int ctcx_result_copy_async(const void* workspace, int T, int B, int P, void* result_host, size_t result_bytes,
                           void* stream_v) {
  if (workspace == nullptr || T <= 0 || B < 0 || P < 1 || ((uintptr_t)workspace & 255u)) return CTCX_ERR_WORKSPACE;
  if (result_host == nullptr || result_bytes < ResultBytes(P)) return CTCX_ERR_BAD_ARGUMENT;
  Workspace ws;
  ws.InitPack(T, B, P);
  CTCX_CUDA(cudaMemcpyAsync(result_host, (const unsigned char*)workspace + ws.result, ResultBytes(P),
                            cudaMemcpyDeviceToHost, (cudaStream_t)stream_v));
  return CTCX_OK;
}

int ctcx_result_parse(const void* result_host, int T, int B, int P, ctcx_sizes* sizes, int32_t* flags_out) {
  if (result_host == nullptr || sizes == nullptr || T <= 0 || B < 0 || P < 1) return CTCX_ERR_BAD_ARGUMENT;
  CollectProfile(B);
  return ParseResult((const unsigned char*)result_host, T, B, P, sizes, flags_out);
}

int ctcx_pack_f64(const void* workspace, int T, int B, int P, int64_t* const* decoded_indices,
                  int64_t* const* decoded_values, int64_t* const* decoded_shape,
                  int64_t* const* alignment_indices, int64_t* const* alignment_values,
                  int64_t* const* alignment_shape, double* log_probability, void* stream_v) {
  return PackImpl(workspace, T, B, P, decoded_indices, decoded_values, decoded_shape, alignment_indices,
                  alignment_values, alignment_shape, log_probability, 8, stream_v);
}

int ctcx_workspace_views(const void* workspace, int T, int B, int P, const int32_t** dec_len,
                         const int32_t** dec, const int32_t** ali_len, const int32_t** ali,
                         const float** logp) {
  if (workspace == nullptr) return CTCX_ERR_WORKSPACE;
  const unsigned char* base = (const unsigned char*)workspace;
  Workspace::Header hdr;
  CTCX_CUDA(cudaMemcpy(&hdr, base, sizeof(hdr), cudaMemcpyDeviceToHost));
  if (hdr.magic != kMagic || hdr.T != T || hdr.B != B || hdr.P != P) return CTCX_ERR_WORKSPACE;
  if (logp != nullptr && hdr.real_bytes != 4) return CTCX_ERR_BAD_ARGUMENT;  // float32 decodes only
  Workspace ws;
  ws.InitPack(T, B, P);
  if (dec_len) *dec_len = (const int32_t*)(base + ws.dec_len);
  if (dec) *dec = (const int32_t*)(base + ws.dec);
  if (ali_len) *ali_len = (const int32_t*)(base + ws.ali_len);
  if (ali) *ali = (const int32_t*)(base + ws.ali);
  if (logp) *logp = (const float*)(base + ws.fin_total);
  return CTCX_OK;
}

void ctcx_free_host(ctcx_host_result* r) {
  if (!r) return;
  auto free_list = [&](int64_t** l) {
    if (!l) return;
    for (int p = 0; p < r->top_paths; ++p) std::free(l[p]);
    std::free(l);
  };
  free_list(r->decoded_indices);
  free_list(r->decoded_values);
  free_list(r->decoded_shape);
  free_list(r->alignment_indices);
  free_list(r->alignment_values);
  free_list(r->alignment_shape);
  std::free(r->n_decoded);
  std::free(r->n_alignment);
  std::free(r->log_probability);
  std::free(r->log_probability_f64);
  std::free(r);
}

static int DecodeHostImpl(const void* logits_host, int dtype, int T, int B, int C, const int32_t* seq_len_host,
                          int W, int P, int merge_repeated, int blank_index, int blank_label,
                          int device, ctcx_host_result** result) {
  if (result == nullptr) return CTCX_ERR_BAD_ARGUMENT;
  *result = nullptr;
  if (T == 0) return CTCX_ERR_MAX_TIME_ZERO;
  if (T < 0 || B < 0 || C <= 0 || W < 1 || P < 1) return CTCX_ERR_BAD_ARGUMENT;
  const int rb = (dtype == CTCX_F64) ? 8 : 4;
  CTCX_CUDA(cudaSetDevice(device));
  cudaStream_t stream = nullptr, copy_stream = nullptr;
  const size_t staging_bytes = ctcx_hostin_staging_bytes(dtype, T, B, C);
  const size_t ws_bytes = ctcx_workspace_bytes(T, B, C, W, P);
  void* d_logits = nullptr;
  void* d_ws = nullptr;
  unsigned char* d_out = nullptr;
  int rc = CTCX_OK;
  std::vector<int64_t> n_dec(P), max_dec(P), n_ali(P), max_ali(P);
  ctcx_sizes sizes = {n_dec.data(), max_dec.data(), n_ali.data(), max_ali.data()};
  int32_t flags = 0;
  ctcx_host_result* r = nullptr;
  std::vector<int64_t*> p_di(P), p_dv(P), p_ds(P), p_ai(P), p_av(P), p_as(P);
  size_t out_bytes = 0;
#define CTCX_TRY(call)                                        \
  do {                                                        \
    if (!Check((call), #call)) { rc = CTCX_ERR_CUDA; goto done; } \
  } while (0)
  CTCX_TRY(cudaStreamCreateWithFlags(&stream, cudaStreamNonBlocking));
  CTCX_TRY(cudaStreamCreateWithFlags(&copy_stream, cudaStreamNonBlocking));
  CTCX_TRY(cudaMalloc(&d_logits, staging_bytes + 8));
  CTCX_TRY(cudaMalloc(&d_ws, ws_bytes));
  rc = ctcx_decode_hostin(logits_host, dtype, 0, T, B, C, seq_len_host, W, P, merge_repeated, blank_index,
                          blank_label, d_logits, staging_bytes + 8, d_ws, ws_bytes, stream, copy_stream, &sizes,
                          &flags);
  if (rc != CTCX_OK) goto done;
  {
    // one device block for all outputs, then one D2H copy
    size_t o = 0;
    auto take = [&](size_t n64) { size_t at = o; o += Align256(n64 * 8); return at; };
    std::vector<size_t> o_di(P), o_dv(P), o_ds(P), o_ai(P), o_av(P), o_as(P);
    for (int p = 0; p < P; ++p) {
      o_di[p] = take((size_t)n_dec[p] * 2); o_dv[p] = take((size_t)n_dec[p]); o_ds[p] = take(2);
      o_ai[p] = take((size_t)n_ali[p] * 2); o_av[p] = take((size_t)n_ali[p]); o_as[p] = take(2);
    }
    const size_t o_lp = o;
    o += Align256((size_t)B * P * rb);
    out_bytes = o;
    CTCX_TRY(cudaMalloc(&d_out, out_bytes + 256));
    for (int p = 0; p < P; ++p) {
      p_di[p] = (int64_t*)(d_out + o_di[p]); p_dv[p] = (int64_t*)(d_out + o_dv[p]); p_ds[p] = (int64_t*)(d_out + o_ds[p]);
      p_ai[p] = (int64_t*)(d_out + o_ai[p]); p_av[p] = (int64_t*)(d_out + o_av[p]); p_as[p] = (int64_t*)(d_out + o_as[p]);
    }
    rc = (rb == 8) ? ctcx_pack_f64(d_ws, T, B, P, p_di.data(), p_dv.data(), p_ds.data(), p_ai.data(), p_av.data(),
                                   p_as.data(), (double*)(d_out + o_lp), stream)
                   : ctcx_pack_f32(d_ws, T, B, P, p_di.data(), p_dv.data(), p_ds.data(), p_ai.data(), p_av.data(),
                                   p_as.data(), (float*)(d_out + o_lp), stream);
    if (rc != CTCX_OK) goto done;
    std::vector<unsigned char> h_out(out_bytes);
    CTCX_TRY(cudaMemcpyAsync(h_out.data(), d_out, out_bytes, cudaMemcpyDeviceToHost, stream));
    CTCX_TRY(cudaStreamSynchronize(stream));
    r = (ctcx_host_result*)std::calloc(1, sizeof(ctcx_host_result));
    r->top_paths = P;
    r->flags = flags;
    r->n_decoded = (int64_t*)std::malloc(sizeof(int64_t) * P);
    r->n_alignment = (int64_t*)std::malloc(sizeof(int64_t) * P);
    auto mk = [&]() { return (int64_t**)std::calloc((size_t)P, sizeof(int64_t*)); };
    r->decoded_indices = mk(); r->decoded_values = mk(); r->decoded_shape = mk();
    r->alignment_indices = mk(); r->alignment_values = mk(); r->alignment_shape = mk();
    auto dup = [&](size_t at, size_t n64) {
      int64_t* m = (int64_t*)std::malloc(n64 * 8 + 8);
      std::memcpy(m, h_out.data() + at, n64 * 8);
      return m;
    };
    for (int p = 0; p < P; ++p) {
      r->n_decoded[p] = n_dec[p];
      r->n_alignment[p] = n_ali[p];
      r->decoded_indices[p] = dup(o_di[p], (size_t)n_dec[p] * 2);
      r->decoded_values[p] = dup(o_dv[p], (size_t)n_dec[p]);
      r->decoded_shape[p] = dup(o_ds[p], 2);
      r->alignment_indices[p] = dup(o_ai[p], (size_t)n_ali[p] * 2);
      r->alignment_values[p] = dup(o_av[p], (size_t)n_ali[p]);
      r->alignment_shape[p] = dup(o_as[p], 2);
    }
    void* lp = std::malloc((size_t)B * P * rb + 8);
    std::memcpy(lp, h_out.data() + o_lp, (size_t)B * P * rb);
    if (rb == 8) r->log_probability_f64 = (double*)lp; else r->log_probability = (float*)lp;
    *result = r;
  }
done:
#undef CTCX_TRY
  if (stream) cudaStreamSynchronize(stream);
  if (copy_stream) cudaStreamSynchronize(copy_stream);
  cudaFree(d_logits);
  cudaFree(d_ws);
  cudaFree(d_out);
  if (stream) cudaStreamDestroy(stream);
  if (copy_stream) cudaStreamDestroy(copy_stream);
  return rc;
}

int ctcx_decode_host_f32(const float* logits_host, int T, int B, int C, const int32_t* seq_len_host,
                         int W, int P, int merge_repeated, int blank_index, int blank_label,
                         int device, ctcx_host_result** result) {
  return DecodeHostImpl(logits_host, CTCX_F32, T, B, C, seq_len_host, W, P, merge_repeated, blank_index, blank_label,
                        device, result);
}

int ctcx_decode_host_f64(const double* logits_host, int T, int B, int C, const int32_t* seq_len_host,
                         int W, int P, int merge_repeated, int blank_index, int blank_label,
                         int device, ctcx_host_result** result) {
  return DecodeHostImpl(logits_host, CTCX_F64, T, B, C, seq_len_host, W, P, merge_repeated, blank_index, blank_label,
                        device, result);
}

/* ---- streaming: Step / TopPaths / Reset of the reference decoder (decoder.h:39-53) ---- */

size_t ctcx_stream_workspace_bytes(int max_time_total, int B, int C, int W, int P) {
  return ctcx_workspace_bytes(max_time_total, B, C, W, P);
}

size_t ctcx_stream_workspace_bytes_v(int score_dtype, int max_time_total, int B, int C, int W, int P) {
  if (score_dtype != CTCX_F32 && score_dtype != CTCX_F64) return 0;
  if (max_time_total <= 0 || B < 0 || C <= 0 || W <= 0 || P <= 0) return 0;
  Workspace ws;
  ws.Init(max_time_total, B, C, W, P, (int)ElemBytes(score_dtype));
  return ws.bytes;
}

int ctcx_stream_reset_v(void* workspace, size_t workspace_bytes, int score_dtype, int T_total, int B, int C, int W,
                        int P, void* stream_v) {
  cudaStream_t stream = (cudaStream_t)stream_v;
  Workspace ws;
  CTCX_RC(CheckStreamReset(workspace, workspace_bytes, score_dtype, T_total, B, C, W, P, &ws));
  const int score_bytes = (int)ElemBytes(score_dtype);
  unsigned char* base = (unsigned char*)workspace;
  Workspace::Header hdr = {kMagic, T_total, B, C, W, P, score_bytes};
  InitBlock init(ws, hdr, B);  // (zeroes the control words: no table with a positive entry yet)
  CTCX_CUDA(cudaMemcpyAsync(base, init.bytes.data(), ws.dec_len, cudaMemcpyHostToDevice, stream));
  if (B > 0) {
    // decoder.h:212-227: with zero frames consumed the kernels start from the root; TopPaths before
    // the first Step() sees the root itself: one leaf, log-probability 0 (ln 1), empty sequences
    CTCX_CUDA(cudaMemsetAsync(base + ws.t_done, 0, (size_t)B * 4, stream));
    CTCX_LAUNCH(ctcx::LaunchStreamReset(base + ws.state, B, W, score_bytes, stream));
    CTCX_CUDA(cudaMemsetAsync(base + ws.fin_total, 0, (size_t)B * P * 8, stream));
    CTCX_CUDA(cudaMemsetAsync(base + ws.fin_kind, 0, (size_t)B * P * 4, stream));
    std::vector<int> ones((size_t)B, 1), fl((size_t)B, (P > 1) ? 2 : 0);  // fewer leaves than top_paths
    CTCX_CUDA(cudaMemcpyAsync(base + ws.fin_n, ones.data(), (size_t)B * 4, cudaMemcpyHostToDevice, stream));
    CTCX_CUDA(cudaMemcpyAsync(base + ws.flags, fl.data(), (size_t)B * 4, cudaMemcpyHostToDevice, stream));
  }
  return CTCX_OK;  // (copies from pageable memory are staged before the calls return)
}

int ctcx_stream_reset_slots(void* workspace, size_t workspace_bytes, int score_dtype, int T_total, int B, int C,
                            int W, int P, const int32_t* slot_mask_dev, void* stream_v) {
  Workspace ws;
  CTCX_RC(CheckStreamReset(workspace, workspace_bytes, score_dtype, T_total, B, C, W, P, &ws));
  if (slot_mask_dev == nullptr) return CTCX_ERR_BAD_ARGUMENT;
  if (B == 0) return CTCX_OK;
  unsigned char* base = (unsigned char*)workspace;
  ctcx::StreamSlotsParams sp;
  sp.state = base + ws.state;
  sp.mask = slot_mask_dev;
  sp.t_done = (int*)(base + ws.t_done);
  sp.fin_total = base + ws.fin_total;
  sp.fin_kind = (int*)(base + ws.fin_kind);
  sp.fin_n = (int*)(base + ws.fin_n);
  sp.flags = (int*)(base + ws.flags);
  sp.B = B; sp.W = W; sp.P = P;
  sp.score_bytes = (int)ElemBytes(score_dtype);
  CTCX_LAUNCH(ctcx::LaunchStreamResetSlots(sp, (cudaStream_t)stream_v));
  return CTCX_OK;
}

int ctcx_stream_reset(void* workspace, size_t workspace_bytes, int T_total, int B, int C, int W, int P,
                      void* stream_v) {
  return ctcx_stream_reset_v(workspace, workspace_bytes, CTCX_F32, T_total, B, C, W, P, stream_v);
}

int ctcx_stream_step_v(void* workspace, size_t workspace_bytes, int T_total, int B, int C, int W, int P,
                       const void* logits_dev, int dtype, int64_t time_stride, int chunk_time,
                       const int32_t* chunk_len_dev, int blank_index, const float* expansion_scores_dev,
                       void* stream_v) {
  cudaStream_t stream = (cudaStream_t)stream_v;
  if (workspace == nullptr || ((uintptr_t)workspace & 255u)) return CTCX_ERR_WORKSPACE;
  if (ElemBytes(dtype) == 0 || time_stride < 0) return CTCX_ERR_BAD_ARGUMENT;
  if (T_total <= 0 || B < 0 || C <= 0 || W < 1 || P < 1 || W > kMaxBeamWidth || C > kMaxClasses || P > W ||
      chunk_time <= 0 || chunk_time > T_total || chunk_len_dev == nullptr || blank_index < 0 || blank_index >= C)
    return CTCX_ERR_BAD_ARGUMENT;
  const long long tstride = time_stride ? time_stride : (long long)B * C;
  if (tstride < (long long)B * C) return CTCX_ERR_BAD_ARGUMENT;
  const bool f64 = (dtype == CTCX_F64);
  if (f64 && expansion_scores_dev != nullptr) return CTCX_ERR_BAD_ARGUMENT;  // tables hold float32 scores
  Workspace ws;
  ws.Init(T_total, B, C, W, P, f64 ? 8 : 4);
  if (workspace_bytes < ws.bytes) return CTCX_ERR_WORKSPACE;
  if (B == 0) return CTCX_OK;
  unsigned char* base = (unsigned char*)workspace;
  int* d_ctrl = (int*)(base + ws.ctrl);
  // a table with a positive entry: sticky until the next reset, reported by ctcx_stream_top_paths
  if (expansion_scores_dev != nullptr)
    CTCX_LAUNCH(ctcx::LaunchPositive(expansion_scores_dev, (long long)(C + 1) * C, d_ctrl + kCtrlTablePositive, stream));
  const Logits x = {logits_dev, InDtypeOf(dtype), tstride};
  return f64 ? StreamStep<double>(ws, base, T_total, B, C, W, P, x, chunk_time, chunk_len_dev, blank_index, nullptr,
                                  stream)
             : StreamStep<float>(ws, base, T_total, B, C, W, P, x, chunk_time, chunk_len_dev, blank_index,
                                 expansion_scores_dev, stream);
}

int ctcx_stream_step_f32(void* workspace, int T_total, int B, int C, int W, int P, const float* logits_dev,
                         int chunk_time, const int32_t* chunk_len_dev, int blank_index, void* stream_v) {
  // (no size argument: the workspace is taken to be the float stream's)
  return ctcx_stream_step_v(workspace, ctcx_stream_workspace_bytes(T_total, B, C, W, P), T_total, B, C, W, P,
                            logits_dev, CTCX_F32, 0, chunk_time, chunk_len_dev, blank_index, nullptr, stream_v);
}

int ctcx_stream_top_paths(void* workspace, int T_total, int B, int C, int W, int P, int merge_repeated,
                          int blank_label, void* stream_v, ctcx_sizes* sizes, int32_t* flags_out) {
  if (workspace == nullptr || sizes == nullptr || ((uintptr_t)workspace & 255u)) return CTCX_ERR_WORKSPACE;
  if (T_total <= 0 || B < 0 || C <= 0 || W < 1 || P < 1 || W > kMaxBeamWidth || C > kMaxClasses)
    return CTCX_ERR_BAD_ARGUMENT;
  return StreamTopPaths(workspace, T_total, B, C, W, P, merge_repeated, blank_label, nullptr, (cudaStream_t)stream_v,
                        sizes, flags_out);
}

int ctcx_stream_top_paths_slots(void* workspace, int T_total, int B, int C, int W, int P, int merge_repeated,
                                int blank_label, const int32_t* slot_mask_dev, void* stream_v, ctcx_sizes* sizes,
                                int32_t* flags_out) {
  if (workspace == nullptr || ((uintptr_t)workspace & 255u)) return CTCX_ERR_WORKSPACE;
  if (T_total <= 0 || B < 0 || C <= 0 || W < 1 || P < 1 || W > kMaxBeamWidth || C > kMaxClasses)
    return CTCX_ERR_BAD_ARGUMENT;
  if (P > W) return CTCX_ERR_TOO_MANY_PATHS;
  if (slot_mask_dev == nullptr) return CTCX_ERR_BAD_ARGUMENT;
  return StreamTopPaths(workspace, T_total, B, C, W, P, merge_repeated, blank_label, slot_mask_dev,
                        (cudaStream_t)stream_v, sizes, flags_out);
}

/* ---- measurement and test hooks (declared at the end of include/ctcx.h) ---- */

/* per-kernel device times of this thread's last decode, from CUDA events recorded on the launching
 * stream. out_ms = {pre-pass, beam, trace, scan + flags, total}. */
void ctcx_profile_enable(int on) { g_profile = on; }
void ctcx_profile_get(float* out_ms) {
  for (int k = 0; k < 5; ++k) out_ms[k] = g_ms[k];
}

/* device buffer [B,24] int64 receiving per-phase clock64 cycles of the fast beam kernels (thread 0
 * of every CTA, summed over frames) for this thread's decodes; NULL switches it off. */
void ctcx_debug_set_cycles_buffer(long long* dev_buf) { ctcx_debug_set_cycles_buffer_n(dev_buf, 24); }

/* the same with [B,slots] rows (slots >= 24; smaller values count as 24): the narrow kernel also
 * fills its revisit-wipe event counters 24-26 where the row has room for them. */
void ctcx_debug_set_cycles_buffer_n(long long* dev_buf, int slots) {
  g_dbg_cycles = dev_buf;
  g_dbg_slots = slots > 24 ? slots : 24;
}

/* 0 = dispatch by shape (default); 1 = route every decode of the process to the generic beam kernel,
 * the independent second implementation the parity tests compare with the fast ones. */
void ctcx_debug_set_beam_impl(int impl) { g_force_generic.store(impl == 1 ? 1 : 0); }

/* The normaliser pre-pass of a decode on its own: the decode's own PrePass, route 0 as the generic path
 * runs it (LaunchLogNorm; half inputs upcast first), route 1 as the wide path does (the fused normaliser
 * and sorted-class list, LaunchNormTopClasses). */
int ctcx_debug_prepass(int route, const void* logits_dev, int in_dtype, int T, int B, int C, long long tstride,
                       int blank_index, int beam_width, void* off_dev, float* srt_pl_dev, uint16_t* srt_cls_dev,
                       int* ks_out, void* stream_v) {
  cudaStream_t stream = (cudaStream_t)stream_v;
  if (tstride == 0) tstride = (long long)B * C;
  if (T < 1 || B < 1 || C < 1 || C > kMaxClasses || blank_index < 0 || blank_index >= C ||
      tstride < (long long)B * C || ElemBytes(in_dtype) == 0 || logits_dev == nullptr || off_dev == nullptr)
    return CTCX_ERR_BAD_ARGUMENT;
  Logits x = {logits_dev, InDtypeOf(in_dtype), tstride};
  if (route == 0) {
    if (ks_out) *ks_out = 0;
    if (in_dtype == CTCX_F64)
      return PrePass<double>(kPathGeneric, x, T, B, C, blank_index, beam_width, (double*)off_dev, nullptr, nullptr,
                             nullptr, stream);
    // half inputs are widened into scratch of the hook's own (a decode has it in its workspace)
    const bool half = (in_dtype != CTCX_F32);
    float* scratch = nullptr;
    if (half) CTCX_CUDA(cudaMallocAsync((void**)&scratch, (size_t)T * B * C * sizeof(float), stream));
    int rc = PrePass<float>(kPathGeneric, x, T, B, C, blank_index, beam_width, (float*)off_dev, nullptr, nullptr,
                            scratch, stream);
    if (half && !Check(cudaFreeAsync(scratch, stream), "cudaFreeAsync") && rc == CTCX_OK) rc = CTCX_ERR_CUDA;
    return rc;
  }
  if (route != 1) return CTCX_ERR_BAD_ARGUMENT;
  if (in_dtype == CTCX_F64 || beam_width < 1 || !ctcx::WideFastShape(beam_width, C)) return CTCX_ERR_UNSUPPORTED;
  if (srt_pl_dev == nullptr || srt_cls_dev == nullptr) return CTCX_ERR_BAD_ARGUMENT;
  if (ks_out) *ks_out = ctcx::WideKs(beam_width, C);
  return PrePass<float>(kPathWide, x, T, B, C, blank_index, beam_width, (float*)off_dev, srt_pl_dev,
                        (unsigned short*)srt_cls_dev, nullptr, stream);
}

/* y = f(x) element-wise with the exact device math; op 0 expf, 1 log1pf, 2 logf, 3 LogSumExp(x, 0),
 * 4 LogSumExp(0, x) */
int ctcx_debug_math_f32(int op, const float* x_dev, float* y_dev, int n, void* stream_v) {
  if (n <= 0) return CTCX_OK;
  CTCX_LAUNCH(ctcx::LaunchMathTest(op, x_dev, y_dev, n, (cudaStream_t)stream_v));
  return CTCX_OK;
}

/* the double-precision twin: op 0 exp (x <= 0), 1 log (x >= 1), 2 LogSumExp(x, 0) */
int ctcx_debug_math_f64(int op, const double* x_dev, double* y_dev, int n, void* stream_v) {
  if (n <= 0) return CTCX_OK;
  CTCX_LAUNCH(ctcx::LaunchMathTest(op, x_dev, y_dev, n, (cudaStream_t)stream_v));
  return CTCX_OK;
}

}  // extern "C"
