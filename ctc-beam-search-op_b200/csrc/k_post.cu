// Translation unit of the kernels after the beam search: trace-back of the top paths, prefix sums of
// the sparse sizes, reduction of the per-utterance flags, sparse packing; plus the math test hooks.
#include "ctcx_kernels.cuh"
#include "ctcx_launch.h"

#include <algorithm>
#include <cstdint>

namespace ctcx {

// ---------------------------------------------------------------------------------------------
// Kernel 3: trace-back. One thread per (utterance, path) walks the back-pointer records from the
// last frame to the first, emitting the alignment (entry.h:137-152) and the decoded labels
// (entry.h:123-136, with optional repeat merging).
// ---------------------------------------------------------------------------------------------
// Back-pointer record formats: the generic / wide kernels write 8-byte records {packed word, label}
// (PackRec), the narrow fast kernel 4-byte ones (PackRec32, ctcx_beam_v4.cuh).
struct RecFields {
  unsigned prev_self, an_src, ab_kind, an_kind;
  int label;
};
__device__ __forceinline__ RecFields UnpackRec(const uint2 r) {
  return {r.x & 0x7ffu, (r.x >> 11) & 0x7ffu, (r.x >> 22) & 1u, (r.x >> 23) & 3u, (int)r.y};
}
__device__ __forceinline__ RecFields UnpackRec(const unsigned r) {
  return {r & 0xffu, (r >> 8) & 0xffu, (r >> 16) & 1u, (r >> 17) & 3u, (int)(r >> 24)};
}


// The trace kernels take their record type as TAG: REC itself, or Masked<REC> for the form that walks
// only the utterances TraceParams::mask selects (the others get lengths 0 and load nothing else). The
// one-shot decodes' instantiations thereby keep both their code and their names.
template <typename REC>
struct Masked {};
template <typename TAG>
struct TraceTag {
  using Rec = TAG;
  static constexpr bool kMasked = false;
};
template <typename REC>
struct TraceTag<Masked<REC>> {
  using Rec = REC;
  static constexpr bool kMasked = true;
};

template <typename TAG>
__global__ void __launch_bounds__(128) TraceKernel(TraceParams p) {
  using REC = typename TraceTag<TAG>::Rec;
  const int idx = blockIdx.x * blockDim.x + threadIdx.x;
  if (idx >= p.B * p.P) return;
  const int b = idx / p.P, path = idx - b * p.P;
  if constexpr (TraceTag<TAG>::kMasked) {
    if (p.mask[b] == 0) {
      p.dec_len[idx] = 0;
      p.ali_len[idx] = 0;
      return;
    }
  }
  const int L = max(0, min(p.seq_len[b], p.T));  // out-of-range lengths are reported by the host, not walked
  int* ali = p.ali + (size_t)idx * p.T;
  int* dec = p.dec + (size_t)idx * p.T;
  if (path >= p.fin_n[b] || L <= 0) {
    p.dec_len[idx] = 0;
    p.ali_len[idx] = 0;
    return;
  }
  int slot = path;
  int kind_ab = p.fin_kind[idx];
  const REC* bp = reinterpret_cast<const REC*>(p.bp) + (size_t)b * p.T * p.W;
  for (int t = L - 1; t >= 0; --t) {
    const RecFields r = UnpackRec(bp[(size_t)t * p.W + min(slot, p.W - 1)]);
    if (kind_ab) {
      ali[t] = p.blank_label;
      dec[t] = -1;
      kind_ab = (r.ab_kind == kAbFromAb) ? 1 : 0;
      slot = (int)r.prev_self;
    } else {
      ali[t] = r.label;
      if (r.an_kind == kAnSelfAn) {
        dec[t] = -1;
        slot = (int)r.prev_self;
      } else {
        dec[t] = r.label;  // a new label was emitted at this frame
        slot = (int)r.an_src;
        kind_ab = (r.an_kind == kAnParAb) ? 1 : 0;
      }
    }
  }
  int pos = 0, prev = -1;
  for (int t = 0; t < L; ++t) {
    const int v = dec[t];
    if (v >= 0) {
      if (!p.merge_repeated || v != prev) dec[pos++] = v;
      prev = v;
    }
  }
  p.dec_len[idx] = pos;
  p.ali_len[idx] = L;
}

// Warp-cooperative trace-back (used when there are too few walks to hide latency by themselves;
// TraceKernel above is the simple form). One warp per (utterance, path). The walk is a dependent
// chain (the slot at frame t-1 comes out of the record at frame t), but WHICH ROWS are needed next is
// known in advance: the warp streams blocks of `rows` consecutive back-pointer rows [rows x W x 8 B,
// contiguous in memory] into a double buffer in shared memory with cp.async, one block ahead of the
// walk, so a step is one shared-memory broadcast read plus a few ALU operations instead of a
// dependent trip to L2/HBM. Symbols are collected 32 frames at a time in registers and written as
// coalesced rows; the decoded labels are compacted with warp ballots.
// When a row of records is a multiple of 16 bytes (beam 100 with 4-byte records: 400 B) a block of rows is
// ONE contiguous, 16-byte aligned span of HBM: it is fetched by a single bulk-copy instruction
// (cp.async.bulk, the TMA unit's 1-D form) issued by one lane and signalled on an mbarrier, instead
// of one 4-byte cp.async per record (3 200 per block).
template <typename TAG, int WARPS>
__global__ void __launch_bounds__(WARPS * 32) TraceWarpKernel(TraceParams p, int rows_log2, int use_bulk) {
  using REC = typename TraceTag<TAG>::Rec;
  extern __shared__ __align__(16) unsigned char tsm[];
  __shared__ __align__(8) unsigned long long s_mbar[WARPS][2];
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const int idx = blockIdx.x * WARPS + warp;
  if (idx >= p.B * p.P) return;
  const int b = idx / p.P, path = idx - b * p.P;
  if constexpr (TraceTag<TAG>::kMasked) {
    if (p.mask[b] == 0) {
      if (lane == 0) {
        p.dec_len[idx] = 0;
        p.ali_len[idx] = 0;
      }
      return;
    }
  }
  const int L = max(0, min(p.seq_len[b], p.T));  // out-of-range lengths are reported by the host, not walked
  int* ali = p.ali + (size_t)idx * p.T;
  int* dec = p.dec + (size_t)idx * p.T;
  if (path >= p.fin_n[b] || L <= 0) {
    if (lane == 0) {
      p.dec_len[idx] = 0;
      p.ali_len[idx] = 0;
    }
    return;
  }
  const int W = p.W;
  const int R = 1 << rows_log2;
  REC* buf = reinterpret_cast<REC*>(tsm) + (size_t)warp * 2 * R * W;
  const REC* bp = reinterpret_cast<const REC*>(p.bp) + (size_t)b * p.T * W;
  const unsigned mbar0 = (unsigned)__cvta_generic_to_shared(&s_mbar[warp][0]);
  if (use_bulk) {
    if (lane == 0) {
      asm volatile("mbarrier.init.shared::cta.b64 [%0], 1;\n" ::"r"(mbar0));
      asm volatile("mbarrier.init.shared::cta.b64 [%0], 1;\n" ::"r"(mbar0 + 8u));
      asm volatile("fence.mbarrier_init.release.cluster;\n" ::: "memory");
    }
    __syncwarp();
  }
  // block k holds frames [k*R, min(L, (k+1)*R)); blocks are walked from the last one down
  auto fetch_block = [&](int k) {
    if (k >= 0) {
      const int t0 = k << rows_log2;
      const int nrec = (min(L, t0 + R) - t0) * W;
      const REC* src = bp + (size_t)t0 * W;
      const unsigned dst = (unsigned)__cvta_generic_to_shared(buf + (size_t)(k & 1) * R * W);
      if (use_bulk) {
        if (lane == 0) {
          const unsigned bytes = (unsigned)nrec * (unsigned)sizeof(REC);
          const unsigned mbar = mbar0 + 8u * (unsigned)(k & 1);
          // the buffer was last read through ordinary loads (two blocks ago): order them before the
          // asynchronous-proxy write
          asm volatile("fence.proxy.async.shared::cta;\n" ::: "memory");
          asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;\n" ::"r"(mbar), "r"(bytes) : "memory");
          asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];\n" ::"r"(dst),
                       "l"(src), "r"(bytes), "r"(mbar)
                       : "memory");
        }
      } else {
        for (int i = lane; i < nrec; i += 32)
          asm volatile("cp.async.ca.shared.global [%0], [%1], %2;\n" ::"r"(dst + (unsigned)sizeof(REC) * (unsigned)i),
                       "l"(src + i), "n"(sizeof(REC)));
      }
    }
    if (!use_bulk) asm volatile("cp.async.commit_group;\n" ::);
  };
  // wait until block k has landed (bulk path: the k-th use of its buffer flips the barrier's phase)
  const int last_block = (L - 1) >> rows_log2;
  auto wait_block = [&](int k) {
    if (use_bulk) {
      const unsigned mbar = mbar0 + 8u * (unsigned)(k & 1);
      const unsigned parity = (unsigned)(((last_block - k) >> 1) & 1);
      unsigned done = 0;
      while (!done) {
        asm volatile(
            "{\n .reg .pred p;\n mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n selp.u32 %0, 1, 0, p;\n}\n"
            : "=r"(done)
            : "r"(mbar), "r"(parity)
            : "memory");
      }
    } else {
      asm volatile("cp.async.wait_group 1;\n" ::);
    }
  };
  fetch_block(last_block);
  int slot = path;
  int kind_ab = p.fin_kind[idx];
  int a_val = 0, d_val = -1;  // this lane's symbols of the current 32-frame store block
  for (int k = last_block; k >= 0; --k) {
    fetch_block(k - 1);  // next block in flight while this one is walked
    wait_block(k);       // block k has landed
    __syncwarp();
    const REC* blk = buf + (size_t)(k & 1) * R * W;
    const int t_lo = k << rows_log2;
    for (int t = min(L, t_lo + R) - 1; t >= t_lo; --t) {
      const RecFields r = UnpackRec(blk[(t - t_lo) * W + min(slot, W - 1)]);
      int sym_a, sym_d = -1;
      if (kind_ab) {  // entry.h:133-136: a blank frame
        sym_a = p.blank_label;
        kind_ab = (r.ab_kind == kAbFromAb) ? 1 : 0;
        slot = (int)r.prev_self;
      } else {
        sym_a = r.label;
        if (r.an_kind == kAnSelfAn) {
          slot = (int)r.prev_self;
        } else {
          sym_d = r.label;  // a new label was emitted at this frame
          slot = (int)r.an_src;
          kind_ab = (r.an_kind == kAnParAb) ? 1 : 0;
        }
      }
      if (lane == (t & 31)) {
        a_val = sym_a;
        d_val = sym_d;
      }
      if ((t & 31) == 0) {  // frames [t, t+32) complete: coalesced store
        const int tt = t + lane;
        if (tt < L) {
          ali[tt] = a_val;
          dec[tt] = d_val;
        }
      }
    }
    __syncwarp();  // buffer (k & 1) is refilled two iterations from now
  }
  __syncwarp();
  // forward compaction of the new labels (entry.h:123-136, optional repeat merging)
  int base = 0, carry = -1;
  for (int t0 = 0; t0 < L; t0 += 32) {
    const int tt = t0 + lane;
    const int v = (tt < L) ? dec[tt] : -1;
    const unsigned mask = __ballot_sync(kFull, v >= 0);
    const unsigned pm = mask & ((1u << lane) - 1u);
    const int prev_lane = pm ? (31 - __clz(pm)) : 0;
    int prev_val = __shfl_sync(kFull, v, prev_lane);
    if (!pm) prev_val = carry;
    const bool keep = (v >= 0) && (!p.merge_repeated || v != prev_val);
    const unsigned kmask = __ballot_sync(kFull, keep);
    __syncwarp();
    if (keep) dec[base + __popc(kmask & ((1u << lane) - 1u))] = v;
    base += __popc(kmask);
    if (mask) carry = __shfl_sync(kFull, v, 31 - __clz(mask));
  }
  if (lane == 0) {
    p.dec_len[idx] = base;
    p.ali_len[idx] = L;
  }
}

// ---------------------------------------------------------------------------------------------
// Kernels 4/5: sparse packing (kernels.cc:163-257). ScanKernel: per path, exclusive prefix sums of
// the lengths over the batch + totals + maxima. PackKernel: indices [b,pos], values, shapes.
// ---------------------------------------------------------------------------------------------

static __global__ void __launch_bounds__(1024) ScanKernel(ScanParams p) {
  __shared__ long long s_sum[2][32];
  __shared__ int s_max[2][32];
  const int path = blockIdx.x;
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const int per = (p.B + 1023) / 1024;
  const int b0 = min(p.B, tid * per), b1 = min(p.B, b0 + per);
  long long sum[2] = {0, 0};
  int mx[2] = {0, 0};
  for (int b = b0; b < b1; ++b) {
    const int d = p.dec_len[(size_t)b * p.P + path], a = p.ali_len[(size_t)b * p.P + path];
    sum[0] += d; sum[1] += a;
    mx[0] = max(mx[0], d); mx[1] = max(mx[1], a);
  }
  long long incl[2];
#pragma unroll
  for (int w = 0; w < 2; ++w) {
    long long v = sum[w];
    int m = mx[w];
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
      const long long u = __shfl_up_sync(kFull, v, o);
      if (lane >= o) v += u;
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) m = max(m, __shfl_xor_sync(kFull, m, o));
    incl[w] = v;
    if (lane == 31) s_sum[w][warp] = v;
    if (lane == 0) s_max[w][warp] = m;
  }
  __syncthreads();
  if (warp == 0) {
#pragma unroll
    for (int w = 0; w < 2; ++w) {
      long long v = s_sum[w][lane];
      int m = s_max[w][lane];
#pragma unroll
      for (int o = 1; o < 32; o <<= 1) {
        const long long u = __shfl_up_sync(kFull, v, o);
        if (lane >= o) v += u;
      }
#pragma unroll
      for (int o = 16; o > 0; o >>= 1) m = max(m, __shfl_xor_sync(kFull, m, o));
      s_sum[w][lane] = v;  // inclusive over warps
      if (lane == 31) p.sizes[(w * 2) * p.P + path] = v;
      if (lane == 0) p.sizes[(w * 2 + 1) * p.P + path] = m;
    }
  }
  __syncthreads();
#pragma unroll
  for (int w = 0; w < 2; ++w) {
    long long base = incl[w] - sum[w] + (warp > 0 ? s_sum[w][warp - 1] : 0);
    long long* out = (w == 0 ? p.dec_off : p.ali_off) + (size_t)path * p.B;
    for (int b = b0; b < b1; ++b) {
      out[b] = base;
      base += (w == 0) ? p.dec_len[(size_t)b * p.P + path] : p.ali_len[(size_t)b * p.P + path];
    }
  }
}


// Pointer table of the COMPACT output layout: all outputs of a decode as consecutive slices of one
// int64 buffer -- per path: decoded indices [n,2], values [n], shape [2], alignment indices, values,
// shape; then log_probability [B,P] (float32 pairs or float64 in int64 slots) -- computed on the device
// from the sizes the scan left there, so that the pack can be enqueued before the host knows them.
static __global__ void PackTableKernel(const long long* sizes, int B, int P, int real_bytes, long long* buf,
                                       unsigned long long buf_elems, long long** ptrs, int* overflow) {
  if (threadIdx.x != 0 || blockIdx.x != 0) return;
  unsigned long long o = 0;
  for (int p = 0; p < P; ++p) {
    const unsigned long long nd = (unsigned long long)sizes[0 * P + p], na = (unsigned long long)sizes[2 * P + p];
    ptrs[0 * P + p] = buf + o; o += 2 * nd;
    ptrs[1 * P + p] = buf + o; o += nd;
    ptrs[2 * P + p] = buf + o; o += 2;
    ptrs[3 * P + p] = buf + o; o += 2 * na;
    ptrs[4 * P + p] = buf + o; o += na;
    ptrs[5 * P + p] = buf + o; o += 2;
  }
  ptrs[6 * P] = buf + o;
  o += (real_bytes == 8) ? (unsigned long long)B * P : ((unsigned long long)B * P + 1) / 2;
  if (o > buf_elems) *overflow = 1;
}

static __global__ void __launch_bounds__(128) PackKernel(PackParams p) {
  if (p.skip != nullptr && *p.skip != 0) return;
  const int b = blockIdx.x, path = blockIdx.y;
  const size_t row = (size_t)b * p.P + path;
  {
    const int n = p.dec_len[row];
    const long long o = p.dec_off[(size_t)path * p.B + b];
    long long* idx = p.ptrs[0 * p.P + path];
    long long* val = p.ptrs[1 * p.P + path];
    const int* src = p.dec + row * p.T;
    for (int i = threadIdx.x; i < n; i += blockDim.x) {
      idx[2 * (o + i)] = b;
      idx[2 * (o + i) + 1] = i;
      val[o + i] = src[i];
    }
  }
  {
    const int n = p.ali_len[row];
    const long long o = p.ali_off[(size_t)path * p.B + b];
    long long* idx = p.ptrs[3 * p.P + path];
    long long* val = p.ptrs[4 * p.P + path];
    const int* src = p.ali + row * p.T;
    for (int i = threadIdx.x; i < n; i += blockDim.x) {
      idx[2 * (o + i)] = b;
      idx[2 * (o + i) + 1] = i;
      val[o + i] = src[i];
    }
  }
  if (threadIdx.x == 0) {
    void* lp = (p.log_prob != nullptr) ? p.log_prob : (void*)p.ptrs[6 * p.P];
    if (p.real_bytes == 8)  // kernels.cc:87-89
      ((double*)lp)[row] = ((const double*)p.fin_total)[row];
    else
      ((float*)lp)[row] = ((const float*)p.fin_total)[row];
    if (b == 0) {
      long long* ds = p.ptrs[2 * p.P + path];
      long long* as = p.ptrs[5 * p.P + path];
      ds[0] = p.B; ds[1] = p.sizes[1 * p.P + path];  // kernels.cc:236-237
      as[0] = p.B; as[1] = p.sizes[3 * p.P + path];  // kernels.cc:253-254
    }
  }
}

// Test hook: element-wise evaluation of the exact math functions.
// op 0: expf, 1: log1pf, 2: logf, 3: LogSumExp(x, 0), 4: LogSumExp(0, x)
static __global__ void MathTestKernel(int op, const float* x, float* y, int n) {
  __shared__ unsigned long long s_tab[32];
  LoadExpTable(s_tab, threadIdx.x, blockDim.x);
  __syncthreads();
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  const float v = x[i];
  y[i] = (op == 0) ? ExpfExact(v, s_tab) : (op == 1) ? Log1pfExact(v) : (op == 2) ? LogfExact(v)
       : (op == 3) ? LogSumExp(v, 0.0f, s_tab) : LogSumExp(0.0f, v, s_tab);
}

// op 0: exp (x <= 0), 1: log (x >= 1), 2: LogSumExp(x, 0) of the double path
static __global__ void MathTestKernelF64(int op, const double* x, double* y, int n) {
  __shared__ unsigned long long s_tab[256];
  __shared__ unsigned long long s_tabf[32];
  for (int i = threadIdx.x; i < 256; i += blockDim.x) s_tab[i] = kCtcxExpTab[i];
  LoadExpTable(s_tabf, threadIdx.x, blockDim.x);
  __syncthreads();
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  const double v = x[i];
  y[i] = (op == 0) ? ExpExactD(v, s_tab) : (op == 1) ? LogExactD(v) : LogSumExp(v, 0.0, s_tabf);
}

namespace {
// Reduces the per-utterance flags to stats[0..5] = {OR of anomaly bits, first b with too few leaves (or
// B), first b with sequence_length > T (or B), first b with negative sequence_length (or B), first b fed
// more frames than a stream holds (or B), first b whose input frames never arrived (or B)}.
// MASKED: only the utterances with mask[b] != 0 take part.
template <bool MASKED>
__device__ __forceinline__ void ReduceFlags(const int* flags, const int* seq_len, int B, int T, int* out,
                                            const int* mask) {
  for (int b = blockIdx.x * blockDim.x + threadIdx.x; b < B; b += gridDim.x * blockDim.x) {
    if constexpr (MASKED) {
      if (mask[b] == 0) continue;
    }
    const int f = flags ? flags[b] : 0;
    if (f & 1) atomicOr(&out[0], 1);
    if (f & 2) atomicMin(&out[1], b);
    if (seq_len[b] > T) atomicMin(&out[2], b);
    if (seq_len[b] < 0) atomicMin(&out[3], b);
    if (f & 4) atomicMin(&out[4], b);
    if (f & 8) atomicMin(&out[5], b);
  }
}
__global__ void FlagsKernel(const int* flags, const int* seq_len, int B, int T, int* out) {
  ReduceFlags<false>(flags, seq_len, B, T, out, nullptr);
}
__global__ void FlagsKernelMasked(const int* flags, const int* seq_len, int B, int T, int* out, const int* mask) {
  ReduceFlags<true>(flags, seq_len, B, T, out, mask);
}

// flag = 1 if any entry is positive or NaN (scorer tables hold log-probabilities)
__global__ void PositiveKernel(const float* v, long long n, int* flag) {
  for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (long long)gridDim.x * blockDim.x)
    if (!(v[i] <= 0.0f)) *flag = 1;
}

// Every float block holds the root (what a float kernel resumes if a float64 step advanced the frame
// count: a valid beam, never foreign bytes), marked "no float step yet" and tagged with the stream's
// score type; the double blocks of a float64 stream are marked unwritten.
__device__ __forceinline__ void ResetStreamBlock(unsigned char* state, int B, int W, int score_bytes, int b) {
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
__global__ void StreamResetKernel(unsigned char* state, int B, int W, int score_bytes) {
  for (int b = blockIdx.x * blockDim.x + threadIdx.x; b < B; b += gridDim.x * blockDim.x)
    ResetStreamBlock(state, B, W, score_bytes, b);
}

// Reset() of the utterances with mask[b] != 0: everything ctcx_stream_reset_v writes for b (the state
// block, no frames consumed, the root as the final beam: one leaf, log-probability 0, and "fewer leaves
// than top_paths" when P > 1), written on the device so that the launch can be captured in a graph.
__global__ void StreamResetSlotsKernel(StreamSlotsParams p) {
  for (int b = blockIdx.x * blockDim.x + threadIdx.x; b < p.B; b += gridDim.x * blockDim.x) {
    if (p.mask[b] == 0) continue;
    ResetStreamBlock(p.state, p.B, p.W, p.score_bytes, b);
    p.t_done[b] = 0;
    for (int k = 0; k < p.P; ++k) {
      if (p.score_bytes == 8) static_cast<double*>(p.fin_total)[(size_t)b * p.P + k] = 0.0;
      else static_cast<float*>(p.fin_total)[(size_t)b * p.P + k] = 0.0f;
      p.fin_kind[(size_t)b * p.P + k] = 0;
    }
    p.fin_n[b] = 1;
    p.flags[b] = (p.P > 1) ? 2 : 0;
  }
}

// A float64 step on a float stream marks the float header's type; a float step on a float64 stream drops
// the "no float step yet" flag (float kernels rewrite the flags of every block they step).
// mask: optional [B], non-zero = the utterance is checked (null = all); the table word is read for the
// first utterance, or for every selected one.
__global__ void StreamCheckKernel(const unsigned char* state, int B, int W, const int* table_flag, int* stats,
                                  const int* mask) {
  for (int b = blockIdx.x * blockDim.x + threadIdx.x; b < B; b += gridDim.x * blockDim.x) {
    if (mask != nullptr && mask[b] == 0) continue;
    const StreamHdr* h = reinterpret_cast<const StreamHdr*>(state + (size_t)b * StreamStateBytes(W));
    const bool mixed = (h->type & kStreamF64Stepped) || (h->type == 8 && !(h->flags & kStreamNoF32Step));
    if (mixed || ((mask != nullptr || b == 0) && *table_flag != 0)) atomicMin(&stats[3], 0);
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
    auto tk = tp.mask != nullptr ? TraceKernel<Masked<REC>> : TraceKernel<REC>;
    tk<<<(unsigned)((walks + 127) / 128), 128, 0, stream>>>(tp);
  } else {
    // one warp per (utterance, path); two blocks of 2^rows_log2 back-pointer rows per warp in
    // shared memory (at most 26 KB per block: a single row of records, 8 KB at beam width 1024, is less)
    constexpr int kTraceWarps = 2;
    constexpr size_t kBlockBytes = 26 * 1024;
    int rows_log2 = 5;
    while (rows_log2 > 0 && ((size_t)W << rows_log2) * sizeof(REC) > kBlockBytes) --rows_log2;
    const size_t tsm = (size_t)kTraceWarps * 2 * ((size_t)W << rows_log2) * sizeof(REC);
    const bool masked = tp.mask != nullptr;
    auto tk = masked ? TraceWarpKernel<Masked<REC>, kTraceWarps> : TraceWarpKernel<REC, kTraceWarps>;
    static KernelSetup setup, setup_masked;
    const cudaError_t e = (masked ? setup_masked : setup).RaiseSmemLimit((const void*)tk, kTraceWarps * 2 * kBlockBytes);
    if (e != cudaSuccess) return LaunchFrom(e, "shared-memory limit of TraceWarpKernel");
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
  if (tp.mask != nullptr) FlagsKernelMasked<<<(tp.B + 255) / 256, 256, 0, stream>>>(flags, tp.seq_len, tp.B, tp.T, stats, tp.mask);
  else FlagsKernel<<<(tp.B + 255) / 256, 256, 0, stream>>>(flags, tp.seq_len, tp.B, tp.T, stats);
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

LaunchStatus LaunchStreamResetSlots(const StreamSlotsParams& p, cudaStream_t stream) {
  StreamResetSlotsKernel<<<(unsigned)((p.B + 127) / 128), 128, 0, stream>>>(p);
  return LaunchFrom(cudaGetLastError(), "StreamResetSlotsKernel launch");
}

LaunchStatus LaunchStreamCheck(unsigned char* state, int B, int W, const int* table_flag, int* stats,
                               const int* mask, cudaStream_t stream) {
  StreamCheckKernel<<<(unsigned)((B + 127) / 128), 128, 0, stream>>>(state, B, W, table_flag, stats, mask);
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
