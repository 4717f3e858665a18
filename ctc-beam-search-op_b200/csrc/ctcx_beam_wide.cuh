// Beam kernel for WIDE vocabularies (32 < num_classes <= 2048: BASELINE's Conformer-BPE shape
// C=1024, W=16). Derived from the third generation of the narrow kernel (since grown into BeamKernelV4,
// ctcx_beam_v4.cuh): same phases, same total order, bit-identical results as the generic BeamKernelT
// (ctcx_beam_generic.cuh). What differs is how candidates are found: the
// pre-pass (NormTopClassesKernel) orders every frame's best classes by log-prob; the children of a row
// above ANY threshold are then a PREFIX of that order (fp addition is monotone), whose length an
// exact binary search finds in ~log2(Kc) steps -- instead of scoring W*C children and issuing W*C
// shared-memory histogram atomics per pass, as the generic kernel's streaming mode does.
//   * member-children are a bitmap [row][class] (few members have their parent in the beam);
//   * the repeated label (base = old blank mass) is re-tested individually;
//   * a revisit-wipe query sums prefix lengths over the rows visited before the parent's turn and
//     scans only the parent's own row for the "labels below label(m)" part.
//
// Why Kc = 2W+2 sorted classes per frame are enough (W = beam_width). A row's children enter the
// next beam in the order (score desc, label asc), at most W of them. Up to W-1 classes of a row are
// already members (skipped) and the repeated label scores lower than its position suggests, so the
// W best children of a row sit in its first 2W sorted positions -- unless scores that differ as
// log-probs round to the SAME sum, in which case the label order can prefer a class further down.
// All classes past position Kc score <= the sentinel (position Kc) <= the W-th best item, so only an
// exact tie with the lowest selected item can matter; the kernel detects that after the cut (rows
// whose prefix hit Kc) and swaps such classes in one by one from the raw row, in order. The
// revisit-wipe counts saturate at W, and a capped row alone contributes >= W+2, so they are exact
// as well (the own-row part falls back to the raw row when capped).
#pragma once
#include "ctcx_beam_common.cuh"

namespace ctcx {


struct BeamSmemWide {
  size_t hash, phash;              // u64 [2][WMAX]
  size_t sorted;                   // u64 [WMAX]   score-grouped survivors
  size_t bnd;                      // u64 [32]     boundary-bin items (fast path)
  size_t exptab;                   // u64 [32]
  size_t row;                      // uint4 [WMAX] {old total, old blank, label, -}
  size_t kid;                      // u32 [WMAX][KW] member-children bitmap
  size_t kids;                     // u32 [WMAX]     the same as a list (parent row << 16 | label)
  size_t cls;                      // u16 [2][Cs]  class at each sorted position (double-buffered)
  size_t list;                     // uint2 [cand_cap] {score key, (row<<16)|label}
  size_t total, blk, lab, ab, an;  // f32 [2][WMAX]
  size_t label;                    // i32 [2][WMAX]
  size_t m_nt, m_nb, m_nl, m_nab, m_nan;  // f32 [WMAX]
  size_t m_key, m_rec;             // u32 [WMAX]
  size_t m_pslot;                  // i32 [WMAX]
  size_t risk, risk_new;           // i32 [WMAX]
  size_t wiped;                    // u32 [WMAX]
  size_t htab;                     // u32 [8*WMAX]  (hash tag << 10 | slot), 0xffffffff = empty
  size_t hist, offs;               // u32 [kBinsV2] each
  size_t bins2;                    // u32 [256]
  size_t wsum;                     // i32 [32]     per-warp candidate counts (block scan)
  size_t pls;                      // f32 [2][Cs]  class log-probs sorted descending (double-buffered)
  size_t x;                        // f32 [2][Cx]  raw logit row (double-buffered), Cx = C rounded up to 4
  size_t scal;                     // 32 x 4 B
  size_t bytes;
  __host__ __device__ void Init(int wmax, int cand_cap, int C, int Cs) {
    const size_t kw = (size_t)(C + 31) / 32;
    size_t o = 0;
    const size_t w = (size_t)wmax;
    hash = o; o += 2 * w * 8;
    phash = o; o += 2 * w * 8;
    sorted = o; o += w * 8;
    bnd = o; o += kBndFast * 8;
    exptab = o; o += 32 * 8;
    row = o; o += w * 16;
    kid = o; o += w * kw * 4;
    kids = o; o += w * 4;
    cls = o; o += 2 * (size_t)Cs * 2;
    list = o; o += ((size_t)cand_cap * 8 + 15) / 16 * 16;  // keep the following arrays 16-byte aligned
    total = o; o += 2 * w * 4;
    blk = o; o += 2 * w * 4;
    lab = o; o += 2 * w * 4;
    ab = o; o += 2 * w * 4;
    an = o; o += 2 * w * 4;
    label = o; o += 2 * w * 4;
    m_nt = o; o += w * 4;
    m_nb = o; o += w * 4;
    m_nl = o; o += w * 4;
    m_nab = o; o += w * 4;
    m_nan = o; o += w * 4;
    m_key = o; o += w * 4;
    m_rec = o; o += w * 4;
    m_pslot = o; o += w * 4;
    risk = o; o += w * 4;
    risk_new = o; o += w * 4;
    wiped = o; o += w * 4;
    htab = o; o += 8 * w * 4;
    hist = o; o += kBinsV2 * 4;
    offs = o; o += kBinsV2 * 4;
    bins2 = o; o += 256 * 4;
    wsum = o; o += 32 * 4;
    pls = o; o += 2 * (size_t)Cs * 4;
    x = o; o += 2 * ((size_t)C + 3) / 4 * 4 * 4;
    scal = o; o += 32 * 4;
    bytes = (o + 15) / 16 * 16;
  }
};

enum { kWNKid = 23, kWCapped = 24, kWBest = 25 };  // scalar slots in addition to the kV2* / kV3* ones

template <typename IN, int WMAX, int NT, bool TIMING>
__global__ void __launch_bounds__(NT, ((NT <= 256 && !TIMING) ? 4 : 1)) BeamKernelWide(BeamParams p) {
  static_assert(NT >= WMAX && 2 * NT >= kBinsV2, "one thread per beam slot and per two histogram bins");
  extern __shared__ __align__(16) unsigned char smem[];
  constexpr int NWARP = NT / 32;
  constexpr int TS = 8 * WMAX;  // parent look-up table slots (load factor <= 1/8: ~97% of the look-ups miss)
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const int b = blockIdx.x;
  const int W = p.W, C = p.C, B = p.B, blank = p.blank_index;
  // streaming: frames already consumed by earlier chunks; this chunk contributes L more
  const int t_done = (p.t_done != nullptr) ? p.t_done[b] : 0;
  const int L = max(0, min(p.seq_len[b], p.Tcap - t_done));
  const bool resume = (p.state != nullptr) && t_done > 0;

  BeamSmemWide lay;
  lay.Init(WMAX, p.cand_cap, p.C, p.Cs);
  unsigned long long* s_hash = (unsigned long long*)(smem + lay.hash);
  unsigned long long* s_phash = (unsigned long long*)(smem + lay.phash);
  unsigned long long* s_sorted = (unsigned long long*)(smem + lay.sorted);
  unsigned long long* s_bnd = (unsigned long long*)(smem + lay.bnd);
  unsigned long long* s_exptab = (unsigned long long*)(smem + lay.exptab);
  uint4* s_row = (uint4*)(smem + lay.row);
  uint2* c_list = (uint2*)(smem + lay.list);
  float* s_total = (float*)(smem + lay.total);
  float* s_blk = (float*)(smem + lay.blk);
  float* s_lab = (float*)(smem + lay.lab);
  float* s_ab = (float*)(smem + lay.ab);
  float* s_an = (float*)(smem + lay.an);
  int* s_label = (int*)(smem + lay.label);
  float* m_nt = (float*)(smem + lay.m_nt);
  float* m_nb = (float*)(smem + lay.m_nb);
  float* m_nl = (float*)(smem + lay.m_nl);
  float* m_nab = (float*)(smem + lay.m_nab);
  float* m_nan = (float*)(smem + lay.m_nan);
  unsigned* m_key = (unsigned*)(smem + lay.m_key);
  unsigned* m_rec = (unsigned*)(smem + lay.m_rec);
  int* m_pslot = (int*)(smem + lay.m_pslot);
  int* s_risk = (int*)(smem + lay.risk);
  int* s_risk_new = (int*)(smem + lay.risk_new);
  unsigned* s_wiped = (unsigned*)(smem + lay.wiped);
  unsigned* s_htab = (unsigned*)(smem + lay.htab);
  unsigned* s_hist = (unsigned*)(smem + lay.hist);
  unsigned* s_offs = (unsigned*)(smem + lay.offs);
  unsigned* s_bins2 = (unsigned*)(smem + lay.bins2);
  float* s_plS2 = (float*)(smem + lay.pls);
  unsigned short* s_cls2 = (unsigned short*)(smem + lay.cls);
  unsigned* s_kid = (unsigned*)(smem + lay.kid);
  unsigned* s_kids = (unsigned*)(smem + lay.kids);
  const int Cs = p.Cs, KW = (C + 31) / 32, Cx = (C + 3) / 4 * 4;
  const int Cv = min(C - 1, p.Kc);      // length of the sorted order the kernel works with
  const bool trunc = Cv < C - 1;        // classes were left out; s_plS[Cv] is the best of them
  int P2 = 1;                           // largest power of two <= Cv (binary search start)
  while (2 * P2 <= Cv) P2 *= 2;
  int* s_wsum = (int*)(smem + lay.wsum);
  float* s_x = (float*)(smem + lay.x);
  volatile int* sc = (volatile int*)(smem + lay.scal);
  int* sci = (int*)(smem + lay.scal);
  unsigned* scu = (unsigned*)(smem + lay.scal);

  // ---- initial state: the root (decoder.h:212-227) ----
  LoadExpTable(s_exptab, tid, NT);
  for (int i = tid; i < TS; i += NT) s_htab[i] = 0xffffffffu;
  for (int i = tid; i < WMAX; i += NT) {
    s_wiped[i] = 0u;
    s_row[i] = make_uint4(0u, 0u, 0u, 0u);
  }
  for (int i = tid; i < kBinsV2; i += NT) s_hist[i] = 0u;
  if (tid == 0) {
    if (!resume) {
      s_total[0] = 0.0f;
      s_blk[0] = 0.0f;
      s_lab[0] = NegInf();
      s_ab[0] = 0.0f;  // empty alignment with probability 1 (entry.h:204-209)
      s_an[0] = NegInf();
      s_label[0] = -1;
      s_hash[0] = kRootHash;
      s_phash[0] = 0ull;
    }
    sci[kV2Anomaly] = 0;
    sci[kV2NCand] = 0;
    sci[kV2NRisk] = 0;
    scu[kV2MinKey] = 0xffffffffu;
    scu[kV2MaxKey] = 0u;
    sci[kV2NBnd] = 0;
    scu[kV2MinBase] = 0xffffffffu;
    scu[kV2Gap] = 0u;
    sci[kV3Found] = 0;
    sci[kWNKid] = 0;
    sci[kWCapped] = 0;
  }
  int n = 1;
  // thread -> (row, class slice) mapping of the candidate pass
  for (int i = tid; i < WMAX * KW; i += NT) s_kid[i] = 0u;
  if (L > 0) {  // frame 0: raw row, normaliser, sorted classes
    for (int l = tid; l < C; l += NT) s_x[l] = LoadLogit<IN>(p.logits, (size_t)b * C + l);
    const float* gp = p.srt_pl + (size_t)b * Cs;
    const unsigned short* gc = p.srt_cls + (size_t)b * Cs;
    for (int j = tid; j < Cs; j += NT) {
      s_plS2[j] = gp[j];
      s_cls2[j] = gc[j];
    }
    if (tid == 0) ((float*)sci)[kV2Off0] = p.off[b];
  }
  __syncthreads();
  if (resume) {  // beam as the previous chunk left it (buffer 0: local frame 0 reads buffer 0)
    StreamView sv(p.state + (size_t)b * StreamStateBytes(W), W);
    n = sv.hdr->n;
    for (int i = tid; i < n; i += NT) {
      s_total[i] = sv.total[i]; s_blk[i] = sv.blk[i]; s_lab[i] = sv.lab[i];
      s_ab[i] = sv.ab[i]; s_an[i] = sv.an[i]; s_label[i] = sv.label[i];
      s_hash[i] = sv.hash[i]; s_phash[i] = sv.phash[i];
    }
    if (tid == 0) {
      scu[kV2Gap] = sv.hdr->gap;
      sci[kV2Anomaly] = sv.hdr->flags & 1;
    }
    __syncthreads();
  }
  for (int i = tid; i < n; i += NT) {  // row info + parent look-up table of the initial beam
    s_row[i] = make_uint4(__float_as_uint(s_total[i]), __float_as_uint(s_blk[i]), (unsigned)s_label[i], 0u);
    const unsigned long long hsh = s_hash[i];
    unsigned h = (unsigned)hsh & (TS - 1);
    const unsigned entry = ((unsigned)(hsh >> 42) << 10) | (unsigned)i;
    while (atomicCAS(&s_htab[h], 0xffffffffu, entry) != 0xffffffffu) h = (h + 1) & (TS - 1);
  }
  __syncthreads();

  // optional per-phase clock64 instrumentation (thread 0), compiled out of the production kernel
  long long cyc[TIMING ? 24 : 1] = {0};
  long long tprev = 0;
  const bool timing = TIMING && (p.dbg_cycles != nullptr) && tid == 0;
#define CTCX_TICK(i)                      \
  if (TIMING && timing) {                 \
    const long long now_ = clock64();     \
    cyc[TIMING ? (i) : 0] += now_ - tprev; \
    tprev = now_;                         \
  }
  if (timing) tprev = clock64();
  for (int t = 0; t < L; ++t) {
    const int cur = t & 1, nxt = cur ^ 1;
    const float* x = s_x + cur * Cx;
    const float* s_plS = s_plS2 + cur * Cs;          // this frame's classes, best first
    const unsigned short* s_cls = s_cls2 + cur * Cs;
    const float off = ((const float*)sci)[kV2Off0 + cur];
    const float* o_total = s_total + cur * WMAX;
    const float* o_blk = s_blk + cur * WMAX;
    const float* o_lab = s_lab + cur * WMAX;
    const float* o_ab = s_ab + cur * WMAX;
    const float* o_an = s_an + cur * WMAX;
    const int* o_label = s_label + cur * WMAX;
    const unsigned long long* o_hash = s_hash + cur * WMAX;
    const unsigned long long* o_phash = s_phash + cur * WMAX;

    // prefetch the next frame (last warp, idle during PA): raw row, normaliser, sorted classes;
    // consumed after the barrier that ends this frame
    if (warp == NWARP - 1 && t + 1 < L) {
      const size_t r1 = (size_t)(t + 1) * B + b;
      const size_t g0 = (size_t)(t + 1) * (size_t)p.tstride + (size_t)b * C;
      if constexpr (sizeof(IN) != 4) {
        // half-precision logits: widened in registers on the way to shared memory. 16-byte loads (eight
        // elements per lane, all in flight together) where the row is aligned; this warp is idle during PA.
        const IN* g = reinterpret_cast<const IN*>(p.logits) + g0;
        if ((C & 7) == 0 && (reinterpret_cast<uintptr_t>(g) & 15u) == 0) {
#pragma unroll 4
          for (int l = lane * 8; l < C; l += 256) {
            const uint4 v = __ldcg(reinterpret_cast<const uint4*>(g + l));
            const float2 a = Unpack2<IN>(v.x), b2 = Unpack2<IN>(v.y), c2 = Unpack2<IN>(v.z), d2 = Unpack2<IN>(v.w);
            float* dst = s_x + nxt * Cx + l;
            *reinterpret_cast<float4*>(dst) = make_float4(a.x, a.y, b2.x, b2.y);
            *reinterpret_cast<float4*>(dst + 4) = make_float4(c2.x, c2.y, d2.x, d2.y);
          }
        } else {
#pragma unroll 4
          for (int l = lane; l < C; l += 32) s_x[nxt * Cx + l] = LoadLogit<IN>(p.logits, g0 + l);
        }
      } else {
        const float* g = reinterpret_cast<const float*>(p.logits) + g0;
        if ((C & 3) == 0 && (reinterpret_cast<uintptr_t>(g) & 15u) == 0) {  // rows 16-byte aligned
          for (int l = lane * 4; l < C; l += 128) {
            const unsigned sa = (unsigned)__cvta_generic_to_shared(s_x + nxt * Cx + l);
            asm volatile("cp.async.cg.shared.global [%0], [%1], 16;\n" ::"r"(sa), "l"(g + l));
          }
        } else {
          for (int l = lane; l < C; l += 32) {
            const unsigned sa = (unsigned)__cvta_generic_to_shared(s_x + nxt * Cx + l);
            asm volatile("cp.async.ca.shared.global [%0], [%1], 4;\n" ::"r"(sa), "l"(g + l));
          }
        }
      }
      const float* gp = p.srt_pl + r1 * Cs;            // rows are 16-byte aligned (Cs % 8 == 0)
      for (int j = lane * 4; j < Cs; j += 128) {
        const unsigned sa = (unsigned)__cvta_generic_to_shared(s_plS2 + nxt * Cs + j);
        asm volatile("cp.async.cg.shared.global [%0], [%1], 16;\n" ::"r"(sa), "l"(gp + j));
      }
      const unsigned short* gc = p.srt_cls + r1 * Cs;
      for (int j = lane * 8; j < Cs; j += 256) {
        const unsigned sa = (unsigned)__cvta_generic_to_shared(s_cls2 + nxt * Cs + j);
        asm volatile("cp.async.cg.shared.global [%0], [%1], 16;\n" ::"r"(sa), "l"(gc + j));
      }
      if (lane == 31) {
        const unsigned sa = (unsigned)__cvta_generic_to_shared((float*)sci + kV2Off0 + nxt);
        asm volatile("cp.async.ca.shared.global [%0], [%1], 4;\n" ::"r"(sa), "l"(p.off + r1));
      }
      asm volatile("cp.async.commit_group;\n" ::);
    }

    const float xb = x[blank];
    const float pb = __fsub_rn(xb, off);
    if (tid == NT - 1) {
      ((float*)sci)[kV2LpMax] = (Cv > 0) ? s_plS[0] : NegInf();
      ((float*)sci)[kV2LpMin] = (Cv > 0) ? s_plS[Cv - 1] : 0.0f;
    }
    CTCX_TICK(7)  // frame setup
    // ---- PA: update the existing members (decoder.h:95-143) ----
    unsigned my_key = 0u;
    bool suspect = false;
    if (tid < n) {
      const int i = tid;
      const int lbl = o_label[i];
      int pslot = -1;
      float v_nl = o_lab[i], v_an = NegInf();
      float rescore = NegInf();  // what the parent's re-score of this member would be (decoder.h:172-182)
      unsigned an_kind = kAnNone, an_src = kInvalidSlot;
      if (lbl >= 0) {
        const unsigned long long ph = o_phash[i];
        unsigned h = (unsigned)ph & (TS - 1);
        const unsigned tag = (unsigned)(ph >> 42);  // 22 hash bits disjoint from the table index
        for (;;) {  // parent->Active() <=> the parent prefix is in the beam (decoder.h:97)
          const unsigned e0 = s_htab[h], e1 = s_htab[(h + 1) & (TS - 1)];  // two probes in flight
          if (e0 == 0xffffffffu) break;
          if ((e0 >> 10) == tag && o_hash[e0 & 1023u] == ph) { pslot = (int)(e0 & 1023u); break; }
          if (e1 == 0xffffffffu) break;
          if ((e1 >> 10) == tag && o_hash[e1 & 1023u] == ph) { pslot = (int)(e1 & 1023u); break; }
          h = (h + 2) & (TS - 1);
        }
        CTCX_TICK(8)  // parent look-up
        const float xl = x[lbl];
        const float pl = __fsub_rn(xl, off);
        const float self_an = __fadd_rn(o_an[i], pl);
        if (pslot >= 0) {
          const bool same = (lbl == o_label[pslot]);
          const float base = same ? o_blk[pslot] : o_total[pslot];
          v_nl = __fsub_rn(__fadd_rn(LogSumExp(o_lab[i], base, s_exptab), xl), off);
          rescore = __fadd_rn(pl, base);
          v_an = __fadd_rn(o_ab[pslot], pl);
          an_kind = kAnParAb;
          an_src = (unsigned)pslot;
          if (!same) {
            const float c2 = __fadd_rn(o_an[pslot], pl);
            if (c2 > v_an) { v_an = c2; an_kind = kAnParAn; }
          }
          if (self_an > v_an) { v_an = self_an; an_kind = kAnSelfAn; an_src = (unsigned)i; }
        } else {
          v_nl = __fadd_rn(o_lab[i], pl);
          v_an = self_an;
          an_kind = kAnSelfAn;
          an_src = (unsigned)i;
        }
      }
      CTCX_TICK(9)  // first LSE + alignment candidates
      const float v_nb = __fsub_rn(__fadd_rn(o_total[i], xb), off);
      const float c1 = __fadd_rn(o_ab[i], pb), c2 = __fadd_rn(o_an[i], pb);
      const unsigned ab_kind = (c2 > c1) ? kAbFromAn : kAbFromAb;
      const float v_nt = LogSumExp(v_nb, v_nl, s_exptab);
      CTCX_TICK(10)  // second LSE
      m_nt[i] = v_nt;
      m_nb[i] = v_nb;
      m_nl[i] = v_nl;
      m_nab[i] = (c2 > c1) ? c2 : c1;
      m_nan[i] = v_an;
      my_key = KeyOf(v_nt);
      m_key[i] = my_key;
      m_rec[i] = PackRec((unsigned)i, an_src, ab_kind, an_kind);
      m_pslot[i] = pslot;
      // precondition of the reference's re-acceptance of an evicted member (decoder.h:189-199): rounding puts
      // the parent's re-score above the member's own total -- reported, not modelled (DESIGN.md "Known deviation")
      suspect = KeyOf(rescore) > my_key;
      if (pslot >= 0) {
        atomicOr(&s_kid[pslot * KW + (lbl >> 5)], 1u << (lbl & 31));
        s_kids[atomicAdd(&sci[kWNKid], 1)] = ((unsigned)pslot << 16) | (unsigned)lbl;
        if (pslot < i) {
          const int q = atomicAdd(&sci[kV2NRisk], 1);
          s_risk[q] = i;
        }
      }
    }
    CTCX_TICK(11)  // stores + atomics
    {
      const unsigned kmin = __reduce_min_sync(kFull, (tid < n) ? my_key : 0xffffffffu);
      const unsigned kmax = __reduce_max_sync(kFull, (tid < n) ? my_key : 0u);
      if (lane == 0 && warp * 32 < n) {
        atomicMin(&scu[kV2MinKey], kmin);
        atomicMax(&scu[kV2MaxKey], kmax);
      }
    }
    CTCX_TICK(12)  // min/max reduction
    if (__builtin_expect(n < W, 0)) {  // beam not full: every finite child is admissible; bound the score range
      unsigned kb = 0xffffffffu;
      if (tid < n) {
        const float ob = o_blk[tid], ot = o_total[tid];
        if (ot > NegInf()) kb = KeyOf((ob > NegInf()) ? fminf(ot, ob) : ot);
      }
      kb = __reduce_min_sync(kFull, kb);
      if (lane == 0 && warp * 32 < n) atomicMin(&scu[kV2MinBase], kb);
    }
    __syncthreads();
    CTCX_TICK(0)  // PA

    const int n_risk = sci[kV2NRisk];

    // Children of one row above a threshold. The classes are sorted by log-prob and fp addition is
    // monotone, so "(x_l - off) + old total > thr" holds exactly for a PREFIX of the sorted order:
    // branch-free binary search for its length (decoder.h:172-182).
    auto prefix_len = [&](const float ot, const float thr) -> int {
      int pos = 0;
      for (int step = P2; step >= 1; step >>= 1) {
        const int q = pos + step;
        if (q <= Cv && __fadd_rn(s_plS[q - 1], ot) > thr) pos = q;
      }
      return pos;
    };
    auto is_kid = [&](int row, int c) -> bool { return (s_kid[row * KW + (c >> 5)] >> (c & 31)) & 1u; };
    // one class of a row: a real candidate above thr? (not already a member, decoder.h:168; the
    // repeated label extends from the old blank mass, decoder.h:172-177)
    auto cand_ok = [&](int row, const uint4 ri, int c, int j, const float thr, float& s_out) -> bool {
      if (is_kid(row, c)) return false;
      const float base = (c == (int)ri.z) ? __uint_as_float(ri.y) : __uint_as_float(ri.x);
      s_out = __fadd_rn(s_plS[j], base);
      return s_out > thr;
    };
    // number of candidates of a row above thr: prefix length minus the member-children above thr
    // minus the repeated label if its own (lower) score fails. A class lies in the prefix exactly
    // when its log-prob + old total exceeds thr. For a capped row (len == Cv < C-1) the result is a
    // lower bound that is still >= W+2, all a revisit-wipe verdict needs (header comment).
    auto cand_count = [&](int row, const uint4 ri, const float thr) -> int {
      const float ot = __uint_as_float(ri.x);
      int cnt = prefix_len(ot, thr);
      const int nk = sci[kWNKid];
      for (int k = 0; k < nk; ++k) {  // members whose parent is in the beam: a handful
        const unsigned kd = s_kids[k];
        if ((int)(kd >> 16) == row && __fadd_rn(__fsub_rn(x[kd & 0xffffu], off), ot) > thr) --cnt;
      }
      const int lb = (int)ri.z;
      if (lb >= 0 && lb != blank && !is_kid(row, lb)) {
        const float pl = __fsub_rn(x[lb], off);
        if (__fadd_rn(pl, ot) > thr && !(__fadd_rn(pl, __uint_as_float(ri.y)) > thr)) --cnt;
      }
      return cnt;
    };

    // ---- PC: revisit-wipe fixed point (SURVEY A.4) ----
    if (__builtin_expect(n_risk > 0, 0)) {
      for (;;) {
        for (int q = warp; q < n_risk; q += NWARP) {  // one warp per at-risk member
          const int m = s_risk[q];
          const int pslot = m_pslot[m];
          int verdict = 0;
          if (!s_wiped[pslot]) {
            const unsigned vkey = m_key[m];
            const float v = m_nt[m];
            int cnt = 0;
            for (int j = lane; j < n; j += 32) {  // members ranking before m
              const unsigned kj = m_key[j];
              cnt += (kj > vkey || (kj == vkey && j < m)) ? 1 : 0;
            }
            const uint4 rp = s_row[pslot];
            const int lblm = o_label[m];
            if (Cv <= 64) {
              // short sorted order (small beam widths): the lanes hold the sorted log-probs, a row's
              // prefix length is one or two ballots -- no dependent shared-memory search per row
              const float pl0 = (lane < Cv) ? s_plS[lane] : NegInf();
              const float pl1 = (32 + lane < Cv) ? s_plS[32 + lane] : NegInf();
              int tot = 0;  // warp-uniform
              for (int r = 0; r < pslot; ++r) {
                if (s_wiped[r]) continue;
                const float ot = o_total[r];
                tot += __popc(__ballot_sync(kFull, __fadd_rn(pl0, ot) > v));
                if (Cv > 32) tot += __popc(__ballot_sync(kFull, __fadd_rn(pl1, ot) > v));
              }
              if (lane == 0) cnt += tot;
              // corrections as in cand_count: member-children above v, repeated labels that fail
              const int nk = sci[kWNKid];
              for (int k = lane; k < nk; k += 32) {
                const unsigned kd = s_kids[k];
                const int r = (int)(kd >> 16);
                if (r < pslot && !s_wiped[r] && __fadd_rn(__fsub_rn(x[kd & 0xffffu], off), o_total[r]) > v) --cnt;
              }
              for (int r = lane; r < pslot; r += 32) {
                if (s_wiped[r]) continue;
                const uint4 ri = s_row[r];
                const int lb = (int)ri.z;
                if (lb >= 0 && lb != blank && !is_kid(r, lb)) {
                  const float pl = __fsub_rn(x[lb], off);
                  if (__fadd_rn(pl, __uint_as_float(ri.x)) > v && !(__fadd_rn(pl, __uint_as_float(ri.y)) > v)) --cnt;
                }
              }
              // the parent's own row: classes below label(m) (an index condition, not a prefix one)
              const float otp = __uint_as_float(rp.x);
              const bool in0 = __fadd_rn(pl0, otp) > v, in1 = __fadd_rn(pl1, otp) > v;
              const unsigned pm_last = __ballot_sync(kFull, (Cv > 32) ? in1 : in0);
              if (trunc && ((pm_last >> ((Cv - 1) & 31)) & 1u)) {  // capped prefix: the raw row has every class
                for (int c = lane; c < lblm; c += 32) {
                  if (c == blank || is_kid(pslot, c)) continue;
                  const float base = (c == (int)rp.z) ? __uint_as_float(rp.y) : __uint_as_float(rp.x);
                  cnt += (__fadd_rn(__fsub_rn(x[c], off), base) > v) ? 1 : 0;
                }
              } else {
                float sv_;
                if (in0) { const int c = (int)s_cls[lane]; cnt += (c < lblm && cand_ok(pslot, rp, c, lane, v, sv_)) ? 1 : 0; }
                if (in1) { const int c = (int)s_cls[32 + lane]; cnt += (c < lblm && cand_ok(pslot, rp, c, 32 + lane, v, sv_)) ? 1 : 0; }
              }
            } else {
              // children visited before the parent's turn, from rows that are not wiped: whole prefixes
              for (int r0 = 0; r0 < pslot; r0 += 32) {
                const int r = r0 + lane;
                if (r < pslot && !s_wiped[r]) cnt += cand_count(r, s_row[r], v);
              }
              // ... and, in the parent's own row, the classes below label(m) (an index condition, not a
              // prefix one: scan the row's prefix)
              const int len = prefix_len(__uint_as_float(rp.x), v);
              if (trunc && len == Cv) {  // capped prefix: the raw row has every class
                for (int c = lane; c < lblm; c += 32) {
                  if (c == blank || is_kid(pslot, c)) continue;
                  const float base = (c == (int)rp.z) ? __uint_as_float(rp.y) : __uint_as_float(rp.x);
                  cnt += (__fadd_rn(__fsub_rn(x[c], off), base) > v) ? 1 : 0;
                }
              } else {
                for (int j = lane; j < len; j += 32) {
                  const int c = (int)s_cls[j];
                  float sv_;
                  cnt += (c < lblm && cand_ok(pslot, rp, c, j, v, sv_)) ? 1 : 0;
                }
              }
            }
            cnt = __reduce_add_sync(kFull, cnt);
            verdict = (cnt >= W) ? 1 : 0;
          }
          if (lane == 0) s_risk_new[q] = verdict;
        }
        __syncthreads();
        // every thread inspects the (few) verdicts itself: no flag, no extra barrier when nothing
        // changes -- the common case
        bool changed = false;
        int min_wiped = 0x7fffffff, max_parent = -1;
        for (int q = 0; q < n_risk; ++q) {
          const int m = s_risk[q];
          const unsigned v = (unsigned)s_risk_new[q];
          changed |= (s_wiped[m] != v);
          if (v) min_wiped = min(min_wiped, m);
          max_parent = max(max_parent, m_pslot[m]);
        }
        if (!changed) break;
        __syncthreads();  // all reads of s_wiped are done
        for (int q = tid; q < n_risk; q += NT) s_wiped[s_risk[q]] = (unsigned)s_risk_new[q];
        __syncthreads();
        // a query only counts rows up to its parent's: if every wiped row lies beyond every parent
        // row, no count (and no parent) is affected and the verdicts are final
        if (min_wiped > max_parent) break;
      }
    }
    CTCX_TICK(2)  // PC

    // ---- PB / PD: list + histogram of the items in the score range, boundary bin ----
    const unsigned minkey_m = scu[kV2MinKey];
    const float lp_max = ((const float*)sci)[kV2LpMax];
    unsigned lo_true;  // no item lies below this key
    if (n == W) {
      lo_true = minkey_m;  // decoder.h:151-155: nothing at or below the W-th member total is admitted
    } else {
      const unsigned kb = scu[kV2MinBase];
      unsigned lo_c = minkey_m;
      if (kb != 0xffffffffu) lo_c = KeyOf(__fadd_rn(UnKey(kb), ((const float*)sci)[kV2LpMin]));
      lo_true = max(min(minkey_m, lo_c), kKeyNegInf);
    }
    // every item is <= max(best member, best possible child); old totals are sorted, slot 0 is the max
    const unsigned hi_key = max(scu[kV2MaxKey], KeyOf(__fadd_rn(lp_max, o_total[0])));
    unsigned lo_key = lo_true;
    int shift = 0;
    bool clamped = false;
    int n_cand = 0;
    auto bucket_of = [&](unsigned key) -> int { return (key > lo_key) ? (int)((key - lo_key) >> shift) : 0; };
    for (int attempt = 0; attempt < 2; ++attempt) {
      // Score range of the histogram. Survivors crowd near the top while the admissible range reaches
      // far below, so the first attempt only looks at [hi - 1.25*gap - 64, hi], gap = the previous
      // frame's top-to-threshold distance; if fewer than W items live there the second attempt
      // takes the whole admissible range. The prediction affects speed only.
      lo_key = lo_true;
      if (attempt == 0 && n == W) {
        const unsigned gap = scu[kV2Gap];
        const unsigned long long reach = (5ull * gap) / 4ull + 64ull;  // measured on the narrow kernel: 1.0-1.25 x gap is best
        if (gap != 0u && reach < (unsigned long long)(hi_key - lo_true)) lo_key = hi_key - (unsigned)reach;
      }
      clamped = (lo_key != lo_true);
      const unsigned span = hi_key - lo_key;
      shift = max(0, (32 - __clz(span | 1u)) - kBinsLog2V2);  // (key - lo) >> shift < kBinsV2
      const float thr = (n == W) ? UnKey(lo_key) : NegInf();  // listed children: score > thr
      const bool member_in = !clamped || my_key > lo_key;
      CTCX_TICK(16)  // PB: range

      // PB: one warp per row (round robin); the row's candidates are a prefix of the sorted classes:
      // 32 positions per step, until a position fails
      for (int row = warp; row < n; row += NWARP) {
        if (s_wiped[row]) continue;
        const uint4 ri = s_row[row];
        const float ot = __uint_as_float(ri.x);
        for (int j0 = 0; j0 < Cv; j0 += 32) {
          const int j = j0 + lane;
          float sc_ = 0.0f;
          int c = 0;
          bool inp = false, ok = false;
          if (j < Cv) {
            inp = __fadd_rn(s_plS[j], ot) > thr;
            if (inp) {
              c = (int)s_cls[j];
              ok = cand_ok(row, ri, c, j, thr, sc_);
            }
          }
          const unsigned pm = __ballot_sync(kFull, inp);
          const unsigned mk = __ballot_sync(kFull, ok);
          // the last sorted position is inside the prefix: classes beyond the sorted ones may be too
          if (trunc && j0 + 32 >= Cv && ((pm >> (Cv - 1 - j0)) & 1u) && lane == 0) sci[kWCapped] = 1;
          if (mk) {
            int base = 0;
            if (lane == 0) base = atomicAdd(&sci[kV2NCand], __popc(mk));  // one atomic per 32 positions
            base = __shfl_sync(kFull, base, 0);
            if (ok) {
              const unsigned key = KeyOf(sc_);
              c_list[base + __popc(mk & ((1u << lane) - 1u))] = make_uint2(key, ((unsigned)row << 16) | (unsigned)c);
              atomicAdd(&s_hist[bucket_of(key)], 1u);
            }
          }
          if (pm != kFull) break;
        }
      }
      if (tid < n && member_in) atomicAdd(&s_hist[bucket_of(my_key)], 1u);
      CTCX_TICK(19)  // PB: list
      __syncthreads();
      n_cand = sci[kV2NCand];
      CTCX_TICK(1)  // PB

      // ---- PD: boundary bin of the W-th item and group offsets (two bins per thread) ----
      {
        // suffix sums over bins kBinsV2-1..0: thread `tid` owns bins hi = kBinsV2-1-2*tid and lo = hi-1, so an
        // inclusive PREFIX scan in thread order is an inclusive SUFFIX scan in bin order
        const int bin_hi = kBinsV2 - 1 - 2 * tid;
        unsigned h_hi = 0u, h_lo = 0u;
        if (bin_hi >= 1) {
          const uint2 hh = *reinterpret_cast<const uint2*>(&s_hist[bin_hi - 1]);
          h_lo = hh.x;
          h_hi = hh.y;
        }
        const unsigned h2 = h_hi + h_lo;
        unsigned incl = h2;
#pragma unroll
        for (int o = 1; o < 32; o <<= 1) {
          const unsigned v = __shfl_up_sync(kFull, incl, o);
          if (lane >= o) incl += v;
        }
        const unsigned nz = __ballot_sync(kFull, h2 != 0u);
        if (lane == 31) s_wsum[warp] = (int)incl;
        {
          const int l0 = nz ? (__ffs(nz) - 1) : 0;  // first lane (highest bins) holding anything
          const unsigned hh = __shfl_sync(kFull, h_hi, l0);
          const int tb = nz ? ((kBinsV2 - 1 - 2 * (warp * 32 + l0)) - (hh ? 0 : 1)) : -1;
          if (lane == 0) s_wsum[16 + warp] = tb;
        }
        __syncthreads();
        unsigned before = 0u, total = 0u;
        int topbin = -1;
#pragma unroll
        for (int w2 = 0; w2 < NWARP; ++w2) {
          const unsigned v = (unsigned)s_wsum[w2];
          total += v;
          if (w2 < warp) before += v;
          topbin = max(topbin, s_wsum[16 + w2]);
        }
        // with a clamped range the cut is valid only if the W-th item lies inside the range
        const bool usable = !clamped || (int)total >= W;
        if (bin_hi >= 1) {
          const int K = min(W, (int)total);
          const unsigned above_hi = before + incl - h2;  // items in bins above bin_hi
          const unsigned above_lo = above_hi + h_hi;
          *reinterpret_cast<uint2*>(&s_offs[bin_hi - 1]) = make_uint2(above_lo, above_hi);
          *reinterpret_cast<uint2*>(&s_hist[bin_hi - 1]) = make_uint2(0u, 0u);  // counters in PE / next attempt
          if (usable && (int)(above_hi + h_hi) >= K && (int)above_hi < K) {
            sci[kV2Bstar] = bin_hi;
            sci[kV2KRem] = K - (int)above_hi;
            sci[kV2E] = (int)h_hi;
            sci[kV2NNew] = K;
            sci[kV2TopBin] = topbin;
            sci[kV3Found] = 1;
          } else if (usable && (int)(above_lo + h_lo) >= K && (int)above_lo < K) {
            sci[kV2Bstar] = bin_hi - 1;
            sci[kV2KRem] = K - (int)above_lo;
            sci[kV2E] = (int)h_lo;
            sci[kV2NNew] = K;
            sci[kV2TopBin] = topbin;
            sci[kV3Found] = 1;
          }
        }
      }
      __syncthreads();
      CTCX_TICK(3)  // PD
      if (__builtin_expect(sc[kV3Found] != 0, 1)) break;  // otherwise the prediction missed: run again over the full range
      if (tid == 0) sci[kV2NCand] = 0;
      __syncthreads();
    }
    const bool member_in = !clamped || my_key > lo_key;
    const int bstar = sc[kV2Bstar], k_rem = sc[kV2KRem], e_b = sc[kV2E], n_new = sc[kV2NNew];
    // a suspect member (see PA) that is not certain to stay in the beam: report the utterance
    if (__builtin_expect(suspect, 0) && (!member_in || bucket_of(my_key) <= bstar)) sci[kV2Anomaly] = 1;
    const bool bnd_all = (e_b == k_rem);
    // next frame's range prediction: the measured top-to-threshold gap
    const unsigned gap_next = (unsigned)(sc[kV2TopBin] - bstar + 1) << shift;

    if (TIMING && timing) {  // event counters next to the cycle counters (slots 20-23)
      cyc[TIMING ? 20 : 0] += (!bnd_all && e_b > kBndFast) ? 1 : 0;  // slow boundary cut
      cyc[TIMING ? 21 : 0] += clamped ? 0 : 1;                        // full-range histogram (miss or no prediction)
      cyc[TIMING ? 22 : 0] += (sc[kWCapped] != 0) ? 1 : 0;           // some row's prefix hit Kc
      cyc[TIMING ? 23 : 0] += n_cand;                                 // listed candidates
    }
    // ---- PE: scatter every item at or above the boundary bin into its score group ----
    auto place = [&](unsigned key, unsigned okey) {
      const int bucket = bucket_of(key);
      const unsigned long long comp = ((unsigned long long)key << 32) | (unsigned long long)(~okey);
      if (bucket > bstar || (bucket == bstar && bnd_all)) {
        const unsigned pos = s_offs[bucket] + atomicAdd(&s_hist[bucket], 1u);
        if (pos < (unsigned)WMAX) s_sorted[pos] = comp;
      } else if (bucket == bstar && e_b <= kBndFast) {
        const int pos = atomicAdd(&sci[kV2NBnd], 1);
        if (pos < kBndFast) s_bnd[pos] = comp;
      }
    };
    if (tid < n && member_in) place(my_key, (unsigned)tid);
    for (int c0 = tid; c0 < n_cand; c0 += 4 * NT) {  // four independent entries in flight
      uint2 e[4];
#pragma unroll
      for (int u = 0; u < 4; ++u) {
        const int c = c0 + u * NT;
        e[u] = (c < n_cand) ? c_list[c] : make_uint2(0u, 0u);
      }
#pragma unroll
      for (int u = 0; u < 4; ++u)
        if (e[u].x) place(e[u].x, 0x80000000u | e[u].y);
    }
    __syncthreads();
    CTCX_TICK(4)  // PE

    // ---- PF: cut the boundary bin exactly ----
    if (!bnd_all) {
      if (__builtin_expect(e_b <= kBndFast, 1)) {
        if (warp == 0) {
          const unsigned long long mine = (lane < e_b) ? s_bnd[lane] : 0ull;
          const unsigned mlo = (unsigned)mine, mhi = (unsigned)(mine >> 32);
          int rank = 0;
          for (int j = 0; j < e_b; ++j) {
            const unsigned olo = __shfl_sync(kFull, mlo, j), ohi = __shfl_sync(kFull, mhi, j);
            const unsigned long long other = ((unsigned long long)ohi << 32) | olo;
            rank += (other > mine) ? 1 : 0;
          }
          if (lane < e_b && rank < k_rem) s_sorted[s_offs[bstar] + rank] = mine;
          if (lane == 0) s_hist[bstar] = (unsigned)k_rem;
        }
      } else {
        // many items in the boundary bin (coarse bins after a missed prediction, or pathological
        // ties such as constant logits): radix select of the k_rem largest (key, ~order) composites
        auto for_each_bnd = [&](auto&& f) {
          if (tid < n && member_in && bucket_of(my_key) == bstar)
            f(((unsigned long long)my_key << 32) | (unsigned long long)(~(unsigned)tid), my_key, (unsigned)tid);
          for (int c = tid; c < n_cand; c += NT) {
            const uint2 e = c_list[c];
            if (e.x && bucket_of(e.x) == bstar)
              f(((unsigned long long)e.x << 32) | (unsigned long long)(~(0x80000000u | e.y)), e.x,
                0x80000000u | e.y);
          }
        };
        const int npass = 8;
        if (tid == 0) { scu[kV2Prefix] = 0u; scu[kV2PrefixHi] = 0u; sci[kV2K] = k_rem; }
        __syncthreads();
        for (int pass = npass - 1; pass >= 0; --pass) {
          const int sh = pass * 8;
          unsigned* bins = s_bins2;
          for (int i = tid; i < 256; i += NT) bins[i] = 0u;
          __syncthreads();
          const unsigned long long prefix =
              ((unsigned long long)scu[kV2PrefixHi] << 32) | (unsigned long long)scu[kV2Prefix];
          for_each_bnd([&](unsigned long long v, unsigned, unsigned) {
            const unsigned long long hi = (sh + 8 >= 64) ? 0ull : (v >> (sh + 8));
            if (hi == prefix) atomicAdd(&bins[(unsigned)(v >> sh) & 255u], 1u);
          });
          __syncthreads();
          if (warp == 0) {
            const int k = sci[kV2K];
            unsigned h[8];
            unsigned loc = 0;
#pragma unroll
            for (int q = 0; q < 8; ++q) { h[q] = bins[lane * 8 + q]; loc += h[q]; }
            unsigned suf = loc;
#pragma unroll
            for (int o = 1; o < 32; o <<= 1) {
              const unsigned v = __shfl_down_sync(kFull, suf, o);
              if (lane + o < 32) suf += v;
            }
            unsigned acc = suf - loc;
            if ((int)suf >= k && (int)acc < k) {
#pragma unroll
              for (int q = 7; q >= 0; --q) {
                if ((int)(acc + h[q]) >= k && (int)acc < k) {
                  const unsigned long long np = (prefix << 8) | (unsigned long long)(lane * 8 + q);
                  scu[kV2Prefix] = (unsigned)np;
                  scu[kV2PrefixHi] = (unsigned)(np >> 32);
                  sci[kV2K] = k - (int)acc;
                }
                acc += h[q];
              }
            }
          }
          __syncthreads();
        }
        const unsigned long long cut =
            ((unsigned long long)scu[kV2PrefixHi] << 32) | (unsigned long long)scu[kV2Prefix];
        for_each_bnd([&](unsigned long long v, unsigned key, unsigned okey) {
          if (v >= cut) {
            const unsigned pos = s_offs[bstar] + atomicAdd(&s_hist[bstar], 1u);
            if (pos < (unsigned)WMAX)
              s_sorted[pos] = ((unsigned long long)key << 32) | (unsigned long long)(~okey);
          }
        });
      }
      __syncthreads();
    }

    // ---- capped rows: classes beyond the sorted ones that TIE with the lowest selected item and
    // precede it in (row, label) order replace it, one at a time in that order (header comment).
    // Every class left out scores <= the sentinel <= that item, so nothing else can be missing. ----
    if (__builtin_expect(trunc && sc[kWCapped] != 0, 0)) {
      const unsigned lastkey = KeyOf(s_plS[Cv - 1]);
      const int lastcls = (int)s_cls[Cv - 1];
      unsigned done_upto = 0u;  // left-out children up to this order key are in already
      for (;;) {
        unsigned long long mn = (tid < n_new) ? s_sorted[tid] : ~0ull;
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) {
          const unsigned long long v = __shfl_xor_sync(kFull, mn, o);
          mn = (v < mn) ? v : mn;
        }
        if (lane == 0) s_bnd[warp] = mn;
        if (tid == 0) scu[kWBest] = 0xffffffffu;
        __syncthreads();
        unsigned long long cutc = ~0ull;
#pragma unroll
        for (int w2 = 0; w2 < NWARP; ++w2) cutc = (s_bnd[w2] < cutc) ? s_bnd[w2] : cutc;
        const unsigned keyc = (unsigned)(cutc >> 32), okc = ~(unsigned)(cutc & 0xffffffffull);
        if (!(okc & 0x80000000u)) break;  // a member: members precede children on equal scores
        const int rowc = (int)((okc & 0x7fffffffu) >> 16);
        // a left-out class of row r scores <= sentinel + old total(r): no tie there, no tie at all
        const bool may_tie = tid <= rowc && !s_wiped[tid] && KeyOf(__fadd_rn(s_plS[Cv], o_total[tid])) == keyc;
        if (!__syncthreads_or(may_tie ? 1 : 0)) break;
        for (int idx = tid; idx < (rowc + 1) * C; idx += NT) {
          const int r = idx / C, c = idx - r * C;
          const unsigned ok = 0x80000000u | ((unsigned)r << 16) | (unsigned)c;
          if (c == blank || ok >= okc || ok <= done_upto || s_wiped[r]) continue;
          const float pl = __fsub_rn(x[c], off);
          const unsigned pk = KeyOf(pl);
          if (pk > lastkey || (pk == lastkey && c <= lastcls)) continue;  // among the sorted classes
          if (is_kid(r, c)) continue;
          const uint4 ri = s_row[r];
          const float base = (c == (int)ri.z) ? __uint_as_float(ri.y) : __uint_as_float(ri.x);
          if (KeyOf(__fadd_rn(pl, base)) == keyc) atomicMin(&scu[kWBest], ok);
        }
        __syncthreads();
        const unsigned best = scu[kWBest];
        if (best == 0xffffffffu) break;
        if (tid < n_new && s_sorted[tid] == cutc)
          s_sorted[tid] = ((unsigned long long)keyc << 32) | (unsigned long long)(~best);
        done_upto = best;
        __syncthreads();
      }
    }
    CTCX_TICK(5)  // PF
    // ---- PG: rank inside the score group = new slot; write the next beam + back-pointers ----
    {
      float* w_total = s_total + nxt * WMAX;
      float* w_blk = s_blk + nxt * WMAX;
      float* w_lab = s_lab + nxt * WMAX;
      float* w_ab = s_ab + nxt * WMAX;
      float* w_an = s_an + nxt * WMAX;
      int* w_label = s_label + nxt * WMAX;
      unsigned long long* w_hash = s_hash + nxt * WMAX;
      unsigned long long* w_phash = s_phash + nxt * WMAX;
      // clear the parent look-up table (this frame's look-ups happened in PA) before re-filling it
      for (int i = tid; i < TS / 4; i += NT)  // 16-byte stores
        reinterpret_cast<uint4*>(s_htab)[i] = make_uint4(0xffffffffu, 0xffffffffu, 0xffffffffu, 0xffffffffu);
      unsigned long long comp = 0ull;
      int r = -1;
      if (tid < n_new) {
        comp = s_sorted[tid];
        const int bucket = bucket_of((unsigned)(comp >> 32));
        const int g0 = (int)s_offs[bucket], g1 = g0 + (int)s_hist[bucket];
        // groups usually hold 1-3 items; quantised logits (bfloat16 inputs) make exact ties, i.e. large
        // groups: four independent loads per round keep the count off the shared-memory latency
        int rank = 0, j = g0;
#pragma unroll 1
        for (; j + 4 <= g1; j += 4) {
          const unsigned long long a = s_sorted[j], b2 = s_sorted[j + 1], c2 = s_sorted[j + 2], d2 = s_sorted[j + 3];
          rank += ((a > comp) ? 1 : 0) + ((b2 > comp) ? 1 : 0) + ((c2 > comp) ? 1 : 0) + ((d2 > comp) ? 1 : 0);
        }
#pragma unroll 1
        for (; j < g1; ++j) rank += (s_sorted[j] > comp) ? 1 : 0;
        r = g0 + rank;
      }
      CTCX_TICK(13)  // PG: rank in group
      __syncthreads();  // table cleared, ranks known; s_hist / scalars no longer needed this frame
      CTCX_TICK(14)  // PG: barrier
      for (int i = tid; i < kBinsV2; i += NT) s_hist[i] = 0u;
      if (tid == 0) {
        sci[kV2NCand] = 0;
        sci[kV2NRisk] = 0;
        scu[kV2MinKey] = 0xffffffffu;
        scu[kV2MaxKey] = 0u;
        sci[kV2NBnd] = 0;
        scu[kV2MinBase] = 0xffffffffu;
        scu[kV2Gap] = gap_next;
        sci[kV3Found] = 0;
        sci[kWNKid] = 0;
        sci[kWCapped] = 0;
      }
      if (tid < n) {
        s_wiped[tid] = 0u;
        const int ps = m_pslot[tid];  // un-mark this frame's member-children
        if (ps >= 0) s_kid[ps * KW + (o_label[tid] >> 5)] = 0u;
      }
      if (r >= 0) {
        const unsigned okey = ~(unsigned)(comp & 0xffffffffull);
        unsigned rec;
        int lbl;
        unsigned long long hsh;
        float nt_, nb_;
        if (!(okey & 0x80000000u)) {  // surviving member
          const int i = (int)okey;
          nt_ = m_nt[i];
          nb_ = m_nb[i];
          w_lab[r] = m_nl[i];
          w_ab[r] = m_nab[i];
          w_an[r] = m_nan[i];
          lbl = o_label[i];
          hsh = o_hash[i];
          w_phash[r] = o_phash[i];
          rec = m_rec[i];
        } else {  // fresh child (decoder.h:170-187)
          const int row = (int)((okey & 0x7fffffffu) >> 16);
          lbl = (int)(okey & 0xffffu);
          const float s = UnKey((unsigned)(comp >> 32));
          const float pl = __fsub_rn(x[lbl], off);
          float v_an = __fadd_rn(o_ab[row], pl);
          unsigned an_kind = kAnParAb;
          if (lbl != o_label[row]) {
            const float c2 = __fadd_rn(o_an[row], pl);
            if (c2 > v_an) { v_an = c2; an_kind = kAnParAn; }
          }
          nt_ = s;
          nb_ = NegInf();
          w_lab[r] = s;
          w_ab[r] = NegInf();
          w_an[r] = v_an;
          hsh = HashChild(o_hash[row], lbl);
          w_phash[r] = o_hash[row];
          rec = PackRec(kInvalidSlot, (unsigned)row, kAbFromAb, an_kind);
        }
        w_total[r] = nt_;
        w_blk[r] = nb_;
        w_label[r] = lbl;
        w_hash[r] = hsh;
        s_row[r] = make_uint4(__float_as_uint(nt_), __float_as_uint(nb_), (unsigned)lbl, 0u);
        if (p.bp32 != nullptr)
          p.bp32[((size_t)b * p.Tcap + (t_done + t)) * W + r] = Rec64To32(rec, (unsigned)lbl);
        else
          p.bp[((size_t)b * p.Tcap + (t_done + t)) * W + r] = make_uint2(rec, (unsigned)lbl);
        unsigned h = (unsigned)hsh & (TS - 1);
        const unsigned entry = ((unsigned)(hsh >> 42) << 10) | (unsigned)r;
        while (atomicCAS(&s_htab[h], 0xffffffffu, entry) != 0xffffffffu) h = (h + 1) & (TS - 1);
      }
      CTCX_TICK(15)  // PG: state write
    }
    asm volatile("cp.async.wait_all;\n" ::);
    __syncthreads();
    CTCX_TICK(6)  // PG
    n = n_new;
  }
  if (TIMING && timing)
    for (int i = 0; i < (TIMING ? 24 : 1); ++i) p.dbg_cycles[(size_t)b * p.dbg_slots + i] = cyc[i];
#undef CTCX_TICK

  // ---- final beam (decoder.h:229-261): sorted, the first P slots are the top paths ----
  {
    const int cur = L & 1;
    if (tid < p.P) {
      if (tid < n) {
        p.fin_total[(size_t)b * p.P + tid] = s_total[cur * WMAX + tid];
        p.fin_kind[(size_t)b * p.P + tid] = (s_ab[cur * WMAX + tid] > s_an[cur * WMAX + tid]) ? 1 : 0;
      } else {
        p.fin_total[(size_t)b * p.P + tid] = 0.0f;
        p.fin_kind[(size_t)b * p.P + tid] = 0;
      }
    }
    const int overflow = (p.seq_len[b] > p.Tcap - t_done) ? 4 : 0;
    if (tid == 0) {
      p.fin_n[b] = n;
      p.flags[b] = (sci[kV2Anomaly] ? 1 : 0) | ((p.P > n) ? 2 : 0) | overflow;
    }
    if (p.state != nullptr) {  // carry the beam (and the score-range prediction) to the next chunk
      StreamView sv(p.state + (size_t)b * StreamStateBytes(W), W);
      for (int i = tid; i < n; i += NT) {
        sv.total[i] = s_total[cur * WMAX + i]; sv.blk[i] = s_blk[cur * WMAX + i];
        sv.lab[i] = s_lab[cur * WMAX + i]; sv.ab[i] = s_ab[cur * WMAX + i];
        sv.an[i] = s_an[cur * WMAX + i]; sv.label[i] = s_label[cur * WMAX + i];
        sv.hash[i] = s_hash[cur * WMAX + i]; sv.phash[i] = s_phash[cur * WMAX + i];
      }
      if (tid == 0) {
        sv.hdr->n = n;
        sv.hdr->gap = scu[kV2Gap];
        sv.hdr->flags = (sci[kV2Anomaly] ? 1 : 0) | overflow | (resume ? (sv.hdr->flags & 4) : 0);
      }
    }
    if (p.t_done != nullptr && tid == 0) p.t_done[b] = t_done + L;
  }
}

}  // namespace ctcx
