// Generic beam kernel (BeamKernelT): any vocabulary width, beam widths up to 1024, float32 and float64
// scores, the scorer table. The fast kernels (ctcx_beam_v4.cuh, ctcx_beam_wide.cuh) take the shapes
// they admit; this kernel takes every other one. Included only by k_generic.cu, which launches it.
#pragma once
#include "ctcx_kernels.cuh"

namespace ctcx {

// Shared-memory carve-up, computed identically on host and device.
struct BeamSmem {
  // byte offsets
  size_t hash, phash;          // u64 [2][WMAX]
  size_t surv;                 // Comp [WMAX]
  size_t exptab;               // u64 [32]
  size_t total, blk, lab, ab, an;  // R [2][WMAX]
  size_t label;                // i32 [2][WMAX]
  size_t m_nt, m_nb, m_nl, m_nab, m_nan;  // R [WMAX]
  size_t m_key;                // Key [WMAX]
  size_t m_rec;                // u32 [WMAX]
  size_t m_pslot;              // i32 [WMAX]
  size_t risk, risk_new;       // i32 [WMAX]
  size_t wiped;                // u32 [WMAX] (0/1)
  size_t part;                 // i32 [NT]
  size_t htab;                 // i32 [2*WMAX]
  size_t hist;                 // u32 [256]
  size_t x;                    // R [2][Cpad]
  size_t kid;                  // u32 [kid_rows*kid_words], kid_rows = beam_width rounded up to 32
  size_t c_key;                // Key [cand_cap]
  size_t c_id;                 // u32 [cand_cap]
  size_t offv;                 // R [2]   this / the next frame's normaliser
  size_t keys;                 // Key [4] min key, max key, radix prefix
  size_t scal;                 // i32/u32 [32] scalars
  size_t bytes;

  __host__ __device__ static size_t Align(size_t v, size_t a) { return (v + a - 1) / a * a; }
  // rs = sizeof(R): 4 (float) or 8 (double); every 8-byte array precedes the 4-byte ones
  __host__ __device__ static int KidRows(int W) { return (W + 31) / 32 * 32; }
  __host__ __device__ void Init(int wmax, int nt, int C, int kid_words, int cand_cap, int rs, int W) {
    size_t o = 0;
    const size_t w = (size_t)wmax, r = (size_t)rs;
    const size_t cpad = Align((size_t)C, 4);
    hash = o; o += 2 * w * 8;
    phash = o; o += 2 * w * 8;
    surv = o; o += w * (rs == 4 ? 8 : 16);
    exptab = o; o += 32 * 8;
    keys = o; o += 4 * 8;
    offv = o; o += 2 * 8;
    total = o; o += 2 * w * r;
    blk = o; o += 2 * w * r;
    lab = o; o += 2 * w * r;
    ab = o; o += 2 * w * r;
    an = o; o += 2 * w * r;
    m_nt = o; o += w * r;
    m_nb = o; o += w * r;
    m_nl = o; o += w * r;
    m_nab = o; o += w * r;
    m_nan = o; o += w * r;
    m_key = o; o += w * r;
    x = o; o += 2 * cpad * r;
    c_key = o; o += Align((size_t)cand_cap * r, 8);
    label = o; o += 2 * w * 4;
    m_rec = o; o += w * 4;
    m_pslot = o; o += w * 4;
    risk = o; o += w * 4;
    risk_new = o; o += w * 4;
    wiped = o; o += w * 4;
    part = o; o += (size_t)nt * 4;
    htab = o; o += 2 * w * 4;
    hist = o; o += 256 * 4;
    kid = o; o += (size_t)KidRows(W) * (size_t)kid_words * 4;  // sized by the beam width, not the tier
    c_id = o; o += (size_t)cand_cap * 4;
    scal = o; o += 32 * 4;
    bytes = Align(o, 16);
  }
};

// indices into the scalar block
enum {
  kScNCand = 0, kScNRisk, kScChanged, kScK, kScE, kScNSurv, kScTotalItems, kScAnomaly
};
enum { kKeyMin = 0, kKeyMaxSlot = 1, kKeyPrefix = 2 };  // slots of the Key-typed scalar block

template <typename R, int WMAX, int NT>
__global__ void __launch_bounds__(NT) BeamKernelT(BeamParamsT<R> p) {
  using Ops = RealOps<R>;
  using Key = typename Ops::Key;
  using Comp = typename Ops::Comp;
  constexpr bool kIsF32 = (sizeof(R) == 4);
  extern __shared__ __align__(16) unsigned char smem[];
  constexpr int NWARP = NT / 32;
  constexpr int TS = 2 * WMAX;  // hash-table slots (power of two)
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const int b = blockIdx.x;
  const int W = p.W, C = p.C, T = p.T, B = p.B, KW = p.kid_words, blank = p.blank_index;
  const bool list_mode = p.cand_cap > 0;
  // streaming: frames already consumed by earlier chunks; this chunk contributes L more
  const int t_done = (p.t_done != nullptr) ? p.t_done[b] : 0;
  const int L = max(0, min(p.seq_len[b], p.Tcap - t_done));
  bool resume = (p.state != nullptr) && t_done > 0;
  if constexpr (!kIsF32) resume = resume && StreamResumable64(p.state, B, W, b);

  BeamSmem lay;
  lay.Init(WMAX, NT, C, KW, p.cand_cap, (int)sizeof(R), W);
  unsigned long long* s_hash = (unsigned long long*)(smem + lay.hash);
  unsigned long long* s_phash = (unsigned long long*)(smem + lay.phash);
  Comp* s_surv = (Comp*)(smem + lay.surv);
  unsigned long long* s_exptab = (unsigned long long*)(smem + lay.exptab);
  R* s_total = (R*)(smem + lay.total);
  R* s_blk = (R*)(smem + lay.blk);
  R* s_lab = (R*)(smem + lay.lab);
  R* s_ab = (R*)(smem + lay.ab);
  R* s_an = (R*)(smem + lay.an);
  int* s_label = (int*)(smem + lay.label);
  R* m_nt = (R*)(smem + lay.m_nt);
  R* m_nb = (R*)(smem + lay.m_nb);
  R* m_nl = (R*)(smem + lay.m_nl);
  R* m_nab = (R*)(smem + lay.m_nab);
  R* m_nan = (R*)(smem + lay.m_nan);
  Key* m_key = (Key*)(smem + lay.m_key);
  unsigned* m_rec = (unsigned*)(smem + lay.m_rec);
  int* m_pslot = (int*)(smem + lay.m_pslot);
  int* s_risk = (int*)(smem + lay.risk);
  int* s_risk_new = (int*)(smem + lay.risk_new);
  unsigned* s_wiped = (unsigned*)(smem + lay.wiped);
  int* s_part = (int*)(smem + lay.part);
  int* s_htab = (int*)(smem + lay.htab);
  unsigned* s_hist = (unsigned*)(smem + lay.hist);
  R* s_x = (R*)(smem + lay.x);
  unsigned* s_kid = (unsigned*)(smem + lay.kid);
  Key* c_key = (Key*)(smem + lay.c_key);
  unsigned* c_id = (unsigned*)(smem + lay.c_id);
  volatile int* sc = (volatile int*)(smem + lay.scal);
  int* sci = (int*)(smem + lay.scal);
  Key* s_keys = (Key*)(smem + lay.keys);
  R* s_offv = (R*)(smem + lay.offv);
  const int cpad = (int)BeamSmem::Align((size_t)C, 4);

  // ---- initial state: the root (decoder.h:212-227) ----
  LoadExpTable(s_exptab, tid, NT);
  for (int i = tid; i < TS; i += NT) s_htab[i] = -1;
  for (int i = tid; i < BeamSmem::KidRows(W) * KW; i += NT) s_kid[i] = 0u;
  for (int i = tid; i < WMAX; i += NT) s_wiped[i] = 0u;
  if (tid == 0 && !resume) {
    s_total[0] = (R)0;
    s_blk[0] = (R)0;
    s_lab[0] = Ops::NegInf();
    s_ab[0] = (R)0;  // empty alignment with probability 1 (entry.h:204-209)
    s_an[0] = Ops::NegInf();
    s_label[0] = -1;
    s_hash[0] = kRootHash;
    s_phash[0] = 0ull;
    sci[kScAnomaly] = 0;
  }
  int n = 1;  // members in the beam (uniform across the CTA)
  if (resume) {  // beam as the previous chunk left it (buffer 0: local frame 0 reads buffer 0)
    const StreamViewT<R> sv = StreamBlock<R>(p.state, B, W, b);
    n = sv.hdr->n;
    for (int i = tid; i < n; i += NT) {
      s_total[i] = sv.total[i]; s_blk[i] = sv.blk[i]; s_lab[i] = sv.lab[i];
      s_ab[i] = sv.ab[i]; s_an[i] = sv.an[i]; s_label[i] = sv.label[i];
      s_hash[i] = sv.hash[i]; s_phash[i] = sv.phash[i];
    }
    if (tid == 0) sci[kScAnomaly] = sv.hdr->flags & 1;
  }
  // row 0 of the logits
  if (L > 0) {
    const R* g = p.logits + (size_t)b * C;
    for (int l = tid; l < C; l += NT) s_x[l] = g[l];
    if (tid == 0) s_offv[0] = p.off[b];
  }
  __syncthreads();
  for (int i = tid; i < n; i += NT) {  // parent look-up table of the initial beam (the root, or the resumed one)
    unsigned h = (unsigned)s_hash[i] & (TS - 1);
    while (atomicCAS(&s_htab[h], -1, i) != -1) h = (h + 1) & (TS - 1);
  }
  __syncthreads();

  for (int t = 0; t < L; ++t) {
    const int cur = t & 1, nxt = cur ^ 1;
    const R* x = s_x + cur * cpad;
    const R off = s_offv[cur];
    const R* o_total = s_total + cur * WMAX;
    const R* o_blk = s_blk + cur * WMAX;
    const R* o_lab = s_lab + cur * WMAX;
    const R* o_ab = s_ab + cur * WMAX;
    const R* o_an = s_an + cur * WMAX;
    const int* o_label = s_label + cur * WMAX;
    const unsigned long long* o_hash = s_hash + cur * WMAX;
    const unsigned long long* o_phash = s_phash + cur * WMAX;

    // prefetch the next frame's row (consumed after the barrier that ends this frame)
    if (t + 1 < L) {
      const R* g = p.logits + (size_t)(t + 1) * (size_t)p.tstride + (size_t)b * C;
      R* dst = s_x + nxt * cpad;
      for (int l = tid; l < C; l += NT) {
        const unsigned sa = (unsigned)__cvta_generic_to_shared(dst + l);
        asm volatile("cp.async.ca.shared.global [%0], [%1], %2;\n" ::"r"(sa), "l"(g + l), "n"(sizeof(R)));
      }
      if (tid == 0) {
        const unsigned sa = (unsigned)__cvta_generic_to_shared(s_offv + nxt);
        asm volatile("cp.async.ca.shared.global [%0], [%1], %2;\n" ::"r"(sa),
                     "l"(p.off + (size_t)(t + 1) * B + b), "n"(sizeof(R)));
      }
      asm volatile("cp.async.commit_group;\n" ::);
    }
    if (tid == 0) {
      sci[kScNCand] = 0;
      sci[kScNRisk] = 0;
      s_keys[kKeyMin] = Ops::kKeyMax;
      s_keys[kKeyMaxSlot] = (Key)0;
      sci[kScNSurv] = 0;
    }
    __syncthreads();

    // ---- (A) update the existing members (decoder.h:95-143) ----
    const R xb = x[blank];
    const R pb = Ops::Sub(xb, off);
    Key my_key = (Key)0;
    bool suspect = false;
    if (tid < n) {
      const int i = tid;
      const int lbl = o_label[i];
      int pslot = -1;
      R v_nl = o_lab[i], v_an = Ops::NegInf();
      R rescore = Ops::NegInf();  // what the parent's re-score of this member would be (decoder.h:172-182)
      unsigned an_kind = kAnNone, an_src = kInvalidSlot;
      if (lbl >= 0) {
        const unsigned long long ph = o_phash[i];
        unsigned h = (unsigned)ph & (TS - 1);
        for (;;) {  // parent->Active() <=> the parent prefix is in the beam (decoder.h:97)
          const int s = s_htab[h];
          if (s < 0) break;
          if (o_hash[s] == ph) { pslot = s; break; }
          h = (h + 1) & (TS - 1);
        }
        const R xl = x[lbl];
        const R pl = Ops::Sub(xl, off);
        const R self_an = Ops::Add(o_an[i], pl);
        if (pslot >= 0) {
          const bool same = (lbl == o_label[pslot]);
          R base = same ? o_blk[pslot] : o_total[pslot];
          if (p.lm != nullptr)  // GetStateExpansionScore(b->state, .), decoder.h:103,114
            base = Ops::Add(base, p.lm[(size_t)(o_label[pslot] + 1) * C + lbl]);
          v_nl = Ops::Sub(Ops::Add(LogSumExp(o_lab[i], base, s_exptab), xl), off);  // :102-104,:113-115
          rescore = Ops::Add(pl, base);
          v_an = Ops::Add(o_ab[pslot], pl);
          an_kind = kAnParAb;
          an_src = (unsigned)pslot;
          if (!same) {
            const R c2 = Ops::Add(o_an[pslot], pl);
            if (c2 > v_an) { v_an = c2; an_kind = kAnParAn; }
          }
          if (self_an > v_an) { v_an = self_an; an_kind = kAnSelfAn; an_src = (unsigned)i; }
        } else {
          v_nl = Ops::Add(o_lab[i], pl);  // :125
          v_an = self_an;
          an_kind = kAnSelfAn;
          an_src = (unsigned)i;
        }
      }
      const R v_nb = Ops::Sub(Ops::Add(o_total[i], xb), off);  // :132
      const R c1 = Ops::Add(o_ab[i], pb), c2 = Ops::Add(o_an[i], pb);
      const unsigned ab_kind = (c2 > c1) ? kAbFromAn : kAbFromAb;
      const R v_nt = LogSumExp(v_nb, v_nl, s_exptab);  // :139
      m_nt[i] = v_nt;
      m_nb[i] = v_nb;
      m_nl[i] = v_nl;
      m_nab[i] = (c2 > c1) ? c2 : c1;
      m_nan[i] = v_an;
      my_key = Ops::KeyOf(v_nt);
      m_key[i] = my_key;
      m_rec[i] = PackRec((unsigned)i, an_src, ab_kind, an_kind);
      m_pslot[i] = pslot;
      // Precondition of the one event that is reported instead of modelled (DESIGN.md "Known deviation"):
      // were this member evicted and then re-scored by its parent, rounding would put the re-score ABOVE
      // the member's own total, so the reference could accept it again (decoder.h:189-199; it does so only
      // when the beam bottom ties with that total). Mathematically total >= re-score always. The utterance
      // is flagged if such a member then drops out of the beam (survivor collection, below).
      suspect = Ops::KeyOf(rescore) > my_key;
      if (pslot >= 0) {
        atomicOr(&s_kid[pslot * KW + (lbl >> 5)], 1u << (lbl & 31));
        if (pslot < i) {  // the parent's turn comes first: candidate for the revisit-wipe
          const int q = atomicAdd(&sci[kScNRisk], 1);
          s_risk[q] = i;
        }
      }
    }
    // min / max member key
    {
      Key kmin = (tid < n) ? my_key : Ops::kKeyMax, kmax = (tid < n) ? my_key : (Key)0;
#pragma unroll
      for (int o = 16; o > 0; o >>= 1) {
        kmin = min(kmin, __shfl_xor_sync(kFull, kmin, o));
        kmax = max(kmax, __shfl_xor_sync(kFull, kmax, o));
      }
      if (lane == 0 && warp * 32 < n) {
        atomicMin(&s_keys[kKeyMin], kmin);
        atomicMax(&s_keys[kKeyMaxSlot], kmax);
      }
    }
    __syncthreads();
    // the hash table has served this frame's look-ups: clear it for the next beam
    for (int i = tid; i < TS; i += NT) s_htab[i] = -1;

    // weakest a-priori threshold: with a full beam nothing at or below the W-th member total can
    // ever be admitted (decoder.h:151-155); keys are compared instead of floats from here on
    const Key th0 = (n == W) ? max(s_keys[kKeyMin], Ops::kKeyNegInf) : Ops::kKeyNegInf;

    // ---- (C) fresh children above the threshold (decoder.h:161-187) ----
    // evaluates (row, label) -> score key; used to build the list or, in streaming mode, directly
    auto eval_child = [&](int row, int l, Key& skey) -> bool {
      if (l == blank) return false;
      if ((s_kid[row * KW + (l >> 5)] >> (l & 31)) & 1u) return false;  // c.Active(): merged in (A)
      const R pl = Ops::Sub(x[l], off);
      R base = (l == o_label[row]) ? o_blk[row] : o_total[row];
      if (p.lm != nullptr) base = Ops::Add(base, p.lm[(size_t)(o_label[row] + 1) * C + l]);  // :171,:176,:182
      skey = Ops::KeyOf(Ops::Add(pl, base));  // :172-182
      return skey > th0;
    };
    {
      Key kmax = (Key)0, kmin = Ops::kKeyMax;
      int cnt_stream = 0;
      for (int row = warp; row < n; row += NWARP) {
        for (int l0 = 0; l0 < C; l0 += 32) {
          const int l = l0 + lane;
          Key skey = (Key)0;
          const bool ok = (l < C) && eval_child(row, l, skey);
          if (ok) { kmax = max(kmax, skey); kmin = min(kmin, skey); }
          if (list_mode) {
            const unsigned m = __ballot_sync(kFull, ok);
            if (m) {
              int base = 0;
              if (lane == 0) base = atomicAdd(&sci[kScNCand], __popc(m));
              base = __shfl_sync(kFull, base, 0);
              if (ok) {
                const int pos = base + __popc(m & ((1u << lane) - 1u));
                c_key[pos] = skey;
                c_id[pos] = ((unsigned)row << 16) | (unsigned)l;
              }
            }
          } else {
            cnt_stream += ok ? 1 : 0;
          }
        }
      }
#pragma unroll
      for (int o = 16; o > 0; o >>= 1) {
        kmin = min(kmin, __shfl_xor_sync(kFull, kmin, o));
        kmax = max(kmax, __shfl_xor_sync(kFull, kmax, o));
        cnt_stream += __shfl_xor_sync(kFull, cnt_stream, o);
      }
      if (lane == 0) {
        if (kmax != (Key)0) {
          atomicMin(&s_keys[kKeyMin], kmin);
          atomicMax(&s_keys[kKeyMaxSlot], kmax);
        }
        if (!list_mode && cnt_stream) atomicAdd(&sci[kScNCand], cnt_stream);
      }
    }
    __syncthreads();
    const int n_cand = sci[kScNCand];
    const int n_risk = sci[kScNRisk];

    // ---- (D) revisit-wipe fixed point (SURVEY A.4; DESIGN.md "Parallel formulation") ----
    bool any_wiped = false;
    if (n_risk > 0) {
      for (;;) {
        if (tid == 0) sci[kScChanged] = 0;
        for (int q = warp; q < n_risk; q += NWARP) {  // one warp per at-risk member
          const int m = s_risk[q];
          const int pb_slot = m_pslot[m];
          int verdict = 0;
          if (!s_wiped[pb_slot]) {
            const Key vkey = m_key[m];
            const unsigned idm = ((unsigned)pb_slot << 16) | (unsigned)o_label[m];
            int cnt = 0;
            for (int j = lane; j < n; j += 32) {
              const Key kj = m_key[j];
              cnt += (kj > vkey || (kj == vkey && j < m)) ? 1 : 0;
            }
            if (list_mode) {
              for (int c = lane; c < n_cand; c += 32) {
                const unsigned id = c_id[c];
                cnt += (c_key[c] > vkey && id < idm && !s_wiped[id >> 16]) ? 1 : 0;
              }
            } else {
              for (int row = 0; row <= pb_slot; ++row) {
                if (s_wiped[row]) continue;
                const int lend = (row == pb_slot) ? o_label[m] : C;
                for (int l = lane; l < lend; l += 32) {
                  Key skey;
                  cnt += (eval_child(row, l, skey) && skey > vkey) ? 1 : 0;
                }
              }
            }
#pragma unroll
            for (int o = 16; o > 0; o >>= 1) cnt += __shfl_xor_sync(kFull, cnt, o);
            verdict = (cnt >= W) ? 1 : 0;
          }
          if (lane == 0) s_risk_new[q] = verdict;
        }
        __syncthreads();
        for (int q = tid; q < n_risk; q += NT) {
          const int m = s_risk[q];
          const unsigned v = (unsigned)s_risk_new[q];
          if (s_wiped[m] != v) {
            s_wiped[m] = v;
            sci[kScChanged] = 1;
          }
        }
        __syncthreads();
        const int changed = sc[kScChanged];
        __syncthreads();  // everyone has read the flag before it is written again
        if (!changed) break;
      }
      for (int q = tid; q < n_risk; q += NT) {
        const int m = s_risk[q];
        if (s_wiped[m]) {
          sci[kScChanged] = 2;  // "some member is wiped"
        }
      }
      __syncthreads();
      any_wiped = (sc[kScChanged] == 2);
    }

    // ---- (E) next beam = first W items in (score desc, members before children, visiting order) ----
    // Items are the members (key m_key, tie order = slot) and the live candidates (tie order =
    // (row,label)). Radix select on the score key finds the W-th key; exact ties at that key are cut
    // by a second select on the tie order.
    auto live = [&](unsigned id) -> bool { return !any_wiped || !s_wiped[id >> 16]; };
    // for_each_item(f): f(score_key, order_key) for every item, each handled by exactly one thread
    auto for_each_item = [&](auto&& f) {
      for (int i = tid; i < n; i += NT) f(m_key[i], (unsigned)i);
      if (list_mode) {
        for (int c = tid; c < n_cand; c += NT) {
          const unsigned id = c_id[c];
          if (live(id)) f(c_key[c], 0x80000000u | id);
        }
      } else {
        for (int row = warp; row < n; row += NWARP) {
          if (any_wiped && s_wiped[row]) continue;
          for (int l = lane; l < C; l += 32) {
            Key skey;
            if (eval_child(row, l, skey)) f(skey, 0x80000000u | ((unsigned)row << 16) | (unsigned)l);
          }
        }
      }
    };
    // one radix-select level: among items with pred(), find the K-th largest of key(); returns the
    // selected key in sc[kScPrefix] (+lo), the number still to take at that key in sc[kScK] and the
    // number of items equal to it in sc[kScE]; sc[kScTotalItems] = number of items seen.
    auto radix_select = [&](Key lo, Key range, int K, auto&& keyfn) {
      const int nbits = Ops::Bits(range);
      int npass = (nbits + 7) / 8;
      if (npass == 0) npass = 1;
      if (tid == 0) { s_keys[kKeyPrefix] = (Key)0; sci[kScK] = K; }
      for (int pass = npass - 1; pass >= 0; --pass) {
        const int shift = pass * 8;
        for (int i = tid; i < 256; i += NT) s_hist[i] = 0u;
        __syncthreads();
        const Key prefix = s_keys[kKeyPrefix];
        for_each_item([&](Key skey, unsigned okey) {
          Key key;
          if (!keyfn(skey, okey, key)) return;
          const Key d = key - lo;
          const Key hi = (shift + 8 >= Ops::kKeyBits) ? (Key)0 : (d >> (shift + 8));
          if (hi == prefix) atomicAdd(&s_hist[(unsigned)(d >> shift) & 255u], 1u);
        });
        __syncthreads();
        if (warp == 0) {
          const int k = sci[kScK];
          unsigned h[8];
          unsigned loc = 0;
#pragma unroll
          for (int q = 0; q < 8; ++q) { h[q] = s_hist[lane * 8 + q]; loc += h[q]; }
          unsigned suf = loc;  // inclusive suffix sum over lanes >= lane
#pragma unroll
          for (int o = 1; o < 32; o <<= 1) {
            const unsigned v = __shfl_down_sync(kFull, suf, o);
            if (lane + o < 32) suf += v;
          }
          const unsigned above = suf - loc;  // items in higher lanes' bins
          if (pass == npass - 1 && lane == 0) sci[kScTotalItems] = (int)suf;
          if ((int)suf >= k && (int)above < k) {
            unsigned acc = above;
#pragma unroll
            for (int q = 7; q >= 0; --q) {
              if ((int)(acc + h[q]) >= k && (int)acc < k) {
                s_keys[kKeyPrefix] = (prefix << 8) | (Key)(lane * 8 + q);
                sci[kScK] = k - (int)acc;
                sci[kScE] = (int)h[q];
              }
              acc += h[q];
            }
          }
        }
        __syncthreads();
      }
    };

    const int n_items_upper = n + n_cand;  // before removing wiped rows
    Key cut_d = (Key)0;  // survivors: d > cut_d || (d == cut_d && ~okey >= cut_o)
    unsigned cut_o = 0u;
    const Key lo = s_keys[kKeyMin];
    bool take_all = (!any_wiped && n_items_upper <= W);
    if (!take_all) {
      const Key range = s_keys[kKeyMaxSlot] - lo;
      radix_select(lo, range, W, [&](Key skey, unsigned, Key& key) { key = skey; return true; });
      const int total_items = sc[kScTotalItems];
      if (total_items <= W) {
        take_all = true;
      } else {
        cut_d = s_keys[kKeyPrefix];
        const int k_rem = sc[kScK], e = sc[kScE];
        __syncthreads();
        if (e != k_rem) {  // exact ties straddle the beam boundary: cut them by tie order
          const Key want = cut_d + lo;
          radix_select((Key)0, (Key)0xffffffffu, k_rem, [&](Key skey, unsigned okey, Key& key) {
            key = (Key)(~okey);
            return skey == want;
          });
          cut_o = (unsigned)s_keys[kKeyPrefix];
          __syncthreads();
        }
      }
    }
    // collect survivors as 64-bit composites (score key, ~tie order): larger = earlier in the beam
    for_each_item([&](Key skey, unsigned okey) {
      const Key d = skey - lo;
      if (take_all || d > cut_d || (d == cut_d && ~okey >= cut_o)) {
        const int pos = atomicAdd(&sci[kScNSurv], 1);
        if (pos < WMAX) s_surv[pos] = Ops::MakeComp(skey, ~okey);
      } else if (okey == (unsigned)tid && suspect) {
        sci[kScAnomaly] = 1;  // a suspect member (see (A)) drops out of the beam: report the utterance
      }
    });
    __syncthreads();
    const int n_new = min(sci[kScNSurv], WMAX);

    // ---- (F) rank the survivors and write the next beam + back-pointers ----
    {
      static_assert(NT >= WMAX && NT % WMAX == 0, "one thread per beam slot is assumed");
      constexpr int PARTS = NT / WMAX;
      const int k = (PARTS > 1) ? (tid % WMAX) : tid;
      const int part = (PARTS > 1) ? (tid / WMAX) : 0;
      int cnt = 0;
      if (k < n_new && part < PARTS) {
        const Comp mine = s_surv[k];
        const int j0 = (int)((long long)n_new * part / PARTS), j1 = (int)((long long)n_new * (part + 1) / PARTS);
        for (int j = j0; j < j1; ++j) cnt += Ops::Greater(s_surv[j], mine) ? 1 : 0;
      }
      if (PARTS > 1) {
        s_part[tid] = cnt;
        __syncthreads();
        if (part == 0 && k < n_new) {
          for (int q = 1; q < PARTS; ++q) cnt += s_part[q * WMAX + k];
        }
      }
      R* w_total = s_total + nxt * WMAX;
      R* w_blk = s_blk + nxt * WMAX;
      R* w_lab = s_lab + nxt * WMAX;
      R* w_ab = s_ab + nxt * WMAX;
      R* w_an = s_an + nxt * WMAX;
      int* w_label = s_label + nxt * WMAX;
      unsigned long long* w_hash = s_hash + nxt * WMAX;
      unsigned long long* w_phash = s_phash + nxt * WMAX;
      if (part == 0 && k < n_new) {
        const int r = cnt;  // new slot
        const Comp comp = s_surv[k];
        const unsigned okey = ~Ops::CompNotOrder(comp);
        unsigned rec;
        int lbl;
        unsigned long long hsh;
        if (!(okey & 0x80000000u)) {  // surviving member
          const int i = (int)okey;
          w_total[r] = m_nt[i];
          w_blk[r] = m_nb[i];
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
          const R s = Ops::UnKey(Ops::CompKey(comp));
          const R pl = Ops::Sub(x[lbl], off);
          R v_an = Ops::Add(o_ab[row], pl);
          unsigned an_kind = kAnParAb;
          if (lbl != o_label[row]) {
            const R c2 = Ops::Add(o_an[row], pl);
            if (c2 > v_an) { v_an = c2; an_kind = kAnParAn; }
          }
          w_total[r] = s;
          w_blk[r] = Ops::NegInf();
          w_lab[r] = s;
          w_ab[r] = Ops::NegInf();
          w_an[r] = v_an;
          hsh = HashChild(o_hash[row], lbl);
          w_phash[r] = o_hash[row];
          rec = PackRec(kInvalidSlot, (unsigned)row, kAbFromAb, an_kind);
        }
        w_label[r] = lbl;
        w_hash[r] = hsh;
        if (p.bp32 != nullptr)
          p.bp32[((size_t)b * p.Tcap + (t_done + t)) * W + r] = Rec64To32(rec, (unsigned)lbl);
        else
          p.bp[((size_t)b * p.Tcap + (t_done + t)) * W + r] = make_uint2(rec, (unsigned)lbl);
        // next frame's parent look-up table
        unsigned h = (unsigned)hsh & (TS - 1);
        while (atomicCAS(&s_htab[h], -1, r) != -1) h = (h + 1) & (TS - 1);
      }
      // un-mark this frame's member children and wipes
      if (tid < n) {
        const int ps = m_pslot[tid];
        if (ps >= 0) s_kid[ps * KW + (o_label[tid] >> 5)] = 0u;
        s_wiped[tid] = 0u;
      }
    }
    asm volatile("cp.async.wait_all;\n" ::);
    __syncthreads();
    n = n_new;
  }

  // ---- final beam (decoder.h:229-261): already sorted, the first P slots are the top paths ----
  {
    const int cur = L & 1;
    if (tid < p.P) {
      if (tid < n) {
        p.fin_total[(size_t)b * p.P + tid] = s_total[cur * WMAX + tid];
        p.fin_kind[(size_t)b * p.P + tid] = (s_ab[cur * WMAX + tid] > s_an[cur * WMAX + tid]) ? 1 : 0;
      } else {
        p.fin_total[(size_t)b * p.P + tid] = (R)0;
        p.fin_kind[(size_t)b * p.P + tid] = 0;
      }
    }
    const int overflow = (p.seq_len[b] > p.Tcap - t_done) ? 4 : 0;
    if (tid == 0) {
      p.fin_n[b] = n;
      p.flags[b] = (sci[kScAnomaly] ? 1 : 0) | ((p.P > n) ? 2 : 0) | overflow;
    }
    if (p.state != nullptr) {  // carry the beam to the next chunk
      const StreamViewT<R> sv = StreamBlock<R>(p.state, B, W, b);
      for (int i = tid; i < n; i += NT) {
        sv.total[i] = s_total[cur * WMAX + i]; sv.blk[i] = s_blk[cur * WMAX + i];
        sv.lab[i] = s_lab[cur * WMAX + i]; sv.ab[i] = s_ab[cur * WMAX + i];
        sv.an[i] = s_an[cur * WMAX + i]; sv.label[i] = s_label[cur * WMAX + i];
        sv.hash[i] = s_hash[cur * WMAX + i]; sv.phash[i] = s_phash[cur * WMAX + i];
      }
      if (tid == 0) {
        sv.hdr->n = n;
        sv.hdr->gap = 0u;
        sv.hdr->flags = (sci[kScAnomaly] ? 1 : 0) | overflow | (resume ? (sv.hdr->flags & 4) : 0);
        if constexpr (!kIsF32) {
          sv.hdr->type = 8;
          StreamMarkF64Step(p.state, W, b);
        }
      }
    }
    if (p.t_done != nullptr && tid == 0) p.t_done[b] = t_done + L;
  }
}

}  // namespace ctcx
