// TEST INFRASTRUCTURE. CPU model of the PARALLEL formulation that the CUDA beam kernel implements
// (ctc-beam-search-op_b200/csrc/ctcx_beam.cu). It exists to validate the formulation -- slot arrays,
// prefix hashes, candidate lists, the count-based "revisit-wipe" fixed point, stable top-W selection,
// per-frame back-pointers and trace-back -- against oracle/ctcx_oracle.c (the sequential
// restatement of the reference) on thousands of utterances on the CPU, where iteration is cheap.
// Every step below is data-parallel over members / candidates, exactly as in the kernel; nothing
// here is used by the product path.
//
// Reference semantics being reproduced: util/ctc_ext_beam_search_decoder.h:67-261 and
// util/ctc_beam_entry.h (see DESIGN.md section "Parallel formulation" for the derivation).
#include <algorithm>
#include <cmath>
#include <cstdint>
#include <cstdio>
#include <cstring>
#include <vector>

namespace {

const float kNegInf = -INFINITY;

struct Stats {
  long long frames, cands, at_risk, fp_iters, fp_iters_max, wiped, wiped_with_cands, anomalies,
      cands_max, frames_wipe_matters, queries, radix_bits_sum,
      fp_unwipes,        // verdicts that flip from wiped back to kept in a later round of the fixed point
      wiped_parents,     // at-risk members whose parent is wiped in the final verdict
      frames_at_risk,    // frames with at least one at-risk member
      suspects_dropped;  // members whose parent's re-score beats their own total and that leave the beam
};

inline float Lse(float a, float b) {  // util/ctc_loss_util.h:33-41
  if (a == kNegInf) return b;
  if (b == kNegInf) return a;
  return (a > b) ? a + log1pf(expf(b - a)) : b + log1pf(expf(a - b));
}

inline uint64_t HashChild(uint64_t h, int label) {
  uint64_t z = (h ^ (uint64_t)(uint32_t)(label + 1)) * 0x9E3779B97F4A7C15ull;
  z ^= z >> 29;
  z *= 0xBF58476D1CE4E5B9ull;
  z ^= z >> 32;
  return z;
}
const uint64_t kRootHash = 0x243F6A8885A308D3ull;

enum { AB_FROM_AB = 0, AB_FROM_AN = 1 };
enum { AN_SELF_AN = 0, AN_PAR_AB = 1, AN_PAR_AN = 2, AN_NONE = 3 };

struct BackPtr {
  int prev_self;  // slot of this hypothesis in the previous frame (-1: fresh this frame)
  int an_src;     // slot (previous frame) the non-blank-ending alignment extends
  int label;      // last label of the hypothesis (-1 root)
  unsigned char ab_kind, an_kind;
};

struct Cand {
  float s;
  int row, label;
  float an;
  unsigned char an_kind;
};

// Variants of the revisit-wipe fixed point with a known mistake, for the test fixture: a case that
// guards against the mistake must decode differently under it (tests/golden/make_wipe_cases.py).
enum { kExact = 0, kCountWipedRows = 1, kFourRounds = 2 };

struct Beam {
  int W, C, blank, blank_label;
  int variant = kExact;
  const float* lm = nullptr;  // scorer table [C + 1, C] (row = label of the extended entry + 1), or null
  int n;
  std::vector<float> total, blk, lab, ab, an;
  std::vector<int> label;
  std::vector<uint64_t> hash, phash;
  std::vector<std::vector<BackPtr> > bp;

  // GetStateExpansionScore (decoder.h:103,114,176,182): the base of a child of an entry with last label
  // `from` (-1: the root) plus the table's entry, or the base unchanged without a table
  float Expand(int from, int to, float base) const { return lm ? base + lm[(size_t)(from + 1) * C + to] : base; }

  void Reset() {  // decoder.h:212-227
    n = 1;
    total.assign(W, kNegInf); blk.assign(W, kNegInf); lab.assign(W, kNegInf);
    ab.assign(W, kNegInf); an.assign(W, kNegInf); label.assign(W, -1);
    hash.assign(W, 0); phash.assign(W, 0);
    total[0] = 0.f; blk[0] = 0.f;
    ab[0] = 0.f;  // "empty alignment with probability 1" (entry.h:204-209 zero_ok case at t=0)
    hash[0] = kRootHash;
    bp.clear();
  }

  // Returns the rounds the revisit-wipe fixed point ran in this frame (the last one changes nothing).
  int Step(const float* x, Stats* st) {
    // decoder.h:71-80
    float mx = x[0];
    for (int j = 1; j < C; ++j) mx = x[j] > mx ? x[j] : mx;
    float sum = 0.f;
    for (int j = 0; j < C; ++j) sum += expf(x[j] - mx);
    const float off = mx + logf(sum);
    const float pb = x[blank] - off;

    // (1) parent slot of every member (trie parent is in the beam <=> parent->Active(), :97)
    std::vector<int> pslot(n, -1);
    for (int i = 0; i < n; ++i)
      if (label[i] >= 0)
        for (int j = 0; j < n; ++j)
          if (hash[j] == phash[i]) { pslot[i] = j; break; }

    // (2) update existing members (decoder.h:95-143), reading only old values
    std::vector<float> nt(n), nb(n), nl(n), nab(n), nan_(n);
    std::vector<BackPtr> rec_m(n);
    for (int i = 0; i < n; ++i) {
      BackPtr r; r.prev_self = i; r.an_src = -1; r.label = label[i]; r.an_kind = AN_NONE;
      float v_nl = lab[i], v_an = kNegInf;
      if (label[i] >= 0) {
        const float p = x[label[i]] - off;
        const int j = pslot[i];
        if (j >= 0) {
          if (label[i] == label[j]) {
            v_nl = Lse(lab[i], Expand(label[j], label[i], blk[j])) + x[label[i]] - off;
            v_an = ab[j] + p; r.an_kind = AN_PAR_AB; r.an_src = j;
            float c2 = an[i] + p;
            if (c2 > v_an) { v_an = c2; r.an_kind = AN_SELF_AN; r.an_src = i; }
          } else {
            v_nl = Lse(lab[i], Expand(label[j], label[i], total[j])) + x[label[i]] - off;
            v_an = ab[j] + p; r.an_kind = AN_PAR_AB; r.an_src = j;
            float c2 = an[j] + p;
            if (c2 > v_an) { v_an = c2; r.an_kind = AN_PAR_AN; r.an_src = j; }
            float c3 = an[i] + p;
            if (c3 > v_an) { v_an = c3; r.an_kind = AN_SELF_AN; r.an_src = i; }
          }
        } else {
          v_nl = lab[i] + p;
          v_an = an[i] + p; r.an_kind = AN_SELF_AN; r.an_src = i;
        }
      }
      nl[i] = v_nl;
      nb[i] = total[i] + x[blank] - off;
      float c1 = ab[i] + pb, c2 = an[i] + pb;
      if (c2 > c1) { nab[i] = c2; r.ab_kind = AB_FROM_AN; } else { nab[i] = c1; r.ab_kind = AB_FROM_AB; }
      nan_[i] = v_an;
      nt[i] = Lse(nb[i], nl[i]);
      rec_m[i] = r;
    }

    // (3) stable rank of every member by new total; weakest a-priori threshold
    std::vector<int> rank(n, 0);
    for (int i = 0; i < n; ++i)
      for (int j = 0; j < n; ++j)
        if (nt[j] > nt[i] || (nt[j] == nt[i] && j < i)) ++rank[i];
    float th0 = kNegInf;
    if (n == W) for (int i = 0; i < n; ++i) if (rank[i] == W - 1) th0 = nt[i];

    // (4) which children of a member are themselves members
    std::vector<char> kid((size_t)n * C, 0);
    for (int i = 0; i < n; ++i) if (pslot[i] >= 0) kid[(size_t)pslot[i] * C + label[i]] = 1;

    // (5) candidates: fresh children above th0, in visiting order (row, label) (decoder.h:161-187)
    std::vector<Cand> cands;
    std::vector<int> row_begin(n + 1, 0);
    for (int b = 0; b < n; ++b) {
      row_begin[b] = (int)cands.size();
      for (int l = 0; l < C; ++l) {
        if (l == blank || kid[(size_t)b * C + l]) continue;
        const float p = x[l] - off;
        Cand c; c.row = b; c.label = l;
        if (l == label[b]) {
          c.s = p + Expand(label[b], l, blk[b]);
          c.an = ab[b] + p; c.an_kind = AN_PAR_AB;
        } else {
          c.s = p + Expand(label[b], l, total[b]);
          c.an = ab[b] + p; c.an_kind = AN_PAR_AB;
          float c2 = an[b] + p;
          if (c2 > c.an) { c.an = c2; c.an_kind = AN_PAR_AN; }
        }
        if (c.s > kNegInf && c.s > th0) cands.push_back(c);
      }
    }
    row_begin[n] = (int)cands.size();

    // (6) revisit-wipe fixed point (SURVEY A.4): member m loses its turn iff its parent b is a
    // member with an earlier turn that is itself not wiped, and m has left the beam by the time b
    // reaches label(m): rank(m) + #{candidates visited before, from un-wiped rows, scoring above
    // m's new total} >= W.
    std::vector<char> wiped(n, 0);
    std::vector<int> at_risk;
    for (int m = 0; m < n; ++m) if (pslot[m] >= 0 && pslot[m] < m) at_risk.push_back(m);
    int iters = 0;
    if (!at_risk.empty()) {
      for (;;) {
        ++iters;
        std::vector<char> nw(n, 0);
        for (size_t q = 0; q < at_risk.size(); ++q) {
          const int m = at_risk[q], b = pslot[m];
          if (wiped[b]) continue;
          int cnt = 0;
          const int end_full = row_begin[b];
          for (int k = 0; k < end_full; ++k)
            if ((variant == kCountWipedRows || !wiped[cands[k].row]) && cands[k].s > nt[m]) ++cnt;
          for (int k = row_begin[b]; k < row_begin[b + 1]; ++k)
            if (cands[k].label < label[m] && cands[k].s > nt[m]) ++cnt;
          if (rank[m] + cnt >= W) nw[m] = 1;
        }
        if (nw == wiped) break;
        if (st)
          for (int m = 0; m < n; ++m) st->fp_unwipes += (wiped[m] && !nw[m]) ? 1 : 0;
        wiped.swap(nw);
        if (variant == kFourRounds && iters == 4) break;
      }
    }
    if (st) {
      st->frames++; st->cands += (long long)cands.size(); st->at_risk += (long long)at_risk.size();
      if ((long long)cands.size() > st->cands_max) st->cands_max = (long long)cands.size();
      st->fp_iters += iters; if (iters > st->fp_iters_max) st->fp_iters_max = iters;
      int matters = 0;
      for (int m = 0; m < n; ++m) if (wiped[m]) {
        st->wiped++;
        if (row_begin[m + 1] > row_begin[m]) { st->wiped_with_cands++; matters = 1; }
        // rounding anomaly: the re-scored member would beat its own former total (see DESIGN.md)
        const int b = pslot[m];
        const float p = x[label[m]] - off;
        const float s = p + Expand(label[b], label[m], (label[m] == label[b]) ? blk[b] : total[b]);
        if (s > nt[m]) st->anomalies++;
      }
      st->frames_wipe_matters += matters;
      st->frames_at_risk += at_risk.empty() ? 0 : 1;
      for (size_t q = 0; q < at_risk.size(); ++q) st->wiped_parents += wiped[pslot[at_risk[q]]] ? 1 : 0;
    }

    // (7) stable top-W over members (first, slot order) and live candidates (visiting order)
    struct Item { float s; int idx; };  // idx < n: member, else candidate idx-n
    std::vector<Item> items;
    for (int i = 0; i < n; ++i) items.push_back(Item{nt[i], i});
    for (size_t k = 0; k < cands.size(); ++k)
      if (!wiped[cands[k].row]) items.push_back(Item{cands[k].s, n + (int)k});
    std::stable_sort(items.begin(), items.end(), [](const Item& a, const Item& b) { return a.s > b.s; });
    const int n_new = std::min<int>((int)items.size(), W);
    if (st) {  // the kernels' rounding-anomaly report (DESIGN.md section 8), exactly as the generic kernel decides it
      std::vector<char> kept(n, 0);
      for (int k = 0; k < n_new; ++k) if (items[k].idx < n) kept[items[k].idx] = 1;
      for (int m = 0; m < n; ++m) {
        const int b = pslot[m];
        if (b < 0 || kept[m]) continue;
        const float p = x[label[m]] - off;
        if (p + Expand(label[b], label[m], (label[m] == label[b]) ? blk[b] : total[b]) > nt[m]) st->suspects_dropped++;
      }
    }

    // (8) write the new beam (sorted) and this frame's back-pointers
    std::vector<float> t2(W, kNegInf), b2(W, kNegInf), l2(W, kNegInf), ab2(W, kNegInf), an2(W, kNegInf);
    std::vector<int> lab2(W, -1);
    std::vector<uint64_t> h2(W, 0), ph2(W, 0);
    std::vector<BackPtr> recs(n_new);
    for (int k = 0; k < n_new; ++k) {
      const int idx = items[k].idx;
      if (idx < n) {
        t2[k] = nt[idx]; b2[k] = nb[idx]; l2[k] = nl[idx]; ab2[k] = nab[idx]; an2[k] = nan_[idx];
        lab2[k] = label[idx]; h2[k] = hash[idx]; ph2[k] = phash[idx];
        recs[k] = rec_m[idx];
      } else {
        const Cand& c = cands[idx - n];
        t2[k] = c.s; b2[k] = kNegInf; l2[k] = c.s; ab2[k] = kNegInf; an2[k] = c.an;
        lab2[k] = c.label; h2[k] = HashChild(hash[c.row], c.label); ph2[k] = hash[c.row];
        BackPtr r; r.prev_self = -1; r.an_src = c.row; r.label = c.label; r.ab_kind = AB_FROM_AB;
        r.an_kind = c.an_kind;
        recs[k] = r;
      }
    }
    total.swap(t2); blk.swap(b2); lab.swap(l2); ab.swap(ab2); an.swap(an2); label.swap(lab2);
    hash.swap(h2); phash.swap(ph2);
    n = n_new;
    bp.push_back(recs);
    return iters;
  }

  // decoder.h:229-261 + entry.h:123-152, from the back-pointers
  void TracePath(int slot, bool merge_repeated, std::vector<int>* dec, std::vector<int>* ali) const {
    dec->clear(); ali->clear();
    const int T = (int)bp.size();
    if (T == 0) return;
    int kind_ab = (ab[slot] > an[slot]) ? 1 : 0;  // entry.h:140
    for (int t = T - 1; t >= 0; --t) {
      const BackPtr& r = bp[t][slot];
      if (kind_ab) {
        ali->push_back(blank_label);
        kind_ab = (r.ab_kind == AB_FROM_AB);
        slot = r.prev_self;
      } else {
        ali->push_back(r.label);
        if (r.an_kind == AN_SELF_AN) { slot = r.prev_self; kind_ab = 0; }
        else {
          dec->push_back(r.label);
          slot = r.an_src; kind_ab = (r.an_kind == AN_PAR_AB);
        }
      }
    }
    std::reverse(ali->begin(), ali->end());
    std::reverse(dec->begin(), dec->end());
    if (merge_repeated) {  // entry.h:123-136
      std::vector<int> m;
      for (size_t i = 0; i < dec->size(); ++i)
        if (i + 1 == dec->size() || (*dec)[i] != (*dec)[i + 1]) m.push_back((*dec)[i]);
      dec->swap(m);
    }
  }
};

}  // namespace

// stats_out: the statistics summed over the batch (maxima for *_max); utt_stats_out: optional [B,16],
// the same per utterance; iters_out: optional [B,T], the fixed-point rounds of every frame (0 past the
// utterance's length). variant: kExact, or one of the mistaken fixed points above. lm: the scorer table
// of ctcx_decode_scorer_f32 ([C + 1, C], entries <= 0, -inf allowed), or null for the default scorer.
extern "C" int ctcx_model_decode_lm_utts_f32(const float* logits, int T, int B, int C, const int* seq_len,
                                             int W, int P, int merge_repeated, int blank_index,
                                             int blank_label, const float* lm, int* dec_len, int* dec,
                                             int* ali_len, int* ali, float* logp, long long* stats_out,
                                             long long* utt_stats_out, int* iters_out, int variant) {
  static_assert(sizeof(Stats) <= 16 * sizeof(long long), "the stats array has 16 slots");
  if (T == 0) return 2;
  for (int b = 0; b < B; ++b) if (!(seq_len[b] <= T)) return 5;
  Stats st; std::memset(&st, 0, sizeof(st));
  Beam beam; beam.W = W; beam.C = C; beam.blank = blank_index; beam.blank_label = blank_label;
  beam.variant = variant;
  beam.lm = lm;
  std::vector<int> d, a;
  for (int b = 0; b < B; ++b) {
    Stats us; std::memset(&us, 0, sizeof(us));
    beam.Reset();
    for (int t = 0; t < seq_len[b]; ++t) {
      const int it = beam.Step(logits + ((size_t)t * B + b) * C, &us);
      if (iters_out) iters_out[(size_t)b * T + t] = it;
    }
    if (iters_out) for (int t = seq_len[b]; t < T; ++t) iters_out[(size_t)b * T + t] = 0;
    if (P > W) return 6;
    if (P > beam.n) return 7;
    for (int p = 0; p < P; ++p) {
      const size_t row = (size_t)b * P + p;
      beam.TracePath(p, merge_repeated != 0, &d, &a);
      logp[row] = beam.total[p];
      dec_len[row] = (int)d.size(); ali_len[row] = (int)a.size();
      for (size_t i = 0; i < d.size(); ++i) dec[row * T + i] = d[i];
      for (size_t i = 0; i < a.size(); ++i) ali[row * T + i] = a[i];
    }
    if (utt_stats_out) {
      std::memset(utt_stats_out + (size_t)b * 16, 0, 16 * sizeof(long long));
      std::memcpy(utt_stats_out + (size_t)b * 16, &us, sizeof(us));
    }
    const long long iters_max = std::max(st.fp_iters_max, us.fp_iters_max);
    const long long cands_max = std::max(st.cands_max, us.cands_max);
    long long* acc = reinterpret_cast<long long*>(&st);
    const long long* u = reinterpret_cast<const long long*>(&us);
    for (size_t i = 0; i < sizeof(Stats) / sizeof(long long); ++i) acc[i] += u[i];
    st.fp_iters_max = iters_max;
    st.cands_max = cands_max;
  }
  if (stats_out) std::memcpy(stats_out, &st, sizeof(st));
  return 0;
}

extern "C" int ctcx_model_decode_utts_f32(const float* logits, int T, int B, int C, const int* seq_len,
                                          int W, int P, int merge_repeated, int blank_index,
                                          int blank_label, int* dec_len, int* dec, int* ali_len, int* ali,
                                          float* logp, long long* stats_out, long long* utt_stats_out,
                                          int* iters_out, int variant) {
  return ctcx_model_decode_lm_utts_f32(logits, T, B, C, seq_len, W, P, merge_repeated, blank_index, blank_label,
                                       nullptr, dec_len, dec, ali_len, ali, logp, stats_out, utt_stats_out,
                                       iters_out, variant);
}

extern "C" int ctcx_model_decode_f32(const float* logits, int T, int B, int C, const int* seq_len,
                                     int W, int P, int merge_repeated, int blank_index,
                                     int blank_label, int* dec_len, int* dec, int* ali_len, int* ali,
                                     float* logp, long long* stats_out) {
  return ctcx_model_decode_utts_f32(logits, T, B, C, seq_len, W, P, merge_repeated, blank_index, blank_label,
                                    dec_len, dec, ali_len, ali, logp, stats_out, nullptr, nullptr, kExact);
}
