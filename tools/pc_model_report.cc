// What the narrow kernel's revisit-wipe fixed point (PC) has to do, per frame, measured on the CPU model of
// the parallel formulation (tests/model/ctcx_model.cc, included below): the model's Beam evolves the beam,
// and before every step this file recomputes the step's member update, ranks and candidates to report,
// for the at-risk members, the round-1 wipe counts. Built and driven by tools/pc_model_report.py.
#include "../tests/model/ctcx_model.cc"

namespace {

// out[11]: frames with at-risk members, at-risk members, contested members (round-1 count >= W), members
// above lp_max + the old best total (never listed by PA), round-1 count / W in quarters (5 bins, the last
// >= 1), fixed-point rounds summed over the frames with at-risk members, their maximum.
void Report(const Beam& bm, const float* x, long long* out) {
  const int n = bm.n, W = bm.W, C = bm.C, blank = bm.blank;
  float mx = x[0];
  for (int j = 1; j < C; ++j) mx = x[j] > mx ? x[j] : mx;
  float sum = 0.f;
  for (int j = 0; j < C; ++j) sum += expf(x[j] - mx);
  const float off = mx + logf(sum);
  std::vector<int> pslot(n, -1);
  for (int i = 0; i < n; ++i)
    if (bm.label[i] >= 0)
      for (int j = 0; j < n; ++j)
        if (bm.hash[j] == bm.phash[i]) { pslot[i] = j; break; }
  std::vector<int> at_risk;
  for (int m = 0; m < n; ++m) if (pslot[m] >= 0 && pslot[m] < m) at_risk.push_back(m);
  if (at_risk.empty()) return;
  std::vector<float> nt(n);  // new totals, as Beam::Step computes them
  for (int i = 0; i < n; ++i) {
    float v_nl = bm.lab[i];
    if (bm.label[i] >= 0) {
      const int j = pslot[i];
      if (j >= 0) v_nl = Lse(bm.lab[i], bm.label[i] == bm.label[j] ? bm.blk[j] : bm.total[j]) + x[bm.label[i]] - off;
      else v_nl = bm.lab[i] + (x[bm.label[i]] - off);
    }
    nt[i] = Lse(bm.total[i] + x[blank] - off, v_nl);
  }
  std::vector<char> kid((size_t)n * C, 0);
  for (int i = 0; i < n; ++i) if (pslot[i] >= 0) kid[(size_t)pslot[i] * C + bm.label[i]] = 1;
  float lp_max = kNegInf;
  for (int l = 0; l < C; ++l) if (l != blank && x[l] - off > lp_max) lp_max = x[l] - off;
  const float bound = lp_max + bm.total[0];
  out[0]++;
  for (size_t q = 0; q < at_risk.size(); ++q) {
    const int m = at_risk[q], b = pslot[m];
    int cnt = 0;  // round 1: members ranking before m, then the children the parent's sweep meets first
    for (int j = 0; j < n; ++j) cnt += (nt[j] > nt[m] || (nt[j] == nt[m] && j < m)) ? 1 : 0;
    for (int r = 0; r <= b; ++r)
      for (int l = 0; l < C; ++l) {
        if (l == blank || kid[(size_t)r * C + l] || (r == b && l >= bm.label[m])) continue;
        const float s = (x[l] - off) + (l == bm.label[r] ? bm.blk[r] : bm.total[r]);
        cnt += (s > nt[m]) ? 1 : 0;
      }
    out[1]++;
    out[2] += (cnt >= W) ? 1 : 0;
    out[3] += (nt[m] > bound) ? 1 : 0;
    out[4 + std::min(4, (4 * cnt) / W)]++;
  }
}

}  // namespace

extern "C" int ctcx_pc_report_f32(const float* logits, int T, int B, int C, const int* seq_len, int W,
                                  int blank_index, long long* out) {
  if (T == 0) return 2;
  for (int b = 0; b < B; ++b) if (!(seq_len[b] <= T)) return 5;
  std::memset(out, 0, 11 * sizeof(long long));
  Beam beam; beam.W = W; beam.C = C; beam.blank = blank_index; beam.blank_label = blank_index;
  for (int b = 0; b < B; ++b) {
    beam.Reset();
    for (int t = 0; t < seq_len[b]; ++t) {
      const float* x = logits + ((size_t)t * B + b) * C;
      const long long frames = out[0];
      Report(beam, x, out);
      const int rounds = beam.Step(x, nullptr);
      if (out[0] != frames) { out[9] += rounds; out[10] = std::max<long long>(out[10], rounds); }
    }
  }
  return 0;
}
