// Beam kernel, fourth generation: the fast path for num_classes <= 32 (all of BASELINE's char-CTC
// shapes). Bit-identical results to the generic BeamKernelT (ctcx_beam_generic.cuh); what changed against
// the third generation (round 1) is how the kernel is fed and scheduled:
//
//   * persistent CTAs: the grid is sized to the machine (resident CTAs per SM x SM count) and every
//     CTA pulls utterances from a queue until it is empty -- no tail wave, ragged lengths balance
//   * the kernel reads the caller's RAW logits -- float32, float16 or bfloat16, any time stride (a
//     batch shard of a larger tensor is decoded in place) -- and the softmax normaliser of
//     decoder.h:71-80 is computed here: the last warp works ONE FRAME AHEAD of the other seven (row
//     t+2 in flight in a register, frame t+1's normaliser / class order / prefix masks being built
//     while the others update frame t), so there is no normaliser kernel, no `off` array, no fp32
//     scratch for half inputs, and nothing of it on the frame's critical path
//   * an optional device word `ready` = number of leading frames that have landed lets the kernel
//     run WHILE the logits are still being copied host->device in time slabs (ctcx_decode_hostin_*)
//   * 4-byte back-pointer records (beam_width <= 256, labels < 256)
//   * the histogram scan (PD) is one bin per thread over all eight warps instead of one warp
//   * PG: survivors are scattered to their final slot first, then slot r is written by thread r
//     (state) and thread WMAX + r (hash, row info, parent table) -- linear stores, half the chain
//   * instantiated on the score type: float for f32 / f16 / bf16 logits, double for f64 logits (the
//     reference's T = double registration) -- RealOps<R> supplies the arithmetic, the key and the
//     (key, ~order) composite, V4Rec<R> the row record and the list item; and on LM, the scorer table
//
// Per frame:
//   S   (last warp, for frame t+1) raw row -> x, off, per-class log-probs, classes ranked by log-prob,
//       prefix masks pref[j] = set of the j best classes
//   PA  member update, one thread per member                          decoder.h:95-143
//   PC  revisit-wipe fixed point (SURVEY A.4). A row's candidates above ANY threshold v are a
//       bitmask: pref[L(v)] & ~member-children, L found by an exact search over the sorted class
//       scores (fp add is monotone); a wipe query is a sum of popcounts -- no list. Rounds after
//       the first correct the counts by the rows whose state changed instead of recounting.
//   PB  only candidates inside the predicted score range (previous top-to-threshold gap x1.25) are
//       listed and histogrammed (256 bins); wiped rows are skipped                 decoder.h:146-187
//   PD  suffix scan -> boundary bin of the W-th item; if the prediction missed (fewer than
//       W items in range) PB/PD run again over the full admissible range
//   PE  items above the boundary bin are scattered into score groups
//   PF  the boundary bin is cut exactly (warp rank, or radix select for pathological ties)
//   PG  rank inside the score group = new slot; next beam, parent table, back-pointer records
//
// Total order of the beam: (score desc, members before children, children by (row, label)) -- the
// order the reference's sequential strict-'>' admission yields with a stable tie policy.
#pragma once
#include "ctcx_beam_common.cuh"

namespace ctcx {

// Shared-memory layout. Every offset is a compile-time constant of the tier (WMAX): the candidate list,
// the only array whose size depends on the shape, comes last -- so the kernel addresses all arrays as
// "base + immediate" and spends no registers on array pointers.
// RB = bytes of the score type R (4: float, 8: double). Keys are as wide as scores; a (key, ~order)
// composite, a row-info record and a list item are 2 / 4 / 2 scores wide.
// Row stride of the scorer table in shared memory, in floats. Lanes read rows of DIFFERENT previous
// labels at the same column: a stride of 32 would put them all on the same banks (a 29-way conflict on
// every 16-byte load of the candidate test); 36 spreads consecutive rows over the banks and keeps
// 16-byte alignment.
constexpr int kLmStride = 36;

template <int WMAX, bool LM = false, int RB = 4>
struct BeamSmemV4 {
  static constexpr size_t w = (size_t)WMAX;
  static constexpr size_t rb = (size_t)RB;
  static constexpr size_t hash = 0;                       // u64 [2][WMAX]
  static constexpr size_t phash = hash + 2 * w * 8;       // u64 [2][WMAX]
  static constexpr size_t sorted = phash + 2 * w * 8;     // Comp [WMAX]  score-grouped survivors
  static constexpr size_t fin = sorted + w * 2 * rb;      // Comp [WMAX]  survivors at their final slot
  static constexpr size_t bnd = fin + w * 2 * rb;         // Comp [32]    boundary-bin items (fast path)
  static constexpr size_t exptab = bnd + kBndFast * 2 * rb;  // u64 [32]  expf table
  static constexpr size_t exptabd = exptab + 32 * 8;      // u64 [256]    exp table of the double normaliser (R = double only)
  static constexpr size_t row = exptabd + (RB == 8 ? 256 * 8 : 0);  // Row [WMAX] {old total, old blank, label, member-children mask}
  static constexpr size_t total = row + w * 4 * rb;       // R [2][WMAX]
  static constexpr size_t blk = total + 2 * w * rb;
  static constexpr size_t lab = blk + 2 * w * rb;
  static constexpr size_t ab = lab + 2 * w * rb;
  static constexpr size_t an = ab + 2 * w * rb;
  static constexpr size_t label = an + 2 * w * rb;        // i32 [2][WMAX]
  static constexpr size_t m_nt = label + 2 * w * 4;       // R [WMAX] x 5: the members' new values
  static constexpr size_t m_nb = m_nt + w * rb;
  static constexpr size_t m_nl = m_nb + w * rb;
  static constexpr size_t m_nab = m_nl + w * rb;
  static constexpr size_t m_nan = m_nab + w * rb;
  static constexpr size_t m_key = m_nan + w * rb;         // Key [WMAX]
  static constexpr size_t m_rec = m_key + w * rb;         // u32 [WMAX]
  static constexpr size_t m_pslot = m_rec + w * 4;        // i32 [WMAX]
  static constexpr size_t risk = m_pslot + w * 4;         // i32 [WMAX]
  static constexpr size_t con = risk + w * 4;             // i32 [WMAX]   contested at-risk members (PC)
  static constexpr size_t wiped = con + w * 4;            // u32 [WMAX]
  static constexpr size_t qcnt = wiped + w * 4;           // i32 [WMAX]   per contested member: items ranking before it
  static constexpr size_t qchg = qcnt + w * 4;            // u32 [WMAX]   rows whose wiped state changed in this round: (row << 1) | new state
  static constexpr size_t htab = qchg + w * 4;            // u32 [8*WMAX]  (hash tag << 10 | slot), 0xffffffff = empty
  static constexpr size_t hist = htab + 8 * w * 4;        // u32 [kBinsV2]
  static constexpr size_t offs = hist + kBinsV2 * 4;      // u32 [kBinsV2]
  static constexpr size_t bins2 = offs + kBinsV2 * 4;     // u32 [256]
  static constexpr size_t wtot = bins2 + 256 * 4;         // u32 [16]     per-warp histogram totals + top bins (PD)
  static constexpr size_t x = wtot + 16 * 4;              // R [2][32]    raw logits of the frame
  static constexpr size_t pl = x + 2 * 32 * rb;           // R [2][32]    x[l] - off
  static constexpr size_t pls = pl + 2 * 32 * rb;         // R [2][32]    class log-probs sorted descending (-inf padding)
  static constexpr size_t plh = pls + 2 * 32 * rb;        // R [2][8]     pls[0,4,8,...]: heads of the groups of four
  static constexpr size_t pref = plh + 2 * 8 * rb;        // u32 [2][36]  pref[j] = classes at sorted positions < j
  static constexpr size_t fsc = pref + 2 * 36 * 4;        // R [2][4]     {off, lp_max, lp_min, -}
  static constexpr size_t bits = fsc + 2 * 4 * rb;        // Key [32]     S warp scratch: sort keys, then class bits (u32)
  static constexpr size_t e = bits + 32 * rb;             // R [32]       S warp scratch: exp terms of the normaliser
  static constexpr size_t scal = e + 32 * rb;             // 32 x 4 B
  static constexpr size_t keys = scal + 32 * 4;           // Key [8]      min / max member key, min base, range prediction
  static constexpr size_t prefix = keys + 8 * rb;         // Comp [1] (+ pad) radix-select prefix of the slow boundary cut
  static constexpr size_t lm = (prefix + 32 + 15) / 16 * 16;      // f32 [33][32]  scorer table (LM kernels only), row = previous label + 1
  static constexpr size_t list = lm + (LM ? 33 * kLmStride * 4 : 0);  // Item [cand_cap] {score key, (row<<16)|label}
  static constexpr size_t Bytes(int cand_cap) { return (list + (size_t)cand_cap * 2 * rb + 15) / 16 * 16; }
};

// Key-typed scalars (shared-memory block `keys`)
enum { kV4KMin = 0, kV4KMax = 1, kV4KMinBase = 2, kV4KGap = 3 };

// The score type a kernel instantiation computes in: double for float64 logits (the reference's
// T = double registration, kernels.cc:275), float for float32 / float16 / bfloat16 logits.
template <typename IN> struct ScoreOf { using type = float; };
template <> struct ScoreOf<double> { using type = double; };

template <typename IN>
__device__ __forceinline__ typename ScoreOf<IN>::type LoadRaw(const void* base, size_t i) {
  if constexpr (sizeof(IN) == 8) return __ldcg(reinterpret_cast<const double*>(base) + i);
  else return LoadLogit<IN>(base, i);
}

// Layout-dependent records of the two score types. float keeps the packed 16-byte row record and the
// 8-byte list item of the single-precision kernel; double doubles both.
template <typename R> struct V4Rec;
template <> struct V4Rec<float> {
  using Row = uint4;   // {old total, old blank, label, member-children mask}
  using Item = uint2;  // {score key, (row << 16) | label}
  __device__ static __forceinline__ Row MakeRow(float ot, float ob, int label) {
    return make_uint4(__float_as_uint(ot), __float_as_uint(ob), (unsigned)label, 0u);
  }
  __device__ static __forceinline__ float Ot(const Row& r) { return __uint_as_float(r.x); }
  __device__ static __forceinline__ float Ob(const Row& r) { return __uint_as_float(r.y); }
  __device__ static __forceinline__ int Label(const Row& r) { return (int)r.z; }
  __device__ static __forceinline__ unsigned Mask(const Row& r) { return r.w; }
  __device__ static __forceinline__ unsigned* MaskPtr(Row* r) { return &r->w; }
  __device__ static __forceinline__ Item MakeItem(unsigned key, unsigned id) { return make_uint2(key, id); }
  __device__ static __forceinline__ Item NoItem() { return make_uint2(0u, 0u); }
  __device__ static __forceinline__ unsigned ItemKey(const Item& e) { return e.x; }
  __device__ static __forceinline__ unsigned ItemId(const Item& e) { return e.y; }
};
template <> struct V4Rec<double> {
  struct __align__(16) Row { double ot, ob; int label; unsigned mask; unsigned long long pad; };
  struct __align__(16) Item { unsigned long long key; unsigned id, pad; };
  __device__ static __forceinline__ Row MakeRow(double ot, double ob, int label) { return Row{ot, ob, label, 0u, 0ull}; }
  __device__ static __forceinline__ double Ot(const Row& r) { return r.ot; }
  __device__ static __forceinline__ double Ob(const Row& r) { return r.ob; }
  __device__ static __forceinline__ int Label(const Row& r) { return r.label; }
  __device__ static __forceinline__ unsigned Mask(const Row& r) { return r.mask; }
  __device__ static __forceinline__ unsigned* MaskPtr(Row* r) { return &r->mask; }
  __device__ static __forceinline__ Item MakeItem(unsigned long long key, unsigned id) { return Item{key, id, 0u}; }
  __device__ static __forceinline__ Item NoItem() { return Item{0ull, 0u, 0u}; }
  __device__ static __forceinline__ unsigned long long ItemKey(const Item& e) { return e.key; }
  __device__ static __forceinline__ unsigned ItemId(const Item& e) { return e.id; }
};

// warp-wide min / max of keys, and a composite taken from another lane
__device__ __forceinline__ unsigned WarpMinKey(unsigned k) { return __reduce_min_sync(kFull, k); }
__device__ __forceinline__ unsigned WarpMaxKey(unsigned k) { return __reduce_max_sync(kFull, k); }
__device__ __forceinline__ unsigned long long WarpMinKey(unsigned long long k) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) k = min(k, __shfl_xor_sync(kFull, k, o));
  return k;
}
__device__ __forceinline__ unsigned long long WarpMaxKey(unsigned long long k) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) k = max(k, __shfl_xor_sync(kFull, k, o));
  return k;
}
__device__ __forceinline__ unsigned long long ShflComp(unsigned long long c, int src) {
  const unsigned lo = __shfl_sync(kFull, (unsigned)c, src), hi = __shfl_sync(kFull, (unsigned)(c >> 32), src);
  return ((unsigned long long)hi << 32) | lo;
}
__device__ __forceinline__ ulonglong2 ShflComp(ulonglong2 c, int src) {
  return make_ulonglong2(__shfl_sync(kFull, c.x, src), (unsigned long long)__shfl_sync(kFull, (unsigned)c.y, src));
}
// The radix select of the slow boundary cut walks the bytes of a composite from the top: byte `pass`
// (0 = least significant), the bytes above it as a "prefix", and a prefix extended by one byte. The
// 64-bit composite keeps its prefix right-aligned (shifted down), the 96-bit one in place (lower bytes
// zero); either way the prefix after pass 0 is the whole composite.
__device__ __forceinline__ unsigned CompByte(unsigned long long c, int pass) { return (unsigned)(c >> (pass * 8)) & 255u; }
__device__ __forceinline__ unsigned long long CompAbove(unsigned long long c, int pass) {
  return (pass >= 7) ? 0ull : (c >> (pass * 8 + 8));
}
__device__ __forceinline__ unsigned long long CompWithByte(unsigned long long prefix, int, unsigned byte) {
  return (prefix << 8) | (unsigned long long)byte;
}
__device__ __forceinline__ unsigned CompByte(ulonglong2 c, int pass) {  // bytes 0-3: ~order, 4-11: key
  return (pass < 4) ? ((unsigned)c.y >> (pass * 8)) & 255u : (unsigned)(c.x >> ((pass - 4) * 8)) & 255u;
}
__device__ __forceinline__ ulonglong2 CompAbove(ulonglong2 c, int pass) {
  if (pass < 3) return make_ulonglong2(c.x, (unsigned long long)(((unsigned)c.y >> (pass * 8 + 8)) << (pass * 8 + 8)));
  if (pass == 3) return make_ulonglong2(c.x, 0ull);
  const int kp = pass - 4;
  return make_ulonglong2((kp >= 7) ? 0ull : (c.x >> (kp * 8 + 8)) << (kp * 8 + 8), 0ull);
}
__device__ __forceinline__ ulonglong2 CompWithByte(ulonglong2 prefix, int pass, unsigned byte) {
  if (pass < 4) return make_ulonglong2(prefix.x, prefix.y | ((unsigned long long)byte << (pass * 8)));
  return make_ulonglong2(prefix.x | ((unsigned long long)byte << ((pass - 4) * 8)), prefix.y);
}
__device__ __forceinline__ bool CompEq(unsigned long long a, unsigned long long b) { return a == b; }
__device__ __forceinline__ bool CompEq(ulonglong2 a, ulonglong2 b) { return a.x == b.x && a.y == b.y; }
__device__ __forceinline__ bool CompGe(unsigned long long a, unsigned long long b) { return a >= b; }
__device__ __forceinline__ bool CompGe(ulonglong2 a, ulonglong2 b) { return a.x > b.x || (a.x == b.x && a.y >= b.y); }
// width of the predicted score range from the previous frame's top-to-threshold gap (in key units)
__device__ __forceinline__ unsigned long long ReachOf(unsigned gap) { return (5ull * gap) / 4ull + 64ull; }
__device__ __forceinline__ unsigned long long ReachOf(unsigned long long gap) {
  return (gap > (1ull << 62)) ? ~0ull : gap + gap / 4ull + 64ull;
}

// scalar slots in addition to the kV2* / kV3* ones. PC: kV4NChg and kV4MinWiped are pairs, one word per
// round parity (a round reads the pair's one half and writes the other); kV4NAtRisk counts at-risk
// members for the timing build's event counters only.
enum { kV4Utt = 23, kV4Abort = 24, kV4NChg = 25, kV4MinWiped = 27, kV4MaxParent = 29, kV4NAtRisk = 30 };
// timing build: clock64 phase slots 0-19, event counters 20-26 (tools/phase_cycles.py names them)
constexpr int kV4DbgSlots = 27;

// MINB = resident CTAs per SM the register allocation is tuned for: 4 (64 registers) for batches that
// fill the machine, 2 (128 registers: more loads in flight, no re-materialisation) for the latency
// regime of at most two utterances per SM.
// LM = a scorer table is plugged in (util/ctc_beam_scorer.h:31-65 as a [C+1, C] table of expansion
// log-probabilities <= 0): a child's base is old total (or old blank) + lm[previous label + 1][label],
// which breaks the "prefix of the sorted classes" shortcut -- the candidate mask of a row is then built
// by testing all 32 classes.
template <typename IN, int WMAX, int NT, bool TIMING, int MINB, bool LM = false>
__global__ void __launch_bounds__(NT, (TIMING ? 1 : MINB)) BeamKernelV4(BeamParamsT<typename ScoreOf<IN>::type> p) {
  using R = typename ScoreOf<IN>::type;
  using Ops = RealOps<R>;
  using Key = typename Ops::Key;
  using Comp = typename Ops::Comp;
  using Rec = V4Rec<R>;
  using Row = typename Rec::Row;
  using Item = typename Rec::Item;
  constexpr bool kF64 = (sizeof(R) == 8);
  static_assert(!kF64 || (!TIMING && !LM), "the double kernel has no timing / scorer variant");
  static_assert(NT >= WMAX && NT >= kBinsV2, "one thread per beam slot and per histogram bin");
  extern __shared__ __align__(16) unsigned char smem[];
  constexpr int NWARP = NT / 32;
  constexpr int TS = 8 * WMAX;  // parent look-up table slots (load factor <= 1/8: ~97% of the look-ups miss)
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const int W = p.W, C = p.C, T = p.T, B = p.B, blank = p.blank_index;
  const bool s_warp = (warp == NWARP - 1);

  using lay = BeamSmemV4<WMAX, LM, (int)sizeof(R)>;
  unsigned long long* s_hash = (unsigned long long*)(smem + lay::hash);
  unsigned long long* s_phash = (unsigned long long*)(smem + lay::phash);
  Comp* s_sorted = (Comp*)(smem + lay::sorted);
  Comp* s_fin = (Comp*)(smem + lay::fin);
  Comp* s_bnd = (Comp*)(smem + lay::bnd);
  unsigned long long* s_exptab = (unsigned long long*)(smem + lay::exptab);
  unsigned long long* s_exptabd = (unsigned long long*)(smem + lay::exptabd);
  Row* s_row = (Row*)(smem + lay::row);
  Item* c_list = (Item*)(smem + lay::list);
  R* s_total = (R*)(smem + lay::total);
  R* s_blk = (R*)(smem + lay::blk);
  R* s_lab = (R*)(smem + lay::lab);
  R* s_ab = (R*)(smem + lay::ab);
  R* s_an = (R*)(smem + lay::an);
  int* s_label = (int*)(smem + lay::label);
  R* m_nt = (R*)(smem + lay::m_nt);
  R* m_nb = (R*)(smem + lay::m_nb);
  R* m_nl = (R*)(smem + lay::m_nl);
  R* m_nab = (R*)(smem + lay::m_nab);
  R* m_nan = (R*)(smem + lay::m_nan);
  Key* m_key = (Key*)(smem + lay::m_key);
  unsigned* m_rec = (unsigned*)(smem + lay::m_rec);
  int* m_pslot = (int*)(smem + lay::m_pslot);
  int* s_risk = (int*)(smem + lay::risk);
  int* s_con = (int*)(smem + lay::con);
  unsigned* s_wiped = (unsigned*)(smem + lay::wiped);
  int* s_qcnt = (int*)(smem + lay::qcnt);
  unsigned* s_qchg = (unsigned*)(smem + lay::qchg);
  unsigned* s_htab = (unsigned*)(smem + lay::htab);
  unsigned* s_hist = (unsigned*)(smem + lay::hist);
  unsigned* s_offs = (unsigned*)(smem + lay::offs);
  unsigned* s_bins2 = (unsigned*)(smem + lay::bins2);
  unsigned* s_wtot = (unsigned*)(smem + lay::wtot);
  R* s_xb = (R*)(smem + lay::x);
  R* s_plb = (R*)(smem + lay::pl);
  R* s_plSb = (R*)(smem + lay::pls);
  R* s_plHb = (R*)(smem + lay::plh);
  unsigned* s_prefb = (unsigned*)(smem + lay::pref);
  R* s_fsc = (R*)(smem + lay::fsc);
  Key* s_bits = (Key*)(smem + lay::bits);
  R* s_e = (R*)(smem + lay::e);
  volatile int* sc = (volatile int*)(smem + lay::scal);
  int* sci = (int*)(smem + lay::scal);
  unsigned* scu = (unsigned*)(smem + lay::scal);
  Key* s_keys = (Key*)(smem + lay::keys);
  Comp* s_prefix = (Comp*)(smem + lay::prefix);

  LoadExpTable(s_exptab, tid, NT);
  if constexpr (kF64)
    for (int i = tid; i < 256; i += NT) s_exptabd[i] = kCtcxExpTab[i];
  const float* s_lm = (const float*)(smem + lay::lm);
  unsigned valid_mask = 0u;  // LM: the non-blank classes
  if constexpr (LM) {
    float* w_lm = (float*)(smem + lay::lm);
    for (int i = tid; i < 33 * 32; i += NT) {
      const int r = i >> 5, l = i & 31;
      w_lm[r * kLmStride + l] = (r <= C && l < C) ? p.lm[(size_t)r * C + l] : 0.0f;
    }
    valid_mask = ((C >= 32) ? 0xffffffffu : ((1u << C) - 1u)) & ~(1u << blank);
  }

  // thread -> (row, class slice) mapping of the candidate pass
  // (latency regime: the threads share the rows -- two per row at the 128-slot tier, at most four (the
  // 32-slot tier: every thread of a row computes the row's whole mask, and more warps in the list scan
  // mean more atomics; eight per row cost 10 % at beam 32); throughput regime: one thread per row -- the
  // candidate search runs on half as many warps, fewer instructions in total)
  constexpr int PARTS = (MINB >= 4 && !TIMING) ? 1 : (NT / WMAX > 4 ? 4 : NT / WMAX);  // threads per row
  constexpr int CP = 32 / PARTS;    // classes per thread
  static_assert(NT % WMAX == 0 && 32 % PARTS == 0, "row/class tiling");
  const int prow = tid / PARTS, pbase = (tid % PARTS) * CP;
  // thread -> (slot, role) mapping of the beam write-out (PG): role 0 = state + record, role 1 = hash side
  constexpr int PGS = (NT >= 2 * WMAX) ? 2 : 1;
  const int pg_slot = tid % WMAX, pg_role = tid / WMAX;

  // optional per-phase clock64 instrumentation (thread 0), compiled out of the production kernel
  long long cyc[TIMING ? kV4DbgSlots : 1] = {0};
  long long tprev = 0;
  const bool timing = TIMING && (p.dbg_cycles != nullptr) && tid == 0;
#define CTCX_TICK(i)                      \
  if (TIMING && timing) {                 \
    const long long now_ = clock64();     \
    cyc[TIMING ? (i) : 0] += now_ - tprev; \
    tprev = now_;                         \
  }

  int ready_known = (p.ready != nullptr) ? 0 : 0x7fffffff;  // S warp: frames known to have landed

  // Tasks: (time slice, utterance), slice-major -- task q is slice q / B of utterance q % B. With one slice
  // per utterance (batches that fit the resident CTAs, streaming) a task is a whole utterance. Larger
  // batches are cut into p.n_slices slices of p.slice_frames frames so that the CTAs stay evenly loaded
  // to the end (no tail wave, ragged lengths balance): the beam is handed from slice to slice through
  // the per-utterance state block in HBM, and a slice waits for its predecessor's release of
  // p.progress[b]. Every predecessor has a smaller task number, i.e. it is already owned by a resident
  // CTA that waits for nothing later: the wait cannot deadlock.
  const int n_tasks = B * p.n_slices;
  for (;;) {  // ---- persistent loop: one task per iteration ----
    if (tid == 0) sci[kV4Utt] = atomicAdd(p.queue, 1);
    __syncthreads();
    const int task = sci[kV4Utt];
    if (task >= n_tasks) break;
    const int slice = task / B, b = task - slice * B;

    // streaming: frames already consumed by earlier calls; this call contributes up to Lall more
    const int t_done = (p.t_done != nullptr) ? p.t_done[b] : 0;
    const int Lall = max(0, min(p.seq_len[b], p.Tcap - t_done));
    const int t0 = slice * p.slice_frames;  // first frame of this task (within this call's logits)
    if (slice > 0 && t0 >= Lall) {  // the utterance ended in an earlier slice
      __syncthreads();
      continue;
    }
    const int L = min(Lall, t0 + p.slice_frames) - t0;  // frames of this task
    const bool last_slice = (t0 + L == Lall);
    bool resume = (p.state != nullptr) && (t_done > 0 || slice > 0);
    if constexpr (kF64) resume = resume && StreamResumable64(p.state, B, W, b);
    const size_t row0 = (size_t)b * C;  // element offset of (t = 0, b) in the logits tensor
    if (slice > 0) {  // wait for the previous slice of this utterance (acquire), then read its state
      if (tid == 0) {
        int done = 0;
        for (;;) {
          asm volatile("ld.acquire.gpu.global.s32 %0, [%1];\n" : "=r"(done) : "l"(p.progress + b) : "memory");
          if (done >= slice) break;
          __nanosleep(100);
        }
      }
      __syncthreads();
    }

    // S warp: raw logit (lane = class) of frame t, as float. Frames arrive in order; wait for the copy
    // that is still in flight (p.ready counts the frames that have landed).
    auto load_row = [&](int t) -> R {
      if (t >= ready_known) {
        int r = 0;
        if (lane == 0) {
          const long long t0 = clock64();
          for (;;) {
            asm volatile("ld.acquire.sys.global.s32 %0, [%1];\n" : "=r"(r) : "l"(p.ready) : "memory");
            if (r > t) break;
            if (clock64() - t0 > 8000000000ll) { sci[kV4Abort] = 1; r = 0x7fffffff; break; }  // ~4 s: copy lost
            __nanosleep(200);
          }
        }
        ready_known = __shfl_sync(kFull, r, 0);
      }
      return (lane < C) ? LoadRaw<IN>(p.logits, (size_t)t * (size_t)p.tstride + row0 + lane) : (R)0;
    };
    // The S warp prepares frame t+1 in three stages, each placed where the warp has nothing else to do:
    // S1 (while the other warps are in PA): max and the exp-sum of the softmax normaliser (decoder.h:71-80)
    auto prepare1 = [&](R xr, R& mx_out) -> R {
      const bool in_row = lane < C;
      const R mx = Ops::UnKey(WarpMaxKey(in_row ? Ops::KeyOf(xr) : (Key)0));
      if constexpr (kF64) s_e[lane] = in_row ? ExpExactD(Ops::Sub(xr, mx), s_exptabd) : 0.0;
      else s_e[lane] = in_row ? ExpfExact(Ops::Sub(xr, mx), s_exptab) : 0.0f;
      __syncwarp();
      R sum = (R)0;  // index order, as the reference sums (trailing +0 terms leave it unchanged)
      if constexpr (kF64) {
#pragma unroll
        for (int i = 0; i < 32; i += 2) {
          const double2 v = *reinterpret_cast<const double2*>(s_e + i);
          sum = Ops::Add(Ops::Add(sum, v.x), v.y);
        }
      } else {
#pragma unroll
        for (int i = 0; i < 32; i += 4) {
          const float4 v = *reinterpret_cast<const float4*>(s_e + i);
          sum = __fadd_rn(__fadd_rn(__fadd_rn(__fadd_rn(sum, v.x), v.y), v.z), v.w);
        }
      }
      mx_out = mx;
      return sum;
    };
    // S2 (while the other warps list the candidates, PB): the normaliser, per-class log-probs, classes
    // ranked by log-prob. Equal keys keep lane order; the order inside a tie never matters (a prefix of
    // the sorted classes never ends inside a group of equal scores). Returns the lane's rank.
    auto prepare2 = [&](R xr, R mx, R sum, int buf) -> int {
      R logsum;
      if constexpr (kF64) logsum = LogExactD(sum); else logsum = LogfExact(sum);
      const R off = Ops::Add(mx, logsum);
      const bool lane_ok = (lane < C) && (lane != blank);
      const R pl_lane = lane_ok ? Ops::Sub(xr, off) : (R)0;
      s_xb[buf * 32 + lane] = xr;
      s_plb[buf * 32 + lane] = pl_lane;
      const Key key = lane_ok ? Ops::KeyOf(pl_lane) : (Key)0;  // blank / padding sort last
      s_bits[lane] = key;  // the keys of the row, read back as broadcasts
      if (lane == 0) s_fsc[buf * 4 + 0] = off;
      __syncwarp();
      int rank = 0;
      if constexpr (kF64) {
#pragma unroll
        for (int i = 0; i < 32; i += 2) {
          const ulonglong2 k = *reinterpret_cast<const ulonglong2*>(s_bits + i);
          rank += (k.x > key) ? 1 : 0;
          rank += (k.y > key) ? 1 : 0;
        }
      } else {
#pragma unroll
        for (int i = 0; i < 32; i += 4) {
          const uint4 k = *reinterpret_cast<const uint4*>(s_bits + i);
          rank += (k.x > key) ? 1 : 0;
          rank += (k.y > key) ? 1 : 0;
          rank += (k.z > key) ? 1 : 0;
          rank += (k.w > key) ? 1 : 0;
        }
      }
      rank += __popc(__match_any_sync(kFull, key) & ((1u << lane) - 1u));
      s_plSb[buf * 32 + rank] = lane_ok ? pl_lane : Ops::NegInf();
      if ((rank & 3) == 0) s_plHb[buf * 8 + (rank >> 2)] = lane_ok ? pl_lane : Ops::NegInf();
      return rank;
    };
    // S3 (while the other warps write the next beam, PG): prefix masks of the sorted classes
    auto prepare3 = [&](int rank, int buf) {
      const bool lane_ok = (lane < C) && (lane != blank);
      unsigned* bpref = s_prefb + buf * 36;
      unsigned* cbits = reinterpret_cast<unsigned*>(s_bits);  // (the sort keys are no longer needed)
      __syncwarp();
      cbits[rank] = lane_ok ? (1u << lane) : 0u;
      __syncwarp();
      unsigned incl = cbits[lane];
#pragma unroll
      for (int o = 1; o < 32; o <<= 1) {
        const unsigned v = __shfl_up_sync(kFull, incl, o);
        if (lane >= o) incl |= v;
      }
      bpref[lane + 1] = incl;
      const int cv = __popc(__ballot_sync(kFull, lane_ok));
      __syncwarp();
      if (lane == 0) {
        bpref[0] = 0u;
        s_fsc[buf * 4 + 1] = (cv > 0) ? s_plSb[buf * 32] : Ops::NegInf();
        s_fsc[buf * 4 + 2] = (cv > 0) ? s_plSb[buf * 32 + cv - 1] : (R)0;
      }
    };

    // ---- initial state: the root (decoder.h:212-227) ----
    for (int i = tid; i < TS; i += NT) s_htab[i] = 0xffffffffu;
    for (int i = tid; i < WMAX; i += NT) {
      s_wiped[i] = 0u;
      s_row[i] = Rec::MakeRow((R)0, (R)0, 0);
    }
    for (int i = tid; i < kBinsV2; i += NT) s_hist[i] = 0u;
    if (tid == 0) {
      if (!resume) {
        s_total[0] = (R)0;
        s_blk[0] = (R)0;
        s_lab[0] = Ops::NegInf();
        s_ab[0] = (R)0;  // empty alignment with probability 1 (entry.h:204-209)
        s_an[0] = Ops::NegInf();
        s_label[0] = -1;
        s_hash[0] = kRootHash;
        s_phash[0] = 0ull;
      }
      sci[kV2Anomaly] = 0;
      sci[kV2NCand] = 0;
      sci[kV2NRisk] = 0;
      sci[kV4NChg] = 0;
      sci[kV4MinWiped] = 0x7fffffff;
      sci[kV4MaxParent] = -1;
      sci[kV4NAtRisk] = 0;
      s_keys[kV4KMin] = Ops::kKeyMax;
      s_keys[kV4KMax] = (Key)0;
      sci[kV2NBnd] = 0;
      s_keys[kV4KMinBase] = Ops::kKeyMax;
      s_keys[kV4KGap] = (Key)0;
      sci[kV3Found] = 0;
      sci[kV4Abort] = 0;
    }
    int n = 1;
    R xr_next = (R)0;  // S warp: raw row of the frame after the one being prepared
    R s_xr = (R)0, s_mx = (R)0, s_sum = (R)0;  // S warp: the row being prepared, between the stages
    int s_rank = 0;
    if (s_warp && L > 0) {
      const R x0 = load_row(t0);
      if (L > 1) xr_next = load_row(t0 + 1);
      const R sum0 = prepare1(x0, s_mx);
      prepare3(prepare2(x0, s_mx, sum0, 0), 0);
    }
    __syncthreads();
    int carried = 0;  // flag bits handed on from the previous slice / call
    if (resume) {  // beam as the previous slice left it (buffer 0: local frame 0 reads buffer 0)
      const StreamViewT<R> sv = StreamBlock<R>(p.state, B, W, b);
      n = __ldcg(&sv.hdr->n);
      carried = __ldcg(&sv.hdr->flags);
      for (int i = tid; i < n; i += NT) {  // (L2 loads: another SM wrote the block)
        s_total[i] = __ldcg(sv.total + i); s_blk[i] = __ldcg(sv.blk + i); s_lab[i] = __ldcg(sv.lab + i);
        s_ab[i] = __ldcg(sv.ab + i); s_an[i] = __ldcg(sv.an + i); s_label[i] = __ldcg(sv.label + i);
        s_hash[i] = __ldcg(sv.hash + i); s_phash[i] = __ldcg(sv.phash + i);
      }
      if (tid == 0) {
        s_keys[kV4KGap] = __ldcg(&sv.hdr->gap);
        sci[kV2Anomaly] = carried & 1;
      }
      __syncthreads();
    }
    for (int i = tid; i < n; i += NT) {  // row info + parent look-up table of the initial beam
      s_row[i] = Rec::MakeRow(s_total[i], s_blk[i], s_label[i]);
      const unsigned long long hsh = s_hash[i];
      unsigned h = (unsigned)hsh & (TS - 1);
      const unsigned entry = ((unsigned)(hsh >> 42) << 10) | (unsigned)i;
      while (atomicCAS(&s_htab[h], 0xffffffffu, entry) != 0xffffffffu) h = (h + 1) & (TS - 1);
    }
    __syncthreads();

    if (timing) tprev = clock64();
    int t_end = L;  // frames actually consumed (smaller only if the input copy was lost)
    for (int t = 0; t < L; ++t) {
      const int cur = t & 1, nxt = cur ^ 1;
      const R* x = s_xb + cur * 32;
      const R* s_pl = s_plb + cur * 32;
      const R* s_plS = s_plSb + cur * 32;
      const R* s_plH = s_plHb + cur * 8;
      const unsigned* s_pref = s_prefb + cur * 36;
      const R off = s_fsc[cur * 4 + 0];
      const R* o_total = s_total + cur * WMAX;
      const R* o_blk = s_blk + cur * WMAX;
      const R* o_lab = s_lab + cur * WMAX;
      const R* o_ab = s_ab + cur * WMAX;
      const R* o_an = s_an + cur * WMAX;
      const int* o_label = s_label + cur * WMAX;
      const unsigned long long* o_hash = s_hash + cur * WMAX;
      const unsigned long long* o_phash = s_phash + cur * WMAX;

      // ---- S: the last warp prepares frame t+1 (and puts row t+2 in flight) while the others run PA ----
      if (s_warp && t + 1 < L) {
        s_xr = xr_next;
        if (t + 2 < L) xr_next = load_row(t0 + t + 2);
        s_sum = prepare1(s_xr, s_mx);
      }
      const R xb = x[blank];
      const R pb = Ops::Sub(xb, off);
      CTCX_TICK(7)  // frame setup
      // ---- PA: update the existing members (decoder.h:95-143) ----
      Key my_key = (Key)0;
      bool suspect = false;
      if (tid < n) {
        const int i = tid;
        const int lbl = o_label[i];
        int pslot = -1;
        R v_nl = o_lab[i], v_an = Ops::NegInf();
        R rescore = Ops::NegInf();  // what the parent's re-score of this member would be (decoder.h:172-182)
        unsigned an_kind = kAnNone, an_src = 0xffu;
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
          const R xl = x[lbl];
          const R pl = Ops::Sub(xl, off);
          const R self_an = Ops::Add(o_an[i], pl);
          if (pslot >= 0) {
            const bool same = (lbl == o_label[pslot]);
            R base = same ? o_blk[pslot] : o_total[pslot];
            if constexpr (LM) base = Ops::Add(base, s_lm[(o_label[pslot] + 1) * kLmStride + lbl]);  // decoder.h:103,114
            v_nl = Ops::Sub(Ops::Add(LogSumExp(o_lab[i], base, s_exptab), xl), off);
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
            v_nl = Ops::Add(o_lab[i], pl);
            v_an = self_an;
            an_kind = kAnSelfAn;
            an_src = (unsigned)i;
          }
        }
        CTCX_TICK(9)  // first LSE + alignment candidates
        const R v_nb = Ops::Sub(Ops::Add(o_total[i], xb), off);
        const R c1 = Ops::Add(o_ab[i], pb), c2 = Ops::Add(o_an[i], pb);
        const unsigned ab_kind = (c2 > c1) ? kAbFromAn : kAbFromAb;
        const R v_nt = LogSumExp(v_nb, v_nl, s_exptab);
        CTCX_TICK(10)  // second LSE
        m_nt[i] = v_nt;
        m_nb[i] = v_nb;
        m_nl[i] = v_nl;
        m_nab[i] = (c2 > c1) ? c2 : c1;
        m_nan[i] = v_an;
        my_key = Ops::KeyOf(v_nt);
        m_key[i] = my_key;
        m_rec[i] = PackRec32((unsigned)i, an_src, ab_kind, an_kind, (unsigned)(lbl & 0xff));
        m_pslot[i] = pslot;
        // Precondition of the one event that is reported instead of modelled (DESIGN.md "Known deviation"):
        // were this member evicted and then re-scored by its parent, rounding would put the re-score ABOVE
        // the member's own total, so the reference could accept it again (decoder.h:189-199; it does so only
        // when the beam bottom ties with that total). Mathematically total >= re-score always. The utterance
        // is flagged if such a member then drops out of the beam (after the selection, below).
        suspect = Ops::KeyOf(rescore) > my_key;
        if (pslot >= 0) {
          atomicOr(Rec::MaskPtr(&s_row[pslot]), 1u << lbl);
          if (pslot < i) {
            atomicMax(&sci[kV4MaxParent], pslot);
            if constexpr (TIMING) atomicAdd(&sci[kV4NAtRisk], 1);
            // A wipe query counts the members ranking before this one (fewer than n <= W) plus the
            // children above v_nt. No child can be: a child's base is a row's old total, or its old blank
            // mass, which is never above it; row 0 holds the largest old total; fp addition is monotone.
            // So a member above lp_max + o_total[0] is never wiped and is not listed. (The scorer's
            // table adds an entry to the base; its sign is not checked on every path, so LM lists all.)
            if (LM || !(v_nt > Ops::Add(s_fsc[cur * 4 + 1], o_total[0]))) {
              const int q = atomicAdd(&sci[kV2NRisk], 1);
              s_risk[q] = i;
            }
          }
        }
      }
      CTCX_TICK(11)  // stores + atomics
      {
        const Key kmin = WarpMinKey((tid < n) ? my_key : Ops::kKeyMax);
        const Key kmax = WarpMaxKey((tid < n) ? my_key : (Key)0);
        if (lane == 0 && warp * 32 < n) {
          atomicMin(&s_keys[kV4KMin], kmin);
          atomicMax(&s_keys[kV4KMax], kmax);
        }
      }
      CTCX_TICK(12)  // min/max reduction
      if (__builtin_expect(n < W, 0)) {  // beam not full: every finite child is admissible; bound the score range
        Key kb = Ops::kKeyMax;
        if (tid < n) {
          const R ob = o_blk[tid], ot = o_total[tid];
          if (ot > Ops::NegInf()) kb = Ops::KeyOf((ob > Ops::NegInf()) ? fmin(ot, ob) : ot);
        }
        kb = WarpMinKey(kb);
        if (lane == 0 && warp * 32 < n) atomicMin(&s_keys[kV4KMinBase], kb);
      }
      __syncthreads();
      CTCX_TICK(0)  // PA
      const int n_risk = sci[kV2NRisk];

      // Candidates of one row above a threshold, as a class bitmask. The classes are sorted by
      // log-prob and fp addition is monotone, so "(x_l - off) + old total > thr" holds exactly for a
      // prefix of the sorted order: 2-round exact search, then drop the classes that are already
      // members (decoder.h:168) and re-test the repeated label, whose base is the old blank
      // probability (decoder.h:172-177).
      auto cand_mask = [&](const Row ri, const R thr, const int c_lo = 0, const int c_n = 32) -> unsigned {
        const R ot = Rec::Ot(ri);
        if constexpr (LM) {  // every class of [c_lo, c_lo + c_n) on its own: score = pl + (base + lm)  (decoder.h:171-182)
          const float ob = Rec::Ob(ri);
          const int lb = Rec::Label(ri);
          const float* lmrow = s_lm + (lb + 1) * kLmStride;
          unsigned m = 0u;
#pragma unroll 2
          for (int g = c_lo; g < c_lo + c_n; g += 4) {
            const float4 q = *reinterpret_cast<const float4*>(s_pl + g);
            const float4 e = *reinterpret_cast<const float4*>(lmrow + g);
            m |= (__fadd_rn(q.x, __fadd_rn((g == lb) ? ob : ot, e.x)) > thr) ? (1u << g) : 0u;
            m |= (__fadd_rn(q.y, __fadd_rn((g + 1 == lb) ? ob : ot, e.y)) > thr) ? (2u << g) : 0u;
            m |= (__fadd_rn(q.z, __fadd_rn((g + 2 == lb) ? ob : ot, e.z)) > thr) ? (4u << g) : 0u;
            m |= (__fadd_rn(q.w, __fadd_rn((g + 3 == lb) ? ob : ot, e.w)) > thr) ? (8u << g) : 0u;
          }
          return m & valid_mask & ~Rec::Mask(ri);
        }
        // prefix length = number of sorted scores above thr (the predicate is monotone): first the
        // heads of the 8 groups of 4, then the group itself. -inf padding never passes.
        int g = 0, pos = 0;
        if constexpr (kF64) {
#pragma unroll
          for (int i = 0; i < 8; i += 2) {
            const double2 h = *reinterpret_cast<const double2*>(s_plH + i);
            g += (Ops::Add(h.x, ot) > thr) ? 1 : 0;
            g += (Ops::Add(h.y, ot) > thr) ? 1 : 0;
          }
          if (g > 0) {  // group g-1 is the last one whose head passes
            const double2 qa = *reinterpret_cast<const double2*>(s_plS + 4 * (g - 1));
            const double2 qb = *reinterpret_cast<const double2*>(s_plS + 4 * (g - 1) + 2);
            pos = 4 * (g - 1) + 1;
            pos += (Ops::Add(qa.y, ot) > thr) ? 1 : 0;
            pos += (Ops::Add(qb.x, ot) > thr) ? 1 : 0;
            pos += (Ops::Add(qb.y, ot) > thr) ? 1 : 0;
          }
        } else {
          const float4 ha = *reinterpret_cast<const float4*>(s_plH), hb = *reinterpret_cast<const float4*>(s_plH + 4);
          g += (__fadd_rn(ha.x, ot) > thr) ? 1 : 0;
          g += (__fadd_rn(ha.y, ot) > thr) ? 1 : 0;
          g += (__fadd_rn(ha.z, ot) > thr) ? 1 : 0;
          g += (__fadd_rn(ha.w, ot) > thr) ? 1 : 0;
          g += (__fadd_rn(hb.x, ot) > thr) ? 1 : 0;
          g += (__fadd_rn(hb.y, ot) > thr) ? 1 : 0;
          g += (__fadd_rn(hb.z, ot) > thr) ? 1 : 0;
          g += (__fadd_rn(hb.w, ot) > thr) ? 1 : 0;
          if (g > 0) {  // group g-1 is the last one whose head passes
            const float4 q = *reinterpret_cast<const float4*>(s_plS + 4 * (g - 1));
            pos = 4 * (g - 1) + 1;
            pos += (__fadd_rn(q.y, ot) > thr) ? 1 : 0;
            pos += (__fadd_rn(q.z, ot) > thr) ? 1 : 0;
            pos += (__fadd_rn(q.w, ot) > thr) ? 1 : 0;
          }
        }
        unsigned m = s_pref[pos] & ~Rec::Mask(ri);
        const int lb = Rec::Label(ri);
        if (lb >= 0 && ((m >> lb) & 1u) && !(Ops::Add(s_pl[lb], Rec::Ob(ri)) > thr)) m &= ~(1u << lb);
        return m;
      };

      // ---- PC: revisit-wipe fixed point (SURVEY A.4) ----
      // Round 1 counts, for every at-risk member, the items the parent's sweep meets before it (one warp
      // per member). When verdicts wipe rows, the counts are not recomputed: a later round only adds or
      // removes the contribution of the rows whose state CHANGED -- one thread per (member, changed row)
      // pair -- and re-derives the verdicts; a handful of candidate tests instead of a full sweep each.
      int fp_contested = 0, fp_rounds = 0;  // timing build: contested members, verdict derivations
      if (__builtin_expect(n_risk > 0, 0)) {
        // Round 1 counts with no row wiped; a later round only subtracts wiped rows or adds restored ones
        // back, so no count ever exceeds its round-1 value. A member whose round-1 count is below W is
        // therefore a final survivor and its row never changes state. Only the others, the contested
        // members, take part in later rounds: round 1 wipes them all (no parent is wiped yet), lists them
        // as the rows that changed, and thread k owns the verdict of contested member k from then on.
        for (int q = warp; q < n_risk; q += NWARP) {  // round 1: one warp per at-risk member (nothing is wiped yet)
          const int m = s_risk[q];
          const int pslot = m_pslot[m];
          const Key vkey = m_key[m];
          const R v = m_nt[m];
          int cnt = 0;
          for (int j = lane; j < n; j += 32) {  // members ranking before m
            const Key kj = m_key[j];
            cnt += (kj > vkey || (kj == vkey && j < m)) ? 1 : 0;
          }
          // children visited before the parent reaches label(m)
          const unsigned below = (1u << o_label[m]) - 1u;
#pragma unroll 1
          for (int r0 = 0; r0 <= pslot; r0 += 32) {
            const int r = r0 + lane;
            if (r <= pslot) {
              unsigned mk = cand_mask(s_row[r], v);
              if (r == pslot) mk &= below;
              cnt += __popc(mk);
            }
          }
          cnt = __reduce_add_sync(kFull, cnt);
          if (lane == 0 && cnt >= W) {
            const int k = atomicAdd(&sci[kV4NChg], 1);
            s_con[k] = m;
            s_qcnt[k] = cnt;
            s_qchg[k] = ((unsigned)m << 1) | 1u;
            s_wiped[m] = 1u;  // (round 1 reads no wiped state)
            atomicMin(&sci[kV4MinWiped], m);
          }
        }
        __syncthreads();
        const int n_con = sci[kV4NChg];
        if (TIMING) {
          fp_contested = n_con;
          fp_rounds = 1;
        }
        // Rounds after the first. Words [par] hold the last round's changes; the apply step writes [par ^ 1].
        for (int par = 0;; par ^= 1) {
          // a query only counts rows up to its parent's: if every wiped row lies beyond every parent
          // row, no count (and no parent) is affected and the verdicts are final (no contested member: no
          // wiped row)
          if (sci[kV4MinWiped + par] > sci[kV4MaxParent]) break;  // (max over every at-risk member, listed or not)
          const int n_chg = sci[kV4NChg + par];
          const bool parent_wiped = (tid < n_con) && s_wiped[m_pslot[s_con[tid]]] != 0u;
          for (int pr = tid; pr < n_con * n_chg; pr += NT) {  // one (contested member, changed row) pair per thread
            const int k = pr / n_chg, c = pr - k * n_chg;
            const unsigned e = s_qchg[c];
            const int r = (int)(e >> 1);
            const int m = s_con[k];
            const int pslot = m_pslot[m];
            if (r <= pslot) {
              unsigned mk = cand_mask(s_row[r], m_nt[m]);
              if (r == pslot) mk &= (1u << o_label[m]) - 1u;
              const int d = __popc(mk);
              if (d) atomicAdd(&s_qcnt[k], (e & 1u) ? -d : d);  // wiped rows stop counting, restored ones count again
            }
          }
          if (tid == 0) {  // nobody reads these words again before the next barrier
            sci[kV4NChg + (par ^ 1)] = 0;
            sci[kV4MinWiped + (par ^ 1)] = 0x7fffffff;
          }
          __syncthreads();
          if (TIMING) ++fp_rounds;
          bool changed = false;
          if (tid < n_con) {  // re-derive the verdict, apply it, list the row if it changed
            const int m = s_con[tid];  // (only this thread writes s_wiped[m] after round 1)
            const unsigned nv = (!parent_wiped && s_qcnt[tid] >= W) ? 1u : 0u;  // a wiped parent never sweeps (decoder.h:167)
            if (nv != s_wiped[m]) {
              changed = true;
              s_wiped[m] = nv;
              s_qchg[atomicAdd(&sci[kV4NChg + (par ^ 1)], 1)] = ((unsigned)m << 1) | nv;
            }
            if (nv) atomicMin(&sci[kV4MinWiped + (par ^ 1)], m);
          }
          if (!__syncthreads_or(changed)) break;
        }
      }
      CTCX_TICK(2)  // PC

      // ---- S, second and third part: normaliser, log-probs, class ranks and prefix masks of frame t+1,
      // while the others list the candidates ----
      if (s_warp && t + 1 < L) {
        s_rank = prepare2(s_xr, s_mx, s_sum, nxt);
        prepare3(s_rank, nxt);
      }

      // ---- PB / PD: list + histogram of the items in the score range, boundary bin ----
      const Key minkey_m = s_keys[kV4KMin];
      const R lp_max = s_fsc[cur * 4 + 1];
      Key lo_true;  // no item lies below this key
      if (n == W) {
        lo_true = minkey_m;  // decoder.h:151-155: nothing at or below the W-th member total is admitted
      } else {
        const Key kb = s_keys[kV4KMinBase];
        Key lo_c = minkey_m;
        if (kb != Ops::kKeyMax) lo_c = Ops::KeyOf(Ops::Add(Ops::UnKey(kb), s_fsc[cur * 4 + 2]));
        lo_true = max(min(minkey_m, lo_c), Ops::kKeyNegInf);
      }
      // every item is <= max(best member, best possible child); old totals are sorted, slot 0 is the max
      const Key hi_key = max(s_keys[kV4KMax], Ops::KeyOf(Ops::Add(lp_max, o_total[0])));
      Key lo_key = lo_true;
      int shift = 0;
      bool clamped = false;
      int n_cand = 0;
      auto bucket_of = [&](Key key) -> int { return (key > lo_key) ? (int)((key - lo_key) >> shift) : 0; };
      for (int attempt = 0; attempt < 2; ++attempt) {
        // Score range of the histogram. Survivors crowd near the top while the admissible range reaches
        // far below, so the first attempt only looks at [hi - 1.25*gap - 64, hi], gap = the previous
        // frame's top-to-threshold distance; if fewer than W items live there the second attempt
        // takes the whole admissible range. The prediction affects speed only.
        lo_key = lo_true;
        if (attempt == 0 && n == W) {
          const Key gap = s_keys[kV4KGap];
          const unsigned long long reach = ReachOf(gap);  // 1.25 x gap + 64; measured: 1.0-1.25 x gap is best, below 1.0 it always misses
          if (gap != (Key)0 && reach < (unsigned long long)(hi_key - lo_true)) lo_key = hi_key - (Key)reach;
        }
        clamped = (lo_key != lo_true);
        const Key span = hi_key - lo_key;
        shift = max(0, Ops::Bits(span | (Key)1) - kBinsLog2V2);  // (key - lo) >> shift < kBinsV2
        const R thr = (n == W) ? Ops::UnKey(lo_key) : Ops::NegInf();  // listed children: score > thr
        const bool member_in = !clamped || my_key > lo_key;
        CTCX_TICK(16)  // PB: range

        // PB pass 1: admissible classes of this thread's (row, class slice). A warp whose rows all lie
        // beyond the beam (the S warp at beam widths up to 112, for one) has nothing to list.
        const bool warp_has_rows = ((warp * 32) / PARTS) < n;
        unsigned mymask = 0u;
        R r_ot = (R)0, r_ob = (R)0;
        int r_label = -1;
        if (prow < n && !s_wiped[prow]) {
          const Row ri = s_row[prow];
          r_ot = Rec::Ot(ri);
          r_ob = Rec::Ob(ri);
          r_label = Rec::Label(ri);
          if (Ops::Add(lp_max, r_ot) > thr) {
            const unsigned m = cand_mask(ri, thr, pbase, CP) >> pbase;
            mymask = (CP == 32) ? m : (m & ((1u << (CP & 31)) - 1u));
          }
        }
        CTCX_TICK(17)  // PB: masks
        int pos0 = 0;
        if (warp_has_rows && __any_sync(kFull, mymask != 0u)) {  // (warp-uniform) somebody has something to list
          const int cnt = __popc(mymask);
          int incl = cnt;
#pragma unroll
          for (int o = 1; o < 32; o <<= 1) {
            const int v = __shfl_up_sync(kFull, incl, o);
            if (lane >= o) incl += v;
          }
          // list positions: one shared-memory atomic per warp (the order of the list does not matter)
          int base = 0;
          if (lane == 31 && incl) base = atomicAdd(&sci[kV2NCand], incl);
          base = __shfl_sync(kFull, base, 31);
          pos0 = base + incl - cnt;
        }
        CTCX_TICK(18)  // PB: scan
        // PB pass 2: list + histogram
        {
          unsigned m = mymask;
          int pos = pos0;
          while (m) {
            const int k = __ffs(m) - 1;
            m &= m - 1u;
            const int l = pbase + k;
            R cbase = (l == r_label) ? r_ob : r_ot;
            if constexpr (LM) cbase = Ops::Add(cbase, s_lm[(r_label + 1) * kLmStride + l]);
            const Key key = Ops::KeyOf(Ops::Add(s_pl[l], cbase));  // :172-182
            c_list[pos++] = Rec::MakeItem(key, ((unsigned)prow << 16) | (unsigned)l);
            atomicAdd(&s_hist[bucket_of(key)], 1u);
          }
          if (tid < n && member_in) atomicAdd(&s_hist[bucket_of(my_key)], 1u);
        }
        CTCX_TICK(19)  // PB: list
        __syncthreads();
        n_cand = sci[kV2NCand];
        CTCX_TICK(1)  // PB

        // ---- PD: boundary bin of the W-th item and group offsets: one bin per thread ----
        // Thread d (0..255) owns bin 255 - d, so an inclusive PREFIX scan in thread order is a SUFFIX
        // scan in bin order: warp scan, per-warp totals through shared memory, one barrier.
        static_assert(kBinsV2 == 256 && NT >= 256, "one bin per thread");
        unsigned pd_h = 0u, pd_incl = 0u;
        const int pd_bin = kBinsV2 - 1 - tid;
        if (tid < kBinsV2) {
          pd_h = s_hist[pd_bin];
          pd_incl = pd_h;
#pragma unroll
          for (int o = 1; o < 32; o <<= 1) {
            const unsigned v = __shfl_up_sync(kFull, pd_incl, o);
            if (lane >= o) pd_incl += v;
          }
          const unsigned nz = __ballot_sync(kFull, pd_h != 0u);
          if (lane == 31) {
            s_wtot[warp] = pd_incl;
            s_wtot[8 + warp] = nz ? (unsigned)(kBinsV2 - 1 - (warp * 32 + (__ffs(nz) - 1))) : 0xffffffffu;  // highest non-empty bin of the warp
          }
        }
        __syncthreads();
        if (tid < kBinsV2) {
          const uint4 wa = *reinterpret_cast<const uint4*>(s_wtot), wb = *reinterpret_cast<const uint4*>(s_wtot + 4);
          const unsigned wt[8] = {wa.x, wa.y, wa.z, wa.w, wb.x, wb.y, wb.z, wb.w};
          unsigned before = 0u, total = 0u;
#pragma unroll
          for (int q = 0; q < 8; ++q) {
            before += (q < warp) ? wt[q] : 0u;
            total += wt[q];
          }
          const unsigned above = before + pd_incl - pd_h;  // items in bins above this thread's
          s_offs[pd_bin] = above;
          s_hist[pd_bin] = 0u;  // counters in PE / next attempt
          // with a clamped range the cut is valid only if the W-th item lies inside the range
          const bool usable = !clamped || (int)total >= W;
          const int K = min(W, (int)total);
          if (usable && (int)(above + pd_h) >= K && (int)above < K) {  // the boundary bin
            const uint4 ta = *reinterpret_cast<const uint4*>(s_wtot + 8), tb = *reinterpret_cast<const uint4*>(s_wtot + 12);
            const unsigned tops[8] = {ta.x, ta.y, ta.z, ta.w, tb.x, tb.y, tb.z, tb.w};
            int topbin = -1;
#pragma unroll
            for (int q = 7; q >= 0; --q)
              if (tops[q] != 0xffffffffu) topbin = (int)tops[q];  // warp 0 owns the highest bins
            sci[kV2Bstar] = pd_bin;
            sci[kV2KRem] = K - (int)above;
            sci[kV2E] = (int)pd_h;
            sci[kV2NNew] = K;
            sci[kV2TopBin] = topbin;
            sci[kV3Found] = 1;
          }
        }
        __syncthreads();
        CTCX_TICK(3)  // PD
        if (__builtin_expect(sc[kV3Found] != 0, 1)) break;  // otherwise the prediction missed: run again over the full range
        if (tid == 0) sci[kV2NCand] = 0;  // the list is rebuilt
        __syncthreads();
      }
      const bool member_in = !clamped || my_key > lo_key;
      const int bstar = sc[kV2Bstar], k_rem = sc[kV2KRem], e_b = sc[kV2E], n_new = sc[kV2NNew];
      if (TIMING && timing) {  // event counters (slots 20-26): how selective would a "below the cut" filter be?
        int below = 0, wiped = 0;
        for (int q = 0; q < n_risk; ++q) {  // (the members PA listed; the others are never wiped)
          const int m = s_risk[q];
          below += (bucket_of(m_key[m]) <= bstar || (clamped && m_key[m] <= lo_key)) ? 1 : 0;
          wiped += s_wiped[m] ? 1 : 0;
        }
        const int at_risk = sci[kV4NAtRisk];
        cyc[TIMING ? 20 : 0] += at_risk;
        cyc[TIMING ? 21 : 0] += below;
        cyc[TIMING ? 22 : 0] += wiped;
        cyc[TIMING ? 23 : 0] += (at_risk > 0) ? 1 : 0;
        cyc[TIMING ? 24 : 0] += n_risk;                                   // listed by PA
        cyc[TIMING ? 25 : 0] += fp_contested;
        cyc[TIMING ? 26 : 0] += fp_rounds;
      }
      // a suspect member (see PA) that is not certain to stay in the beam: report the utterance
      if (__builtin_expect(suspect, 0) && (!member_in || bucket_of(my_key) <= bstar)) sci[kV2Anomaly] = 1;
      const bool bnd_all = (e_b == k_rem);
      // next frame's range prediction: the measured top-to-threshold gap
      const Key gap_next = (Key)(unsigned)(sc[kV2TopBin] - bstar + 1) << shift;

      // ---- PE: scatter every item at or above the boundary bin into its score group ----
      auto place = [&](Key key, unsigned okey) {
        const int bucket = bucket_of(key);
        const Comp comp = Ops::MakeComp(key, ~okey);
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
        Item e[4];
#pragma unroll
        for (int u = 0; u < 4; ++u) {
          const int c = c0 + u * NT;
          e[u] = (c < n_cand) ? c_list[c] : Rec::NoItem();
        }
#pragma unroll
        for (int u = 0; u < 4; ++u)
          if (Rec::ItemKey(e[u])) place(Rec::ItemKey(e[u]), 0x80000000u | Rec::ItemId(e[u]));
      }
      __syncthreads();
      CTCX_TICK(4)  // PE

      // ---- PF: cut the boundary bin exactly ----
      // Usual case (at most 32 items in the boundary bin): the LAST warp ranks them with shuffles and
      // writes the k_rem best straight into their final positions, while the other warps already rank
      // the groups above the boundary (PG) -- no barrier between the two phases.
      const bool pf_fast = !bnd_all && e_b <= kBndFast;
      const int bnd_start = pf_fast ? (int)s_offs[bstar] : 0x7fffffff;  // slots from here on are set by PF
      if (!bnd_all) {
        if (__builtin_expect(e_b <= kBndFast, 1)) {
          if (s_warp) {
            const Comp mine = (lane < e_b) ? s_bnd[lane] : Ops::MakeComp((Key)0, 0u);
            int rank = 0;
            for (int j = 0; j < e_b; ++j) rank += Ops::Greater(ShflComp(mine, j), mine) ? 1 : 0;
            if (lane < e_b && rank < k_rem) s_fin[s_offs[bstar] + rank] = mine;
          }
        } else {
          // many items in the boundary bin (coarse bins after a missed prediction, or pathological
          // ties such as constant logits): radix select of the k_rem largest (key, ~order) composites
          auto for_each_bnd = [&](auto&& f) {
            if (tid < n && member_in && bucket_of(my_key) == bstar)
              f(Ops::MakeComp(my_key, ~(unsigned)tid), my_key, (unsigned)tid);
            for (int c = tid; c < n_cand; c += NT) {
              const Item e = c_list[c];
              const Key ek = Rec::ItemKey(e);
              if (ek && bucket_of(ek) == bstar)
                f(Ops::MakeComp(ek, ~(0x80000000u | Rec::ItemId(e))), ek, 0x80000000u | Rec::ItemId(e));
            }
          };
          constexpr int npass = (int)sizeof(Key) + 4;  // bytes of a (key, ~order) composite
          if (tid == 0) { *s_prefix = Ops::MakeComp((Key)0, 0u); sci[kV2K] = k_rem; }
          __syncthreads();
          for (int pass = npass - 1; pass >= 0; --pass) {
            unsigned* bins = s_bins2;
            for (int i = tid; i < 256; i += NT) bins[i] = 0u;
            __syncthreads();
            const Comp prefix = *s_prefix;  // the bytes above `pass` of the composite being selected
            for_each_bnd([&](Comp v, Key, unsigned) {
              if (CompEq(CompAbove(v, pass), prefix)) atomicAdd(&bins[CompByte(v, pass)], 1u);
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
                    *s_prefix = CompWithByte(prefix, pass, (unsigned)(lane * 8 + q));
                    sci[kV2K] = k - (int)acc;
                  }
                  acc += h[q];
                }
              }
            }
            __syncthreads();
          }
          const Comp cut = *s_prefix;
          for_each_bnd([&](Comp v, Key, unsigned) {
            if (CompGe(v, cut)) {
              const unsigned pos = s_offs[bstar] + atomicAdd(&s_hist[bstar], 1u);
              if (pos < (unsigned)WMAX) s_sorted[pos] = v;
            }
          });
          __syncthreads();
        }
      }

      CTCX_TICK(5)  // PF
      // ---- PG: rank inside the score group = new slot; write the next beam + back-pointers ----
      {
        R* w_total = s_total + nxt * WMAX;
        R* w_blk = s_blk + nxt * WMAX;
        R* w_lab = s_lab + nxt * WMAX;
        R* w_ab = s_ab + nxt * WMAX;
        R* w_an = s_an + nxt * WMAX;
        int* w_label = s_label + nxt * WMAX;
        unsigned long long* w_hash = s_hash + nxt * WMAX;
        unsigned long long* w_phash = s_phash + nxt * WMAX;
        // clear the parent look-up table (this frame's look-ups happened in PA) before re-filling it
        for (int i = tid; i < TS / 4; i += NT)  // 16-byte stores
          reinterpret_cast<uint4*>(s_htab)[i] = make_uint4(0xffffffffu, 0xffffffffu, 0xffffffffu, 0xffffffffu);
        // survivors above the boundary (and the radix-selected boundary items): scatter to the final slot
        const int n_grouped = min(n_new, bnd_start);
        if (tid < n_grouped) {
          const Comp comp = s_sorted[tid];
          const int bucket = bucket_of(Ops::CompKey(comp));
          const int g0 = (int)s_offs[bucket];
          const int g1 = (bucket == bstar && !bnd_all) ? n_new : g0 + (int)s_hist[bucket];
          // Groups usually hold 1-3 items; quantised logits (bfloat16 inputs) make exact ties, i.e. groups of
          // dozens: four independent loads per round keep the count off the shared-memory latency.
          int rank = 0, j = g0;
#pragma unroll 1
          for (; j + 4 <= g1; j += 4) {
            const Comp a = s_sorted[j], b2 = s_sorted[j + 1], c2 = s_sorted[j + 2], d2 = s_sorted[j + 3];
            rank += (Ops::Greater(a, comp) ? 1 : 0) + (Ops::Greater(b2, comp) ? 1 : 0) + (Ops::Greater(c2, comp) ? 1 : 0) +
                    (Ops::Greater(d2, comp) ? 1 : 0);
          }
#pragma unroll 1
          for (; j < g1; ++j) rank += Ops::Greater(s_sorted[j], comp) ? 1 : 0;
          s_fin[g0 + rank] = comp;
        }
        CTCX_TICK(13)  // PG: rank in group
        __syncthreads();  // table cleared, final order known; s_hist / scalars no longer needed this frame
        CTCX_TICK(14)  // PG: barrier
        for (int i = tid; i < kBinsV2; i += NT) s_hist[i] = 0u;
        if (tid == 0) {
          sci[kV2NCand] = 0;
          sci[kV2NRisk] = 0;
          sci[kV4NChg] = 0;
          sci[kV4MinWiped] = 0x7fffffff;
          sci[kV4MaxParent] = -1;
          if (TIMING) sci[kV4NAtRisk] = 0;
          s_keys[kV4KMin] = Ops::kKeyMax;
          s_keys[kV4KMax] = (Key)0;
          sci[kV2NBnd] = 0;
          s_keys[kV4KMinBase] = Ops::kKeyMax;
          s_keys[kV4KGap] = gap_next;
          sci[kV3Found] = 0;
        }
        if (tid < n) s_wiped[tid] = 0u;
        if (pg_role < PGS && pg_slot < n_new) {
          const int r = pg_slot;
          const Comp comp = s_fin[r];
          const unsigned okey = ~Ops::CompNotOrder(comp);
          const bool fresh = (okey & 0x80000000u) != 0u;
          const int src = fresh ? (int)((okey & 0x7fffffffu) >> 16) : (int)okey;  // parent row / old slot
          const int lbl = fresh ? (int)(okey & 0xffffu) : o_label[src];
          const R s = Ops::UnKey(Ops::CompKey(comp));
          if (pg_role == 0) {  // state arrays + back-pointer record
            unsigned rec;
            if (!fresh) {  // surviving member
              w_total[r] = m_nt[src];
              w_blk[r] = m_nb[src];
              w_lab[r] = m_nl[src];
              w_ab[r] = m_nab[src];
              w_an[r] = m_nan[src];
              rec = m_rec[src];
            } else {  // fresh child (decoder.h:170-187)
              const R pl = Ops::Sub(x[lbl], off);
              R v_an = Ops::Add(o_ab[src], pl);
              unsigned an_kind = kAnParAb;
              if (lbl != o_label[src]) {
                const R c2 = Ops::Add(o_an[src], pl);
                if (c2 > v_an) { v_an = c2; an_kind = kAnParAn; }
              }
              w_total[r] = s;
              w_blk[r] = Ops::NegInf();
              w_lab[r] = s;
              w_ab[r] = Ops::NegInf();
              w_an[r] = v_an;
              rec = PackRec32(0xffu, (unsigned)src, kAbFromAb, an_kind, (unsigned)lbl);
            }
            w_label[r] = lbl;
            p.bp32[((size_t)b * p.Tcap + (t_done + t0 + t)) * W + r] = rec;
          }
          if (PGS == 1 || pg_role == 1) {  // prefix hash, row info of the next frame, parent look-up table
            unsigned long long hsh;
            R nt_, nb_;
            if (!fresh) {
              hsh = o_hash[src];
              w_phash[r] = o_phash[src];
              nt_ = m_nt[src];
              nb_ = m_nb[src];
            } else {
              hsh = HashChild(o_hash[src], lbl);
              w_phash[r] = o_hash[src];
              nt_ = s;
              nb_ = Ops::NegInf();
            }
            w_hash[r] = hsh;
            s_row[r] = Rec::MakeRow(nt_, nb_, lbl);
            unsigned h = (unsigned)hsh & (TS - 1);
            const unsigned entry = ((unsigned)(hsh >> 42) << 10) | (unsigned)r;
            while (atomicCAS(&s_htab[h], 0xffffffffu, entry) != 0xffffffffu) h = (h + 1) & (TS - 1);
          }
        }
        CTCX_TICK(15)  // PG: state write
      }
      __syncthreads();
      CTCX_TICK(6)  // PG
      n = n_new;
      if (__builtin_expect(p.ready != nullptr && sc[kV4Abort] != 0, 0)) {  // the input copy never arrived
        t_end = t + 1;
        break;
      }
    }
    if (TIMING && timing)
      for (int i = 0; i < (TIMING ? kV4DbgSlots : 1); ++i) {
        if (i < p.dbg_slots) atomicAdd(reinterpret_cast<unsigned long long*>(p.dbg_cycles + (size_t)b * p.dbg_slots + i), (unsigned long long)cyc[i]);
        cyc[TIMING ? i : 0] = 0;
      }

    {
      const int cur = t_end & 1;
      const int overflow = (p.seq_len[b] > p.Tcap - t_done) ? 4 : 0;
      const int lost = ((t_end != L) ? 8 : 0) | (carried & 8);  // an input frame never arrived (this slice or before)
      // ---- final beam (decoder.h:229-261): sorted, the first P slots are the top paths ----
      if (last_slice || lost) {
        for (int q = tid; q < p.P; q += NT) {
          if (q < n) {
            p.fin_total[(size_t)b * p.P + q] = s_total[cur * WMAX + q];
            p.fin_kind[(size_t)b * p.P + q] = (s_ab[cur * WMAX + q] > s_an[cur * WMAX + q]) ? 1 : 0;
          } else {
            p.fin_total[(size_t)b * p.P + q] = (R)0;
            p.fin_kind[(size_t)b * p.P + q] = 0;
          }
        }
        if (tid == 0) {
          p.fin_n[b] = n;
          p.flags[b] = (sci[kV2Anomaly] ? 1 : 0) | ((p.P > n) ? 2 : 0) | overflow | lost;
        }
      }
      // ---- carry the beam (and the score-range prediction) to the next slice / the next call ----
      if (p.state != nullptr && (!last_slice || p.t_done != nullptr)) {
        const StreamViewT<R> sv = StreamBlock<R>(p.state, B, W, b);
        for (int i = tid; i < n; i += NT) {
          sv.total[i] = s_total[cur * WMAX + i]; sv.blk[i] = s_blk[cur * WMAX + i];
          sv.lab[i] = s_lab[cur * WMAX + i]; sv.ab[i] = s_ab[cur * WMAX + i];
          sv.an[i] = s_an[cur * WMAX + i]; sv.label[i] = s_label[cur * WMAX + i];
          sv.hash[i] = s_hash[cur * WMAX + i]; sv.phash[i] = s_phash[cur * WMAX + i];
        }
        if (tid == 0) {
          sv.hdr->n = n;
          sv.hdr->gap = s_keys[kV4KGap];
          sv.hdr->flags = (sci[kV2Anomaly] ? 1 : 0) | overflow | lost | (carried & 4);
          if constexpr (kF64) {
            sv.hdr->type = 8;
            StreamMarkF64Step(p.state, W, b);
          }
        }
      }
      if (p.t_done != nullptr && tid == 0) p.t_done[b] = t_done + t_end;
      if (p.n_slices > 1 && !last_slice) {  // release the next slice of this utterance
        __threadfence();
        __syncthreads();
        if (tid == 0) asm volatile("st.release.gpu.global.s32 [%0], %1;\n" ::"l"(p.progress + b), "r"(slice + 1) : "memory");
      }
    }
    __syncthreads();  // the next task re-initialises the shared state
  }
#undef CTCX_TICK
}

}  // namespace ctcx
