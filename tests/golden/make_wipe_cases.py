"""Generator of tests/golden/wipe_cases.npz: single utterances that drive the revisit-wipe fixed point
(DESIGN.md section 3, item 3) far deeper than random inputs do, found by a seeded search on the CPU
model (tests/model/ctcx_model.cc) alone.

    python tests/golden/make_wipe_cases.py [out.npz]

Random inputs reach at most 4 rounds of the fixed point (the round that changes nothing included). A
hill-climb over the logits, keeping every change that does not lower its objective, reaches 5 to 7
in every beam tier. Every logit is k/16 for an integer k in [-128, 128] (stored as int16 k; -32768
stands for -inf), so float32, float16 and bfloat16 hold the same values exactly and one case serves
all three input types.

Per case the fixture stores the logits (`<name>/k`, [T, C]), the decode attributes (`<name>/attrs`:
beam width, blank index, merge_repeated, top paths, and the mistaken fixed point the case exposes: a
ctcx_testlib.MODEL_VARIANTS value, 0 for none), the model's statistics of the utterance (`<name>/stats`,
the 16 slots of ctcx_testlib.MODEL_STATS) and the fixed-point rounds of every frame (`<name>/iters`).
The tests check that each case still reaches the statistics recorded here.

The search is deterministic: every case has its own seed and a fixed number of steps, so the
fixture regenerates bit for bit (on the same glibc, whose expf/logf/log1pf the model calls).
"""
import os
import sys
from multiprocessing import Pool

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, os.path.dirname(HERE))
import ctcx_testlib as L  # noqa: E402

NEG_INF_K = -32768  # int16 code of -inf
KMAX = 128          # logits are k/16 with |k| <= 128

# name, T, C, W, blank, merge, seed, steps, objective (see _objective)
SEARCHED = [
    ("t32-c3-w16", 40, 3, 16, 2, False, 22, 30000, "depth"),
    ("t32-c5-w32", 40, 5, 32, 2, True, 12, 30000, "depth"),
    ("t32-c4-w8", 40, 4, 8, 0, False, 27, 30000, "depth"),
    ("t128-c8-w64", 60, 8, 64, 7, False, 14, 12000, "depth"),
    ("t128-c8-w100", 60, 8, 100, 3, True, 15, 8000, "depth"),
    ("t256-c6-w160", 50, 6, 160, 0, False, 16, 3000, "depth"),
    ("t256-c4-w256", 50, 4, 256, 3, True, 17, 2000, "depth"),
    ("generic-c4-w300", 50, 4, 300, 0, True, 18, 1500, "depth"),
    ("generic-c3-w512", 40, 3, 512, 1, False, 19, 800, "depth"),
    # deep frames on both sides of the narrow kernel's time-slice boundaries at T = 128 (slices of
    # ceil(128 / n) frames: 32 with 4 slices, 64 with 2) -- the search only sees the first 66 frames
    ("slices-t32-c5-w16", 128, 5, 16, 4, False, 20, 12000, "slices"),
    ("slices-t128-c6-w64", 128, 6, 64, 0, True, 21, 5000, "slices"),
]
SLICE_FRAMES = (31, 32, 63, 64)


def decode(k, W, blank, T=None):
    """Model statistics and per-frame rounds of one utterance (optionally of its first T frames)."""
    x = np.where(k == NEG_INF_K, -np.inf, k.astype(np.float32) / 16).astype(np.float32)[:, None, :]
    sl = np.array([x.shape[0] if T is None else T], np.int32)
    _, st, it = L.model_decode_utts(x, sl, W, 1, False, blank)
    return st[0], it[0]


def _objective(kind, it):
    if kind == "depth":  # the deepest frame first, then how many frames go past 2 rounds, and how far
        return (int(it.max()), int(np.sum(np.maximum(it - 2, 0) ** 2)))
    v = it[list(SLICE_FRAMES)]
    return (int(v.min()), int(v.sum()), int(it.max()))


def search(spec):
    name, T, C, W, blank, merge, seed, steps, kind = spec
    rng = np.random.default_rng(seed)
    k = np.clip(np.round(rng.standard_normal((T, C)) * 24), -KMAX, KMAX).astype(np.int16)
    horizon = None if kind == "depth" else max(SLICE_FRAMES) + 2
    lo = 0 if kind == "depth" else min(SLICE_FRAMES) - 16
    best = _objective(kind, decode(k, W, blank, horizon)[1])
    for _ in range(steps):
        k2 = k.copy()
        for _ in range(int(rng.integers(1, 4))):
            t, c = int(rng.integers(lo, horizon or T)), int(rng.integers(0, C))
            k2[t, c] = np.clip(int(k2[t, c]) + int(rng.integers(-32, 33)), -KMAX, KMAX)
        o = _objective(kind, decode(k2, W, blank, horizon)[1])
        if o >= best:
            k, best = k2, o
    return name, k, W, blank, merge


def early_case():
    """At-risk members while the beam is not yet full: fewer labelings than beam slots in every frame."""
    rng = np.random.default_rng(31)
    T, C, W, blank = 4, 4, 128, 1
    for _ in range(1000):
        k = np.clip(np.round(rng.standard_normal((T, C)) * 24), -KMAX, KMAX).astype(np.int16)
        st, _ = decode(k, W, blank)
        if st["frames_at_risk"] == T - 1 and st["wiped"] == 0:
            return "early-c4-w128", k, W, blank, True
    raise RuntimeError("no early case")


def anomaly_case():
    """A wiped member whose parent's re-score beats its own total (the kernels report it as the
    rounding anomaly, DESIGN.md section 8): label-symmetric frames (every label shares one logit)
    tie label-permuted prefixes exactly. Random search, first hit."""
    rng = np.random.default_rng(41)
    for _ in range(2000000):
        T, C, W = int(rng.integers(10, 40)), int(rng.integers(3, 8)), int(rng.integers(2, 12))
        blank = int(rng.integers(0, C))
        a, b = rng.integers(-KMAX, KMAX + 1, (T, 1)), rng.integers(-KMAX, KMAX + 1, (T, 1))
        k = np.repeat(b, C, axis=1)
        k[:, blank] = a[:, 0]
        if rng.random() < 0.5:
            k = k + rng.integers(-1, 2, k.shape) * rng.integers(0, 2, (T, 1))
        k = np.clip(k, -KMAX, KMAX).astype(np.int16)
        st, _ = decode(k, W, blank)
        if st["anomalies"] > 0:
            return "anomaly-c%d-w%d" % (C, W), k, W, blank, False
    raise RuntimeError("no anomaly case")


def tied_wide_case():
    """Few-level wide vocabulary: 48 labels tie at the top level of a frame, more than the wide kernel's
    sorted prefix holds at W = 16 (2W + 2 = 34 classes), so capped rows meet at-risk members."""
    rng = np.random.default_rng(51)
    T, C, W, blank = 30, 1024, 16, 0
    k = np.full((T, C), -KMAX, np.int16)
    for t in range(T):
        top = rng.choice(np.arange(1, C), 48, replace=False)
        mid = rng.choice(np.arange(1, C), 200, replace=False)
        k[t, mid] = int(rng.integers(-64, 0))
        k[t, top] = int(rng.integers(-16, 48))
        k[t, blank] = int(rng.integers(-16, 64))
    return "tied-c1024-w16", k, W, blank, False


# wide vocabularies: a searched case padded with classes after its own, at -inf (the model's result
# does not change) or at the lowest logit of the grid (it does: new candidates, re-verified)
PADDED = [
    # base, C, pad
    ("t32-c3-w16", 33, "inf"),
    ("t32-c3-w16", 64, "low"),
    ("t32-c3-w16", 65, "inf"),
    ("t32-c3-w16", 1024, "inf"),
    ("t32-c3-w16", 1024, "low"),
    ("t32-c5-w32", 33, "inf"),
    ("t32-c5-w32", 65, "low"),
    ("t128-c8-w64", 65, "inf"),
    ("t128-c8-w64", 1024, "inf"),
    ("t128-c8-w64", 1024, "low"),
    ("t256-c6-w160", 65, "low"),
]


# cases that a kernel with a mistaken fixed point decodes differently (the variants of the CPU model):
# a searched case cut right after the first frame at which the variant's beam differs, every path of
# that beam returned. Counting the candidates of wiped rows (a verdict that ignores s_wiped) never
# changes the top few paths of the searched cases; stopping after 4 rounds needs a frame with 6 (the
# generic range's deep cases have such frames, but the cap changes none of their beams).
EXPOSING = [
    # base, variant, pad to C (0: none)
    ("t32-c5-w32", "count_wiped_rows", 0),
    ("t32-c5-w32", "count_wiped_rows", 33),
    ("t128-c8-w64", "count_wiped_rows", 0),
    ("t128-c8-w64", "count_wiped_rows", 65),
    ("t128-c8-w64", "four_rounds", 0),
    ("t128-c8-w100", "four_rounds", 0),
    ("t256-c6-w160", "count_wiped_rows", 0),
    ("t256-c4-w256", "four_rounds", 0),
    ("generic-c4-w300", "count_wiped_rows", 0),
]


def differs(k, W, blank, merge, variant):
    """Top paths (the whole final beam) that differ between the model and its mistaken variant, and
    that number of paths; (0, 0) if the beam holds fewer than W hypotheses."""
    x = np.where(k == NEG_INF_K, -np.inf, k.astype(np.float32) / 16).astype(np.float32)[:, None, :]
    sl = np.array([k.shape[0]], np.int32)
    try:
        exact = L.model_decode_utts(x, sl, W, W, merge, blank)[0]
    except L.OracleError:
        return 0, 0
    other = L.model_decode_utts(x, sl, W, W, merge, blank, variant=variant)[0]
    return len(L.same_result(exact, other)), W


def exposing(base, variant):
    name, k, W, blank, merge = base
    for T in range(2, k.shape[0] + 1):
        if differs(k[:T], W, blank, merge, variant)[0]:
            return "%s-%s-t%d" % (name, variant.replace("_", "-"), T), k[:T].copy(), W, blank, merge
    raise RuntimeError("%s does not expose %s" % (name, variant))


def pad(k, C, how):
    out = np.full((k.shape[0], C), NEG_INF_K if how == "inf" else -KMAX, np.int16)
    out[:, :k.shape[1]] = k
    return out


def build(out_path):
    with Pool(min(len(SEARCHED), os.cpu_count() or 1)) as p:
        cases = p.map(search, SEARCHED)
    cases += [early_case(), anomaly_case(), tied_wide_case()]
    base = {c[0]: c for c in cases}
    for name, C, how in PADDED:
        _, k, W, blank, merge = base[name]
        cases.append(("%s-pad%s-c%d" % (name, how, C), pad(k, C, how), W, blank, merge))
    paths, exposes = {}, {}
    for name, variant, C in EXPOSING:
        c = exposing(base[name], variant)
        if C:
            c = ("%s-padinf-c%d" % (c[0], C), pad(c[1], C, "inf")) + c[2:]
        cases.append(c)
        paths[c[0]] = c[2]
        exposes[c[0]] = L.MODEL_VARIANTS[variant]
    arrays = {"names": np.array([c[0] for c in cases])}
    for name, k, W, blank, merge in cases:
        st, it = decode(k, W, blank)
        arrays[name + "/k"] = k
        arrays[name + "/attrs"] = np.array([W, blank, int(merge), paths.get(name, min(4, W)),
                                            exposes.get(name, 0)], np.int32)
        arrays[name + "/stats"] = np.array([st[s] for s in L.MODEL_STATS], np.int64)
        arrays[name + "/iters"] = it.astype(np.int8)
        print("%-34s T=%3d C=%4d W=%3d  fp_iters_max %d  fp_unwipes %3d  wiped_parents %3d  frames_at_risk %3d  "
              "wipe_matters %3d  anomalies %d" % (name, k.shape[0], k.shape[1], W, st["fp_iters_max"], st["fp_unwipes"],
                                                  st["wiped_parents"], st["frames_at_risk"],
                                                  st["frames_wipe_matters"], st["anomalies"]))
    np.savez_compressed(out_path, **arrays)


if __name__ == "__main__":
    L.build_model()
    build(sys.argv[1] if len(sys.argv) > 1 else os.path.join(HERE, "wipe_cases.npz"))
