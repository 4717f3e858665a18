"""Generator of tests/golden/wipe_table_cases.npz: revisit-wipe cases with a scorer table, found by a seeded
hill-climb on the CPU model (tests/model/ctcx_model.cc) over the logits AND the table entries.

    python tests/golden/make_wipe_table_cases.py [out.npz]

With a table the candidate scores are no longer monotone in a frame's log-probabilities, so the beam
kernels test every class of a row and list every member whose parent holds an earlier slot; the zero-table
cases of tests/golden/wipe_cases.npz never reach those paths with a non-zero entry. Each search starts
from one of that fixture's searched cases with an all-zero table (so from its depth) and keeps every
change of a few logits or table entries that lowers neither the deepest frame's rounds, nor how many
frames go past 2 rounds and how far, nor the number of non-zero table entries. Table entries are on the
same k/16 grid as the logits, in [-8, 0], and a change may also turn an entry to -inf (a forbidden
extension); both are stored as int16 k with -32768 for -inf.

Per case the fixture stores what wipe_cases.npz stores (`<name>/k`, `/attrs`, `/stats`, `/iters`) plus
the table (`<name>/lm`, [C + 1, C] int16 k). Exposing cases are cut, as there, right after the first
frame at which the model with a mistaken fixed point (the candidates of wiped rows still counted, or the
search stopped after 4 rounds) leaves another beam, and return every path of that beam.

The search is deterministic (own seed, fixed steps per case): the fixture regenerates bit for bit on the
same glibc.
"""
import os
import sys
from multiprocessing import Pool

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, os.path.dirname(HERE))
import ctcx_testlib as L  # noqa: E402

NEG_INF_K = -32768
KMAX = 128

# name, zero-table case it starts from, seed, steps, objective ("depth", or "slices": deep frames on both
# sides of the narrow kernel's time-slice boundaries at T = 128, as in make_wipe_cases.py)
SEARCHED = [
    ("lm-t32-c3-w16", "t32-c3-w16", 61, 12000, "depth"),
    ("lm-t32-c5-w32", "t32-c5-w32", 62, 12000, "depth"),
    ("lm-t128-c8-w64", "t128-c8-w64", 63, 5000, "depth"),
    ("lm-t128-c8-w100", "t128-c8-w100", 64, 4000, "depth"),
    ("lm-t256-c6-w160", "t256-c6-w160", 65, 1500, "depth"),
    ("lm-t256-c4-w256", "t256-c4-w256", 66, 1200, "depth"),
    ("lm-generic-c4-w300", "generic-c4-w300", 67, 900, "depth"),
    ("lm-generic-c3-w512", "generic-c3-w512", 68, 500, "depth"),
    ("lm-slices-t32-c5-w16", "slices-t32-c5-w16", 69, 4000, "slices"),
    ("lm-slices-t128-c6-w64", "slices-t128-c6-w64", 70, 2000, "slices"),
]
SLICE_FRAMES = (31, 32, 63, 64)

# searched case, the mistaken fixed point it must expose
EXPOSING = [
    ("lm-t32-c5-w32", "count_wiped_rows"),
    ("lm-t128-c8-w64", "count_wiped_rows"),
    ("lm-t128-c8-w100", "count_wiped_rows"),
    ("lm-t128-c8-w64", "four_rounds"),
    ("lm-t128-c8-w100", "four_rounds"),
    ("lm-t256-c6-w160", "count_wiped_rows"),
    ("lm-t256-c4-w256", "count_wiped_rows"),
    ("lm-t256-c4-w256", "four_rounds"),
    ("lm-generic-c4-w300", "count_wiped_rows"),
]


def values(k):
    return np.where(k == NEG_INF_K, -np.inf, k.astype(np.float32) / 16).astype(np.float32)


def decode(k, lm, W, blank):
    """Model statistics and per-frame rounds of one utterance with its table."""
    x = values(k)[:, None, :]
    _, st, it = L.model_decode_utts(x, np.array([k.shape[0]], np.int32), W, 1, False, blank, lm=values(lm))
    return st[0], it[0]


def _objective(kind, it, lm):
    if kind == "depth":
        return (int(it.max()), int(np.sum(np.maximum(it - 2, 0) ** 2)), int(np.count_nonzero(lm)))
    v = it[list(SLICE_FRAMES)]
    return (int(v.min()), int(v.sum()), int(np.count_nonzero(lm)), int(it.max()))


def search(spec):
    name, base, seed, steps, kind = spec
    c = {c.name: c for c in L.wipe_cases()}[base]
    k = np.where(np.isneginf(c.x[:, 0]), NEG_INF_K, np.round(c.x[:, 0] * 16)).astype(np.int16)
    T, C = k.shape
    lm = np.zeros((C + 1, C), np.int16)
    rng = np.random.default_rng(seed)
    best = _objective(kind, decode(k, lm, c.W, c.blank)[1], lm)
    for _ in range(steps):
        k2, lm2 = k.copy(), lm.copy()
        for _ in range(int(rng.integers(1, 4))):
            if rng.random() < 0.5:
                t, j = int(rng.integers(0, T)), int(rng.integers(0, C))
                if k2[t, j] != NEG_INF_K:
                    k2[t, j] = np.clip(int(k2[t, j]) + int(rng.integers(-32, 33)), -KMAX, KMAX)
            else:
                r, j = int(rng.integers(0, C + 1)), int(rng.integers(0, C))
                if rng.random() < 0.1:
                    lm2[r, j] = NEG_INF_K
                else:
                    v = 0 if lm2[r, j] == NEG_INF_K else int(lm2[r, j])
                    lm2[r, j] = np.clip(v + int(rng.integers(-32, 17)), -KMAX, 0)
        o = _objective(kind, decode(k2, lm2, c.W, c.blank)[1], lm2)
        if o >= best:
            k, lm, best = k2, lm2, o
    return name, k, lm, c.W, c.blank, c.merge


def differs(k, lm, W, blank, merge, variant):
    """Paths of the whole final beam that differ between the model and its mistaken variant."""
    x = values(k)[:, None, :]
    sl = np.array([k.shape[0]], np.int32)
    try:
        exact = L.model_decode_utts(x, sl, W, W, merge, blank, lm=values(lm))[0]
    except L.OracleError:  # fewer than W hypotheses
        return 0
    other = L.model_decode_utts(x, sl, W, W, merge, blank, variant=variant, lm=values(lm))[0]
    return len(L.same_result(exact, other))


def exposing(base, variant):
    name, k, lm, W, blank, merge = base
    for T in range(2, k.shape[0] + 1):
        if differs(k[:T], lm, W, blank, merge, variant):
            return "%s-%s-t%d" % (name, variant.replace("_", "-"), T), k[:T].copy(), lm, W, blank, merge
    raise RuntimeError("%s does not expose %s" % (name, variant))


def build(out_path):
    with Pool(min(len(SEARCHED), os.cpu_count() or 1)) as p:
        cases = p.map(search, SEARCHED)
    base = {c[0]: c for c in cases}
    paths, exposes = {}, {}
    for name, variant in EXPOSING:
        c = exposing(base[name], variant)
        cases.append(c)
        paths[c[0]] = c[3]
        exposes[c[0]] = L.MODEL_VARIANTS[variant]
    arrays = {"names": np.array([c[0] for c in cases])}
    for name, k, lm, W, blank, merge in cases:
        st, it = decode(k, lm, W, blank)
        arrays[name + "/k"] = k
        arrays[name + "/lm"] = lm
        arrays[name + "/attrs"] = np.array([W, blank, int(merge), paths.get(name, min(4, W)),
                                            exposes.get(name, 0)], np.int32)
        arrays[name + "/stats"] = np.array([st[s] for s in L.MODEL_STATS], np.int64)
        arrays[name + "/iters"] = it.astype(np.int8)
        print("%-42s T=%3d C=%d W=%3d  fp_iters_max %d  fp_unwipes %3d  wiped_parents %3d  table: %d non-zero, "
              "%d -inf" % (name, k.shape[0], k.shape[1], W, st["fp_iters_max"], st["fp_unwipes"],
                           st["wiped_parents"], np.count_nonzero(lm), np.count_nonzero(lm == NEG_INF_K)))
    np.savez_compressed(out_path, **arrays)


if __name__ == "__main__":
    L.build_model()
    build(sys.argv[1] if len(sys.argv) > 1 else os.path.join(HERE, "wipe_table_cases.npz"))
