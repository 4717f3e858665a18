"""The exact-CTC reference (tests/ctcx_exact.py) against brute force, and the CPU oracle against
exact CTC. CPU only.

With a beam at least as wide as the number of labelings that can have non-zero probability the
decoder prunes nothing, so its results are fixed by the definition of CTC alone: this checks the
oracle's reading of the semantics without the original project's compiled code. With pruning only
the bounds log_probability <= log p(l|x) and alignment score <= log_probability remain.
"""
import itertools

import numpy as np
import pytest

import ctcx_exact as X
import ctcx_testlib as L


def _brute_force(lp, blank):
    """All C^T frame paths grouped by their CTC collapse: labeling -> (log-sum, max)."""
    T, C = lp.shape
    groups = {}
    for path in itertools.product(range(C), repeat=T):
        lab = X.collapse([-1 if c == blank else c for c in path], -1)
        s = float(sum(lp[t, c] for t, c in enumerate(path)))
        if s == -np.inf:
            continue
        v = groups.setdefault(lab, [])
        v.append(s)
    return {k: (float(np.logaddexp.reduce(v)), max(v)) for k, v in groups.items()}


@pytest.mark.parametrize("T,C,blank", [(1, 2, 0), (2, 3, 1), (3, 2, 1), (4, 3, 0), (5, 3, 2), (6, 3, 1),
                                       (4, 4, 3), (5, 4, 0), (6, 2, 0)])
def test_exact_reference_against_brute_force(T, C, blank):
    rng = np.random.default_rng(100 * T + C)
    x = rng.standard_normal((T, C)) * 2.0
    lp = X.log_softmax(x)
    want = _brute_force(lp, blank)
    got = X.enumerate_labelings(lp, blank)
    assert set(got) == set(want)
    assert len(got) == X.labeling_count(T, C - 1)
    for lab, (s, m) in want.items():
        assert abs(got[lab][0] - s) <= 1e-12 * (1 + abs(s)), lab
        assert abs(got[lab][1] - m) <= 1e-12 * (1 + abs(m)), lab
        assert abs(X.ctc_forward(lp, lab, blank) - s) <= 1e-12 * (1 + abs(s)), lab
        assert abs(X.ctc_viterbi(lp, lab, blank) - m) <= 1e-12 * (1 + abs(m)), lab
    # probabilities of all labelings sum to one
    assert abs(np.logaddexp.reduce([v[0] for v in want.values()])) < 1e-12
    # a labeling that cannot fit has probability zero
    assert X.ctc_forward(lp, tuple([c for c in range(C) if c != blank][:1]) * (T + 1), blank) == -np.inf


def test_exact_reference_with_masked_classes():
    """-inf logits: the enumeration skips masked classes and agrees with brute force."""
    rng = np.random.default_rng(7)
    x = rng.standard_normal((5, 4))
    x[rng.random((5, 4)) < 0.4] = -np.inf
    x[:, 2] = rng.standard_normal(5)  # blank stays finite
    lp = X.log_softmax(x)
    want = _brute_force(lp, 2)
    got = X.enumerate_labelings(lp, 2)
    assert set(got) == set(want)
    for lab, (s, m) in want.items():
        assert abs(got[lab][0] - s) <= 1e-12 * (1 + abs(s)) and abs(got[lab][1] - m) <= 1e-12 * (1 + abs(m))


def _dense_paths(res, b, P):
    return [(res.decoded(b, p), res.alignment(b, p), float(res.logp[b, p])) for p in range(P)]


def _check_exact_regime(x, sl, W, P, merge, blank, table=None, exact=True):
    """Oracle decode of x compared utterance by utterance with exact CTC."""
    res = L.oracle_decode(x, sl, W, P, merge, blank, -1, lm=table)
    for b in range(x.shape[1]):
        lp = X.log_softmax(x[:sl[b], b])
        labs = X.enumerate_labelings(lp, blank) if exact else None
        if exact:
            assert len(labs) <= W, "the beam can prune: %d labelings, beam %d" % (len(labs), W)
        bad = X.check_paths(_dense_paths(res, b, P), lp, blank, -1, merge, exact=exact, table=table,
                            logits=x[:sl[b], b], labelings=labs)
        assert not bad, "utterance %d: %s" % (b, bad[:4])
    return res


EXACT_CASES = [
    # T, C, W, P, merge, blank, dtype
    (4, 3, 15, 9, False, 0, np.float32),      # W = the labeling count: the beam just fills
    (6, 3, 41, 8, True, 1, np.float32),
    (7, 3, 67, 5, False, 2, np.float64),
    (3, 5, 57, 4, True, 4, np.float32),
    (4, 5, 189, 10, False, 2, np.float64),
    (2, 29, 785, 6, False, 28, np.float32),
    (2, 29, 813, 3, True, 0, np.float64),
    (9, 2, 10, 5, False, 0, np.float32),      # one label: a long chain of LogSumExps per labeling
    (40, 2, 41, 3, True, 1, np.float32),
]


@pytest.mark.parametrize("case", EXACT_CASES, ids=lambda c: "T%d-C%d-W%d-P%d-%s-blank%d-%s" % (
    c[0], c[1], c[2], c[3], "merge" if c[4] else "nomerge", c[5], np.dtype(c[6]).name))
def test_oracle_in_the_exact_regime(case):
    T, C, W, P, merge, blank, dt = case
    rng = np.random.default_rng(T * 1000 + C)
    x = (rng.standard_normal((T, 3, C)) * 1.5).astype(dt)
    sl = np.array([T, T, max(T - 1, 1)], np.int32)
    _check_exact_regime(x, sl, W, P, merge, blank)


@pytest.mark.parametrize("merge", [False, True])
def test_oracle_scorer_in_the_exact_regime(merge):
    """With a scorer table, log_probability = log p(l|x) + S(l), S(l) = sum_k table[l_{k-1}+1][l_k]."""
    rng = np.random.default_rng(3)
    for T, C, W, blank in ((5, 3, 25, 0), (6, 4, 358, 2), (2, 29, 785, 28)):
        x = rng.standard_normal((T, 3, C)).astype(np.float32)
        table = (-np.abs(rng.standard_normal((C + 1, C))) * 1.5).astype(np.float32)
        _check_exact_regime(x, np.full(3, T, np.int32), W, 4, merge, blank, table=table)


def test_oracle_masked_vocabulary_in_the_exact_regime():
    """-inf masking with a wide vocabulary: 2-3 finite non-blank classes per frame at high label ids."""
    rng = np.random.default_rng(11)
    for T, C, blank in ((4, 300, 0), (3, 4096, 4095), (3, 4096, 7), (3, 65535, 65534)):
        x = X.masked_logits(T, 2, C, blank, rng)
        sl = np.full(2, T, np.int32)
        _check_exact_regime(x, sl, X.max_labelings(x, sl, blank), 5, False, blank)


@pytest.mark.parametrize("kind", ["gauss", "peaky"])
def test_oracle_bounds_with_pruning(kind):
    """cfg2 shape (C=29, beam 100, merge_repeated, blank last), shortened: every returned path obeys
    log_probability <= log p(l|x) and alignment score <= log_probability; on Gaussian logits the beam
    loses many nats, so the first bound is far from tight there."""
    T, B, C, W, P = 300, 3, 29, 100, 4
    x = L.make_logits(kind, T, B, C, 28, seed=5)
    sl = L.ragged_lengths(T, B, 5)
    res = _check_exact_regime(x, sl, W, P, True, 28, exact=False)
    if kind == "gauss":
        lp = X.log_softmax(x[:sl[0], 0])
        lab = X.collapse(res.alignment(0, 0), -1)
        assert res.logp[0, 0] < X.ctc_forward(lp, lab, 28) - 1.0  # pruning lost mass: the check is not vacuous


def test_batched_scores_equal_the_single_recursions():
    """ctc_scores_many (used to bound thousands of returned paths) == ctc_forward / ctc_viterbi."""
    rng = np.random.default_rng(4)
    lps, labs = [], []
    for _ in range(60):
        T = int(rng.integers(0, 40))
        lps.append(X.log_softmax(rng.standard_normal((T, 6)) * 2))
        labs.append(tuple(int(v) for v in rng.integers(1, 6, int(rng.integers(0, T // 2 + 2)))))
    for lp, lab, (f, v) in zip(lps, labs, X.ctc_scores_many(lps, labs, 0)):
        for got, want in ((f, X.ctc_forward(lp, lab, 0)), (v, X.ctc_viterbi(lp, lab, 0))):
            assert got == want or abs(got - want) <= 1e-12 * (1 + abs(want)), (lp.shape, lab)
