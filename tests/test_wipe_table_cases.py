"""The revisit-wipe cases with a scorer table of tests/golden/wipe_table_cases.npz on the CPU
(tests/golden/make_wipe_table_cases.py).

With a table the narrow kernel tests every class of a row for candidates and lists every member whose
parent holds an earlier slot; the cases drive that fixed point at least as deep as the zero-table cases
of tests/golden/wipe_cases.npz, with non-zero and -inf entries in the table. Here:

* every case still reaches what the fixture records for it on the CPU model (with its table), and each
  beam tier reaches its targets;
* the exposing cases decode differently under the mistaken fixed point they name, so a kernel making
  that mistake fails on them;
* the oracle equals the model bit for bit, and every path meets the pruning bounds of exact CTC + S(l).

tests/test_gpu_scorer_table.py compares the kernels with the oracle on the same cases.
"""
import numpy as np
import pytest

import ctcx_exact as X
import ctcx_testlib as L

CASES = L.wipe_table_cases()


def tier(c):
    if c.W > 256:
        return "generic"
    return "narrow%d" % (32 if c.W <= 32 else 128 if c.W <= 128 else 256)


@pytest.mark.parametrize("c", CASES, ids=lambda c: c.name)
def test_case_reaches_its_recorded_statistics(c):
    _, st, iters = L.model_decode_utts(c.x, c.sl, c.W, c.P, c.merge, c.blank, lm=c.lm)
    assert st[0] == c.stats
    np.testing.assert_array_equal(iters[0], c.iters)


# at least the rounds the zero-table fixture reaches per tier (the final, unchanged round included)
TARGETS = {"narrow32": 5, "narrow128": 6, "narrow256": 6, "generic": 7}


@pytest.mark.parametrize("name", sorted(TARGETS))
def test_each_tier_reaches_its_targets(name):
    cs = [c for c in CASES if tier(c) == name]
    assert max(c.stats["fp_iters_max"] for c in cs) >= TARGETS[name]
    for key in ("fp_unwipes", "wiped_parents", "frames_wipe_matters"):
        assert max(c.stats[key] for c in cs) > 0, key
    # the tables are not a no-op: non-zero entries, and -inf constraints somewhere in the tier
    assert all(np.count_nonzero(c.lm) >= c.C for c in cs)
    assert any(np.isneginf(c.lm).any() for c in cs)


def test_deep_frames_at_the_time_slice_boundaries():
    """At T = 128 the time-sliced queue cuts utterances at 32 or 64 frames: deep frames on both sides."""
    for name in ("lm-slices-t32-c5-w16", "lm-slices-t128-c6-w64"):
        c = next(c for c in CASES if c.name == name)
        assert c.T == 128
        for b in (32, 64):
            assert min(c.iters[b - 1], c.iters[b]) >= 2 and max(c.iters[b - 1], c.iters[b]) >= 3, (c.name, b)


def test_every_kernel_has_cases_that_expose_the_mistakes():
    got = {(tier(c), c.exposes) for c in CASES if c.exposes}
    want = {(t, "count_wiped_rows") for t in TARGETS} | {("narrow128", "four_rounds"), ("narrow256", "four_rounds")}
    assert got >= want


@pytest.mark.parametrize("c", [c for c in CASES if c.exposes], ids=lambda c: c.name)
def test_case_decodes_differently_under_the_mistake_it_exposes(c):
    exact = L.model_decode_utts(c.x, c.sl, c.W, c.P, c.merge, c.blank, lm=c.lm)[0]
    assert L.same_result(exact, L.model_decode_utts(c.x, c.sl, c.W, c.P, c.merge, c.blank, variant=c.exposes,
                                                    lm=c.lm)[0])


@pytest.mark.parametrize("c", CASES, ids=lambda c: c.name)
def test_oracle_equals_the_model_and_meets_the_bounds(c):
    res = L.oracle_decode(c.x, c.sl, c.W, c.P, c.merge, c.blank, -1, lm=c.lm)
    model = L.model_decode_utts(c.x, c.sl, c.W, c.P, c.merge, c.blank, lm=c.lm)[0]
    assert L.same_result(model, res) == []
    lp = X.log_softmax(c.x[:, 0].astype(np.float64))
    paths = [(res.decoded(0, p), res.alignment(0, p), float(res.logp[0, p])) for p in range(c.P)]
    assert not X.check_paths(paths, lp, c.blank, -1, c.merge, table=c.lm, logits=c.x[:, 0])
