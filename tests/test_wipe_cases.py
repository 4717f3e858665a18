"""The revisit-wipe cases of tests/golden/wipe_cases.npz on the CPU (tests/golden/make_wipe_cases.py).

A member evicted during the grow phase and revisited by its parent is reset and loses its turn
(DESIGN.md section 2). The kernels decide these wipes as a count-based fixed point; random inputs
settle it in at most 4 rounds. The fixture's cases go deeper, with verdicts that flip back in later
rounds, wiped parents, wipes that remove candidates, at-risk members in a beam that is not full, the
rounding anomaly and deep frames at time-slice boundaries. Here:

* every case still reaches what the fixture records for it on the CPU model, and the fixture as a
  whole reaches the targets below per beam tier: a fixture that loses its depth fails here;
* some cases decode differently under a fixed point that makes a known mistake (the candidates of
  wiped rows still count, or the search stops after 4 rounds), so a kernel making it fails on them;
* the oracle equals the model bit for bit on every case, and its own counts agree that wipes happen;
* every path the oracle returns meets the pruning bounds of exact CTC (tests/ctcx_exact.py).

tests/test_gpu_wipe_fixed_point.py compares every kernel with the oracle on the same cases.
"""
import numpy as np
import pytest

import ctcx_exact as X
import ctcx_testlib as L

CASES = L.wipe_cases()
BY_NAME = {c.name: c for c in CASES}


def tier(c):
    """Which beam kernel a case is written for: the narrow tiers (C <= 32), the wide vocabularies, or
    the generic range (W > 256)."""
    if c.W > 256:
        return "generic"
    if c.C > 32:
        return "wide"
    return "narrow%d" % (32 if c.W <= 32 else 128 if c.W <= 128 else 256)


@pytest.mark.parametrize("c", CASES, ids=lambda c: c.name)
def test_case_reaches_its_recorded_statistics(c):
    res, st, iters = L.model_decode_utts(c.x, c.sl, c.W, c.P, c.merge, c.blank)
    assert st[0] == c.stats
    np.testing.assert_array_equal(iters[0], c.iters)
    assert c.stats["fp_iters_max"] == c.iters.max() and c.stats["frames_at_risk"] == np.count_nonzero(c.iters)


# the least each tier's cases reach together: fixed-point rounds (the final, unchanged one included),
# verdicts flipped back, wiped parents, frames where a wipe removes candidates
TARGETS = {"narrow32": 5, "narrow128": 6, "narrow256": 5, "generic": 6, "wide": 5}


@pytest.mark.parametrize("name", sorted(TARGETS))
def test_each_tier_reaches_its_targets(name):
    cs = [c for c in CASES if tier(c) == name]
    assert max(c.stats["fp_iters_max"] for c in cs) >= TARGETS[name]
    for key in ("fp_unwipes", "wiped_parents", "frames_wipe_matters"):
        assert max(c.stats[key] for c in cs) > 0, key
    assert {c.merge for c in cs} == {False, True} or name == "wide"


def test_the_fixture_covers_blank_positions_and_special_cases():
    blanks = {("first" if c.blank == 0 else "last" if c.blank == c.C - 1 else "middle") for c in CASES}
    assert blanks == {"first", "middle", "last"}
    assert {c.merge for c in CASES} == {False, True}
    # at-risk members while the beam is not full: nothing can be pruned, every frame has n < W
    e = BY_NAME["early-c4-w128"]
    assert e.stats["frames_at_risk"] > 0 and X.max_labelings(e.x, e.sl, e.blank) < e.W
    # a wiped member whose parent's re-score beats its own total: the kernels must raise the flag
    assert sum(c.stats["anomalies"] > 0 for c in CASES) >= 1
    # deep frames on both sides of the time-slice boundaries at 32 and 64 frames (T = 128)
    for c in (BY_NAME["slices-t32-c5-w16"], BY_NAME["slices-t128-c6-w64"]):
        assert c.T == 128
        for b in (32, 64):
            assert min(c.iters[b - 1], c.iters[b]) >= 2 and max(c.iters[b - 1], c.iters[b]) >= 4, (c.name, b)
    # wide vocabularies: the ballot branch (sorted prefix <= 64 classes) and the per-row count, with
    # the prefix capped (C - 1 > 2W + 2) and not
    wide = [c for c in CASES if tier(c) == "wide"]
    cv = [min(c.C - 1, 2 * c.W + 2) for c in wide]
    assert min(cv) <= 64 < max(cv)
    assert {c.C - 1 > 2 * c.W + 2 for c in wide} == {False, True}
    assert {c.C for c in wide} >= {33, 64, 65, 1024}


EXPOSING = [c for c in CASES if c.exposes]


@pytest.mark.parametrize("c", EXPOSING, ids=lambda c: c.name)
def test_case_decodes_differently_under_the_mistake_it_exposes(c):
    """A kernel whose fixed point makes this mistake returns other paths than the oracle on this case."""
    exact = L.model_decode(c.x, c.sl, c.W, c.P, c.merge, c.blank)
    assert L.same_result(exact, L.model_decode_utts(c.x, c.sl, c.W, c.P, c.merge, c.blank, variant=c.exposes)[0])


def test_every_kernel_has_cases_that_expose_the_mistakes():
    """Counting the candidates of wiped rows: every narrow tier, the wide kernel's ballot count (sorted
    prefix <= 64 classes) and the generic kernel. Stopping after 4 rounds: the 128- and 256-slot tiers
    (a cap can only matter where a frame takes 6 rounds)."""
    got = {(tier(c), c.exposes) for c in EXPOSING}
    want = {(t, "count_wiped_rows") for t in ("narrow32", "narrow128", "narrow256", "wide", "generic")}
    want |= {("narrow128", "four_rounds"), ("narrow256", "four_rounds")}
    assert got >= want
    assert all(min(c.C - 1, 2 * c.W + 2) <= 64 for c in EXPOSING if tier(c) == "wide")


@pytest.mark.parametrize("c", CASES, ids=lambda c: c.name)
def test_oracle_equals_the_model_and_meets_the_bounds(c):
    res, st = L.oracle_decode(c.x, c.sl, c.W, c.P, c.merge, c.blank, -1, want_stats=True)
    model = L.model_decode(c.x, c.sl, c.W, c.P, c.merge, c.blank)
    assert L.same_result(model, res) == []
    # the oracle's own counts (oracle/ctcx_oracle.c): members re-scored and reset before their turn, and
    # resets that cost the beam a child it would have accepted
    assert (st.wipes_before_turn > 0) == (c.stats["wiped"] > 0)
    if c.stats["fp_iters_max"] >= 5:
        assert st.effective_wipes > 0 and st.frames_with_effective_wipe > 0
    lp = X.log_softmax(c.x[:, 0].astype(np.float64))
    paths = [(res.decoded(0, p), res.alignment(0, p), float(res.logp[0, p])) for p in range(c.P)]
    assert not X.check_paths(paths, lp, c.blank, -1, c.merge, logits=c.x[:, 0])
