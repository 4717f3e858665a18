"""Every beam kernel's revisit-wipe fixed point on the cases of tests/golden/wipe_cases.npz, which take
it to 5-7 rounds, flip verdicts back in later rounds and wipe parents (tests/test_wipe_cases.py checks
the cases themselves on the CPU). Each decode is compared with the oracle bit for bit:

* narrow kernel, 32/128/256-slot tiers: two CTAs per SM (one utterance), four (the case replicated
  past 2 x SMs) and the time-sliced queue (replicated past the resident CTAs, deep frames at the slice
  boundaries); float32, float16 and bfloat16 on the same values, float64 too; the scorer-table
  variant with an all-zero table (an exact no-op on the scores);
* wide kernel on the cases padded to C = 33 ... 1024 (the ballot count of short sorted prefixes, the
  per-row count, capped prefixes);
* generic kernel, forced, in its candidate-list and full-sweep forms;
* streaming with chunk boundaries at the deepest frames, and page-locked host logits.

Some cases return every path of a beam that a fixed point with a known mistake (the candidates of
wiped rows still counted, or the search stopped after 4 rounds) leaves different; the CPU tests show
that the mistaken model decodes them differently, so a kernel with the mistake fails here.

The rounding-anomaly flag is checked against the CPU model. The timing build of the narrow kernel
(a separate instantiation of the same fixed-point code) counts at-risk members, wiped members and
frames with at-risk members; these must equal the model's counts exactly.
"""
import numpy as np
import pytest

import ctcx_testlib as L

pytestmark = pytest.mark.gpu

CASES = L.wipe_cases()
NARROW = [c for c in CASES if c.C <= 32 and c.W <= 256]
WIDE = [c for c in CASES if c.C > 32 and c.W <= 256]
_want = {}


@pytest.fixture(scope="module")
def op():
    import torch
    if not torch.cuda.is_available():
        pytest.skip("no CUDA device")
    import ctc_beam_search_op_b200 as m
    m.set_beam_impl(None)
    yield m
    m.set_beam_impl(None)


@pytest.fixture(scope="module")
def dev():
    """SM count and the most 256-thread CTAs an SM can hold: what the dispatch thresholds depend on."""
    import torch
    p = torch.cuda.get_device_properties(torch.cuda.current_device())
    sms = int(p.multi_processor_count)
    return {"sms": sms, "minb4": 2 * sms + 1, "sliced": sms * (int(p.max_threads_per_multi_processor) // 256) + 1}


def _ids(cs):
    return [c.name for c in cs]


def want(c, f64=False, B=1):
    """The oracle's result for case c, as a batch of B copies."""
    key = (c.name, f64)
    if key not in _want:
        _want[key] = L.oracle_decode(c.x.astype(np.float64) if f64 else c.x, c.sl, c.W, c.P, c.merge, c.blank, -1)
    r = _want[key]
    if B == 1:
        return r
    src = np.zeros(B, np.int64)
    t = L.DenseResult.__new__(L.DenseResult)
    t.B, t.P, t.T = B, r.P, r.T
    t.dec_len, t.ali_len, t.dec, t.ali, t.logp = r.dec_len[src], r.ali_len[src], r.dec[src], r.ali[src], r.logp[src]
    return t


def inputs(c, dt, B=1, device="cuda"):
    import torch
    x = torch.from_numpy(np.ascontiguousarray(np.repeat(c.x, B, axis=1))).to(getattr(torch, dt))
    return (x.cuda() if device == "cuda" else x.pin_memory()), torch.full((B,), c.T, dtype=torch.int32)


def decode(op, c, x, sl, **kw):
    return op.ctc_ext_beam_search_decoder_raw(x, sl, beam_width=c.W, top_paths=c.P, merge_repeated=c.merge,
                                              blank_index=c.blank, blank_label=-1, **kw)


def check(raw, c, what, f64=False, B=1, exact_flag=False):
    bad = L.raw_mismatches(raw, want(c, f64, B))
    assert not bad, "%s %s: %d of %d utterances differ from the oracle, first %s" % (c.name, what, len(bad), B, bad[:8])
    # the rounding anomaly (DESIGN.md section 8): a member whose parent's re-score beats its own total
    # leaves the beam. The generic kernel reports exactly that; the fast kernels report every such member
    # that is not certain to stay (a superset). The model rounds in float32: float64 decodes round
    # differently and are not held to its count.
    flagged = bool(int(raw.flags) & 1)
    if f64:
        return
    if exact_flag:
        assert flagged == (c.stats["suspects_dropped"] > 0), (c.name, what, raw.flags, c.stats)
    elif c.stats["suspects_dropped"] > 0:
        assert flagged, (c.name, what, c.stats)


# ------------------------------------------------------------------------------------------------
# narrow kernel
@pytest.mark.parametrize("dt", ["float32", "float16", "bfloat16", "float64"])
@pytest.mark.parametrize("c", NARROW, ids=_ids(NARROW))
def test_narrow_two_ctas_per_sm(op, c, dt):
    x, sl = inputs(c, dt)
    check(decode(op, c, x, sl.cuda()), c, dt, f64=dt == "float64")


@pytest.mark.parametrize("dt", ["float32", "bfloat16"])
@pytest.mark.parametrize("c", NARROW, ids=_ids(NARROW))
def test_narrow_four_ctas_per_sm(op, dev, c, dt):
    B = dev["minb4"]
    assert B > 2 * dev["sms"]
    x, sl = inputs(c, dt, B)
    check(decode(op, c, x, sl.cuda()), c, dt, B=B)


SLICED = [c for c in NARROW if c.T >= 64]


@pytest.mark.parametrize("dt", ["float32", "float16"])
@pytest.mark.parametrize("c", SLICED, ids=_ids(SLICED))
def test_narrow_time_sliced_queue(op, dev, c, dt):
    """More utterances than resident CTAs: every utterance is cut into ceil(T / n) frame slices, n =
    min(16, T // 32, ~12 x resident / B); at T = 128 with at least 4 CTAs per SM that is 4 slices of 32
    frames, and the cases have deep frames on both sides of 32 and 64."""
    B = dev["sliced"]
    assert B > 2 * dev["sms"] and c.T == 128
    x, sl = inputs(c, dt, B)
    check(decode(op, c, x, sl.cuda()), c, dt, B=B)


SCORER = [c for c in NARROW if c.C <= 32]


@pytest.mark.parametrize("c", SCORER, ids=_ids(SCORER))
def test_scorer_variant_with_an_all_zero_table(op, dev, c):
    """Adding +0 to every expansion leaves every score as it was, but runs the scorer variants' own
    candidate test (narrow `LM` and generic); both CTA regimes."""
    import torch
    table = torch.zeros((c.C + 1, c.C), dtype=torch.float32).cuda()
    for B in (1, dev["minb4"]):
        x, sl = inputs(c, "float32", B)
        check(decode(op, c, x, sl.cuda(), expansion_scores=table), c, "scorer B=%d" % B, B=B)


# ------------------------------------------------------------------------------------------------
# wide kernel, generic kernel
@pytest.mark.parametrize("dt", ["float32", "float16", "bfloat16"])
@pytest.mark.parametrize("c", WIDE, ids=_ids(WIDE))
def test_wide_vocabularies(op, c, dt):
    x, sl = inputs(c, dt)
    check(decode(op, c, x, sl.cuda()), c, dt)


@pytest.mark.parametrize("dt", ["float32", "bfloat16", "float64"])
def test_generic_kernel_list_and_sweep(op, dt):
    """Every case on the generic kernel: its candidate list holds W x C entries up to 4608, beyond that
    it sweeps every (row, class) pair again in each query."""
    import torch
    modes = set()
    op.set_beam_impl("generic")
    try:
        for c in CASES:
            if dt == "float64" and (c.W > 512 or c.C > 65):
                continue
            modes.add(c.W * c.C <= 4608)
            x, sl = inputs(c, dt)
            check(decode(op, c, x, sl.cuda()), c, "generic " + dt, f64=dt == "float64", exact_flag=True)
            if dt == "float32" and c.C <= 32:
                table = torch.zeros((c.C + 1, c.C), dtype=torch.float32).cuda()
                check(decode(op, c, x, sl.cuda(), expansion_scores=table), c, "generic scorer", exact_flag=True)
    finally:
        op.set_beam_impl(None)
    assert modes == {False, True}


# ------------------------------------------------------------------------------------------------
# streaming, host feed
@pytest.mark.parametrize("c", NARROW + WIDE, ids=_ids(NARROW + WIDE))
def test_streaming_with_chunk_boundaries_at_the_deep_frames(op, c):
    """One chunk ends right before the deepest frame and one right after it (and, at T = 128, at the
    32/64 frame marks as well): the carried beam enters the fixed point's deepest frames."""
    t = int(np.argmax(c.iters))
    cuts = sorted({0, t, t + 1, c.T} | ({32, 64} if c.T >= 64 else set()))
    dec = op.CTCExtBeamSearchDecoderStream(batch_size=1, num_classes=c.C, beam_width=c.W, top_paths=c.P,
                                           max_time=c.T, merge_repeated=c.merge, blank_index=c.blank)
    for a, b in zip(cuts[:-1], cuts[1:]):
        if b > a:
            dec.step(np.ascontiguousarray(c.x[a:b]), np.array([b - a], np.int32))
    check(dec.top_paths_raw(), c, "stream cuts %s" % cuts)


@pytest.mark.parametrize("dt", ["float32", "bfloat16"])
@pytest.mark.parametrize("c", NARROW + WIDE, ids=_ids(NARROW + WIDE))
def test_page_locked_host_logits(op, c, dt):
    x, sl = inputs(c, dt, device="host")
    raw = decode(op, c, x, sl)
    assert not raw[6].is_cuda
    check(raw, c, "host " + dt)


# ------------------------------------------------------------------------------------------------
# the kernels' own counts (timing builds, through the measurement hook)
def _counted(op, c):
    import torch
    from ctc_beam_search_op_b200 import _lib
    lib = _lib.load()
    buf = torch.zeros((1, 24), dtype=torch.int64, device="cuda")
    x, sl = inputs(c, "float32")
    lib.ctcx_debug_set_cycles_buffer(buf.data_ptr())
    try:
        raw = decode(op, c, x, sl.cuda())
        torch.cuda.synchronize()
    finally:
        lib.ctcx_debug_set_cycles_buffer(None)
    check(raw, c, "timing build")
    return buf[0].cpu().numpy()


@pytest.mark.parametrize("c", NARROW, ids=_ids(NARROW))
def test_narrow_timing_build_counts_equal_the_model(op, c):
    """Slots 20, 22 and 23: at-risk members, wiped members (final verdicts) and frames with at-risk
    members, summed over the frames."""
    cyc = _counted(op, c)
    assert (cyc[20], cyc[22], cyc[23]) == (c.stats["at_risk"], c.stats["wiped"], c.stats["frames_at_risk"]), c.stats


def test_wide_timing_build_meets_capped_prefixes(op):
    """Slot 22: frames in which some row's candidates reach past the sorted prefix (2W + 2 classes)."""
    c = next(c for c in CASES if c.name.startswith("tied-"))
    assert c.stats["frames_at_risk"] > 0
    assert _counted(op, c)[22] > 0
