"""GPU parity tests proper: the CUDA path (through the C-ABI) against the CPU oracle on the same
seeded inputs. Labels, alignments and the float32 bits of log_probability must be IDENTICAL: the
device arithmetic reproduces the host libm bit for bit and the beam order is the oracle's stable
order (DESIGN.md "Numerics" / "Tie policy")."""
import numpy as np
import pytest

import ctcx_testlib as L

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module", params=["fast", "generic"])
def op(request):
    """Both beam-kernel families: the default dispatch (the fast kernels where they apply) and the
    generic kernel forced through the test hook ctcx_debug_set_beam_impl."""
    import torch
    if not torch.cuda.is_available():
        pytest.skip("no CUDA device")
    import ctc_beam_search_op_b200 as m
    m.set_beam_impl(request.param)
    yield m
    m.set_beam_impl(None)


def _dense_from_raw(raw, B, P, T):
    """Raw sparse outputs -> per (b,p) python lists."""
    dec = [[[] for _ in range(P)] for _ in range(B)]
    ali = [[[] for _ in range(P)] for _ in range(B)]
    for p in range(P):
        for (b, i), v in zip(np.asarray(raw[0][p]).tolist(), np.asarray(raw[1][p]).tolist()):
            assert i == len(dec[b][p])
            dec[b][p].append(v)
        for (b, i), v in zip(np.asarray(raw[3][p]).tolist(), np.asarray(raw[4][p]).tolist()):
            assert i == len(ali[b][p])
            ali[b][p].append(v)
    return dec, ali


def check_against_oracle(op, x, sl, W, P, merge, blank, blank_label, expect_all=True):
    T, B, C = x.shape
    want = L.oracle_decode(x, sl, W, P, merge, blank, blank_label)
    raw = op.ctc_ext_beam_search_decoder_raw(x, sl, beam_width=W, top_paths=P, merge_repeated=merge,
                                             blank_index=blank, blank_label=blank_label)
    packed = L.pack_sparse(want)
    bad = []
    dec, ali = _dense_from_raw(raw, B, P, T)
    for b in range(B):
        for p in range(P):
            if dec[b][p] != want.decoded(b, p) or ali[b][p] != want.alignment(b, p) or \
                    np.float32(raw[6][b, p]).view(np.uint32) != np.float32(want.logp[b, p]).view(np.uint32):
                bad.append((b, p))
    if expect_all:
        assert not bad, "mismatching (utterance, path): %s" % bad[:10]
        for g in range(6):
            for p in range(P):
                np.testing.assert_array_equal(np.asarray(raw[g][p]), packed[g][p])
    return bad


CASES = [
    # kind, T, B, C, W, P, merge, blank, blank_label, ragged
    ("gauss", 50, 8, 29, 10, 3, False, 28, -1, False),   # BASELINE cfg1
    ("peaky", 50, 8, 29, 10, 3, False, 28, -1, True),
    ("peaky", 60, 6, 29, 100, 1, True, 28, -1, False),   # cfg2 shape, short
    ("gauss", 60, 6, 29, 100, 1, True, 28, -1, True),
    ("gauss", 40, 4, 32, 64, 4, False, 31, -1, False),   # cfg3 shape, short
    ("peaky", 30, 3, 1024, 16, 1, False, 1023, -1, False),  # cfg4 shape, short (streaming mode)
    ("gauss", 30, 16, 6, 4, 4, True, 3, 1, True),
    ("gauss", 20, 16, 3, 2, 2, False, 1, 9, False),
    ("gauss", 20, 16, 5, 1, 1, True, 0, -1, False),
    ("gauss", 25, 4, 40, 200, 2, False, 7, -1, False),   # WMAX=256 tier (wide kernel)
    ("gauss", 30, 3, 29, 140, 2, False, 28, -1, False),  # WMAX=256 tier of the narrow fast kernel
    ("peaky", 40, 3, 12, 256, 3, True, 0, -1, True),     # beam_width = 256 exactly, narrow fast kernel
    ("gauss", 12, 2, 12, 300, 3, False, 0, -1, False),   # WMAX=1024 tier
]


@pytest.mark.parametrize("case", CASES, ids=lambda c: "%s-T%d-B%d-C%d-W%d-P%d" % c[:6])
def test_parity_small(op, case):
    kind, T, B, C, W, P, merge, blank, blank_label, ragged = case
    x = L.make_logits(kind, T, B, C, blank, seed=11)
    sl = L.ragged_lengths(T, B, 11) if ragged else np.full(B, T, np.int32)
    check_against_oracle(op, x, sl, W, P, merge, blank, blank_label)


def test_constant_logits_pathological_ties(op):
    """All classes equally likely: every child of a row ties exactly; the cut through the tied
    scores must follow the stable order (members, then (row, label))."""
    for (T, B, C, W, P) in [(12, 2, 8, 10, 3), (10, 2, 29, 100, 2), (8, 1, 4, 3, 3)]:
        x = np.zeros((T, B, C), np.float32)
        check_against_oracle(op, x, np.full(B, T, np.int32), W, P, False, C - 1, -1)
    # two distinct values only
    rng = np.random.default_rng(3)
    x = rng.integers(0, 2, (15, 4, 12)).astype(np.float32)
    check_against_oracle(op, x, np.full(4, 15, np.int32), 20, 4, True, 0, -1)


def _micro_spaced(T, B, C, seed, step, levels=None, ascending=True):
    """Logits whose classes differ by ~1e-6: after a few dozen frames the running scores are large
    enough that DIFFERENT log-probs round to the SAME sum, so the (score, label) order of a row's
    children is no longer the per-frame order of the log-probs."""
    rng = np.random.default_rng(seed)
    if levels is None:
        base = np.arange(C, dtype=np.float64) * step
        if not ascending:
            base = base[::-1]
        x = np.tile(base, (T, B, 1))
        for t in range(T):
            for b in range(B):
                if rng.random() < 0.5:  # some frames: a random class -> value assignment
                    x[t, b] = rng.permutation(base)
    else:
        x = rng.integers(0, levels, (T, B, C)).astype(np.float64) * step
    return x.astype(np.float32)


WIDE_CASES = [
    # kind, T, B, C, W, P, merge, blank  (all with 2W+2 < C-1: the beam kernel sees a truncated order)
    ("gauss", 60, 4, 100, 4, 2, False, 99),
    ("peaky", 60, 4, 300, 8, 3, True, 0),
    ("gauss", 50, 3, 1024, 16, 1, False, 1023),   # BASELINE cfg4 shape
    ("peaky", 40, 2, 2048, 5, 2, False, 17),
    ("gauss", 40, 3, 37, 1, 1, False, 5),
    ("gauss", 40, 3, 700, 40, 2, False, 3),       # WMAX=128 tier
]


@pytest.mark.parametrize("case", WIDE_CASES, ids=lambda c: "%s-T%d-C%d-W%d" % (c[0], c[1], c[3], c[4]))
def test_wide_vocabulary_truncated_order(op, case):
    kind, T, B, C, W, P, merge, blank = case
    x = L.make_logits(kind, T, B, C, blank, seed=31)
    check_against_oracle(op, x, L.ragged_lengths(T, B, 31), W, P, merge, blank, -1)


def test_wide_vocabulary_ties_beyond_the_sorted_classes(op):
    """Wide kernel corner: classes that were left out of the per-frame top-Kc order but tie exactly
    (after rounding) with the lowest selected item and precede it in label order must be swapped in."""
    full = lambda T, B: np.full(B, T, np.int32)
    # constant logits: every class of every row ties, every prefix is capped
    for (T, B, C, W, P) in [(20, 2, 64, 3, 3), (12, 2, 200, 16, 2), (10, 1, 1024, 2, 1)]:
        check_against_oracle(op, np.zeros((T, B, C), np.float32), full(T, B), W, P, False, C - 1, -1)
    # log-probs 1e-6 apart, higher label = higher log-prob: the sorted order starts at the highest
    # labels while the reference's order prefers the lowest label among equal sums
    for (T, B, C, W, P, step, asc, blank) in [(90, 3, 100, 2, 2, 1e-6, True, 0), (90, 3, 100, 2, 1, 1e-6, True, 99),
                                              (120, 2, 64, 4, 3, 3e-6, True, 10), (80, 2, 150, 3, 2, 1e-6, False, 7),
                                              (100, 2, 1024, 16, 2, 2e-7, True, 1023)]:
        x = _micro_spaced(T, B, C, 5, step, ascending=asc)
        check_against_oracle(op, x, full(T, B), W, P, False, blank, -1)
    # few distinct levels, tiny and coarse spacing (many exact ties + revisits)
    for (T, B, C, W, P, step, levels) in [(80, 3, 90, 3, 3, 1e-6, 3), (40, 3, 48, 6, 4, 1.0, 3),
                                          (60, 2, 120, 5, 2, 0.5, 2), (100, 2, 70, 2, 2, 5e-7, 4)]:
        x = _micro_spaced(T, B, C, 9, step, levels=levels)
        check_against_oracle(op, x, full(T, B), W, P, True, 1, -1)


F64_CASES = [
    # kind, T, B, C, W, P, merge, blank
    ("gauss", 40, 4, 29, 10, 3, False, 28),
    ("peaky", 60, 3, 29, 100, 1, True, 28),    # cfg2 shape, short
    ("gauss", 30, 3, 40, 24, 2, False, 7),
    ("peaky", 20, 2, 300, 8, 2, False, 0),     # streaming candidate mode
    ("gauss", 12, 2, 12, 300, 3, False, 0),    # WMAX=1024 tier
    ("gauss", 25, 2, 40, 200, 2, True, 39),    # WMAX=256 tier
    # the narrow fast kernel computing in double (num_classes <= 32): every beam tier
    ("gauss", 50, 3, 32, 32, 2, False, 31),
    ("peaky", 70, 3, 20, 128, 3, True, 4),
    ("gauss", 40, 2, 12, 256, 2, False, 0),
    ("gauss", 33, 700, 9, 6, 1, True, 8),      # more utterances than resident CTAs: the work queue
]


@pytest.mark.parametrize("case", F64_CASES, ids=lambda c: "%s-T%d-C%d-W%d" % (c[0], c[1], c[3], c[4]))
def test_float64_decode_is_bit_exact(op, case):
    """T = double (kernels.cc:275; the reference's own test feeds float64): decoded in float64 by the
    double instantiations of the narrow fast kernel (num_classes <= 32) and of the generic kernel,
    identical to the float64 oracle down to the bits."""
    kind, T, B, C, W, P, merge, blank = case
    rng = np.random.default_rng(41)
    x = rng.standard_normal((T, B, C))  # genuine float64 values
    if kind == "peaky":
        x += L.make_logits("peaky", T, B, C, blank, 41).astype(np.float64) - L.make_logits("gauss", T, B, C, blank, 41)
    sl = L.ragged_lengths(T, B, 41)
    want = L.oracle_decode(x, sl, W, P, merge, blank, -1)
    assert want.logp.dtype == np.float64
    raw = op.ctc_ext_beam_search_decoder_raw(x, sl, beam_width=W, top_paths=P, merge_repeated=merge,
                                             blank_index=blank, blank_label=-1)
    packed = L.pack_sparse(want)
    for g in range(6):
        for p in range(P):
            np.testing.assert_array_equal(np.asarray(raw[g][p]), packed[g][p])
    assert np.asarray(raw[6]).dtype == np.float64
    np.testing.assert_array_equal(np.asarray(raw[6]).view(np.uint64), np.asarray(packed[6], np.float64).view(np.uint64))
    host = op.decode_host_cabi(x, sl, W, P, merge, blank, -1)  # ctcx_decode_host_f64
    assert host[6].dtype == np.float64
    np.testing.assert_array_equal(host[6].view(np.uint64), np.asarray(raw[6]).view(np.uint64))
    for g in range(6):
        for p in range(P):
            np.testing.assert_array_equal(host[g][p], packed[g][p])
    if W == 300:  # float64 state is twice as wide: beam widths above 512 are refused, never degraded
        with pytest.raises(op.CtcxError, match="not supported"):
            op.ctc_ext_beam_search_decoder_raw(x, sl, beam_width=600, top_paths=1, blank_index=blank)
    # device tensors in, device tensors out
    import torch
    rd = op.ctc_ext_beam_search_decoder_raw(torch.from_numpy(x).cuda(), torch.from_numpy(sl).cuda(), beam_width=W,
                                            top_paths=P, merge_repeated=merge, blank_index=blank)
    assert rd[6].dtype == torch.float64 and rd[6].is_cuda
    np.testing.assert_array_equal(rd[6].cpu().numpy().view(np.uint64), np.asarray(raw[6]).view(np.uint64))


# ------------------------------------------------------------------------------------------------
# The reference's own test, transliterated (ops_test.py:20-100): raw 7-group output, float64 input
def test_paper_known_answer_like_the_reference(op):
    logits = L.paper_logits(np.float64)
    correct_decoded_values = [[1, 1, 2], [1, 2, 1, 2], [1, 2], [1, 1, 2, 1], [1, 2, 1]]
    correct_alignment_values = [[1, 1, 0, 1, 0, 2, 2, 2], [1, 1, 0, 2, 1, 2, 2, 2], [1, 1, 0, 0, 0, 2, 2, 2],
                                [1, 1, 0, 1, 0, 2, 2, 1], [1, 1, 0, 0, 0, 2, 2, 1]]
    correct_log_probs = np.array([[-2.0613022, -2.1155741, -2.713197, -2.8770373, -2.9212725]])
    out = op.ctc_ext_beam_search_decoder_raw(inputs=logits, sequence_length=[8], beam_width=10,
                                             blank_index=0, top_paths=5, blank_label=0,
                                             merge_repeated=False)
    for p in range(5):
        np.testing.assert_allclose(out[0][p], [[0, i] for i in range(len(correct_decoded_values[p]))])
        np.testing.assert_allclose(out[1][p], correct_decoded_values[p])
        np.testing.assert_allclose(out[2][p], [1, len(correct_decoded_values[p])])
        np.testing.assert_allclose(out[3][p], [[0, i] for i in range(8)])
        np.testing.assert_allclose(out[4][p], correct_alignment_values[p])
        np.testing.assert_allclose(out[5][p], [1, 8])
    np.testing.assert_allclose(out[6], correct_log_probs, rtol=1e-6, atol=1e-6)
    assert out[6].dtype == np.float64
    # float64 is computed in float64: identical to the compiled reference's float64 output
    ref64 = L.Golden().result("paper_f64").logp
    assert ref64.dtype == np.float64
    np.testing.assert_array_equal(np.asarray(out[6]).view(np.uint64), ref64.view(np.uint64))
    # documented return value: (decoded, alignment, log_probability) with SparseTensor-like entries
    dec, ali, lp = op.ctc_ext_beam_search_decoder(logits, [8], beam_width=10, top_paths=5,
                                                  blank_index=0, blank_label=0)
    assert dec[0].values.tolist() == [1, 1, 2] and ali[0].dense_shape.tolist() == [1, 8]


def test_no_leak_over_many_calls(op):
    """Counterpart of testCTCExtBeamSearchDecoderMemLeak (ops_test.py:102-123): device memory in
    use must not grow over repeated calls."""
    import torch
    x = torch.from_numpy(L.paper_logits(np.float32)).cuda()
    sl = torch.tensor([8], dtype=torch.int32).cuda()
    kw = dict(beam_width=10, top_paths=5, blank_index=0, blank_label=0)
    op.ctc_ext_beam_search_decoder_raw(x, sl, **kw)
    torch.cuda.synchronize()
    before = torch.cuda.memory_allocated()
    free0 = torch.cuda.mem_get_info()[0]
    for _ in range(300):
        op.ctc_ext_beam_search_decoder_raw(x, sl, **kw)
    torch.cuda.synchronize()
    assert torch.cuda.memory_allocated() <= before
    assert torch.cuda.mem_get_info()[0] >= free0 - (64 << 20)


def test_golden_reference_outputs(op):
    """Fixtures generated from the reference itself (tests/golden/make_golden.py)."""
    g = L.Golden()
    for name, x, sl, W, P, merge, blank, bl in g.random_cases() + g.literal_cases():
        want = g.result(name)
        raw = op.ctc_ext_beam_search_decoder_raw(x, sl, beam_width=W, top_paths=P, merge_repeated=merge,
                                                 blank_index=blank, blank_label=bl)
        B, T = x.shape[1], x.shape[0]
        dec, ali = _dense_from_raw(raw, B, P, T)
        tf = g.tie_free(name)
        for b in range(B):
            if tf is not None and not tf[b]:
                continue  # exact tie in an order-deciding comparison: reference order unspecified
            for p in range(P):
                assert dec[b][p] == want.decoded(b, p), (name, b, p)
                assert ali[b][p] == want.alignment(b, p), (name, b, p)
                if x.dtype == np.float32:
                    assert np.float32(raw[6][b, p]).view(np.uint32) == np.float32(want.logp[b, p]).view(np.uint32)
                else:  # float64 inputs are computed in float32 (DESIGN.md "next" row f1)
                    np.testing.assert_allclose(raw[6][b, p], want.logp[b, p], rtol=1e-4)


def test_host_buffer_cabi_entry(op):
    """ctcx_decode_host_f32: what a TF CPU OpKernel would call with host tensors."""
    x = L.make_logits("peaky", 40, 5, 29, 28, 21)
    sl = L.ragged_lengths(40, 5, 21)
    want = L.pack_sparse(L.oracle_decode(x, sl, 10, 2, True, 28, -1))
    got = op.decode_host_cabi(x, sl, beam_width=10, top_paths=2, merge_repeated=True, blank_index=28)
    for g in range(6):
        for p in range(2):
            np.testing.assert_array_equal(got[g][p], want[g][p])
    np.testing.assert_array_equal(got[6].view(np.uint32), want[6].view(np.uint32))


def test_torch_device_tensors_in_device_tensors_out(op):
    import torch
    x = L.make_logits("peaky", 30, 4, 12, 11, 4)
    sl = np.full(4, 30, np.int32)
    dec, ali, lp = op.ctc_ext_beam_search_decoder(torch.from_numpy(x).cuda(), torch.from_numpy(sl).cuda(),
                                                  beam_width=8, top_paths=2, blank_index=11)
    assert dec[0].indices.is_cuda and ali[1].values.is_cuda and lp.is_cuda and lp.shape == (4, 2)
    want = L.pack_sparse(L.oracle_decode(x, sl, 8, 2, False, 11, -1))
    np.testing.assert_array_equal(ali[1].values.cpu().numpy(), want[4][1])


def test_edge_cases(op):
    x = L.make_logits("gauss", 6, 3, 4, 0, 9)
    # sequence_length 0 with one path: empty sequences, log-prob 0 (SURVEY.md Appendix D)
    raw = op.ctc_ext_beam_search_decoder_raw(x, [0, 6, 3], beam_width=4, top_paths=1)
    want = L.pack_sparse(L.oracle_decode(x, np.asarray([0, 6, 3], np.int32), 4, 1, False, 0, -1))
    for g in range(6):
        np.testing.assert_array_equal(raw[g][0], want[g][0])
    assert raw[6][0, 0] == 0.0
    # empty batch
    raw = op.ctc_ext_beam_search_decoder_raw(np.zeros((5, 0, 4), np.float32), np.zeros((0,), np.int32),
                                             beam_width=4, top_paths=2)
    assert raw[0][0].shape == (0, 2) and raw[6].shape == (0, 2) and raw[2][1].tolist() == [0, 0]
    # beam wider than anything reachable, blank in the middle, custom blank label
    check_against_oracle(op, x, np.full(3, 6, np.int32), 64, 3, True, 2, 7)


def test_device_side_errors(op):
    x = L.paper_logits(np.float32)
    with pytest.raises(op.InvalidArgumentError, match="requested more paths than the beam width"):
        op.ctc_ext_beam_search_decoder(x, [8], beam_width=2, top_paths=3)
    with pytest.raises(op.InvalidArgumentError, match="Less leaves in the beam search than requested"):
        op.ctc_ext_beam_search_decoder(x[:1], [1], beam_width=4, top_paths=4)
    with pytest.raises(op.InvalidArgumentError, match="Less leaves"):
        op.ctc_ext_beam_search_decoder(x, [0], beam_width=4, top_paths=2)
    with pytest.raises(op.FailedPreconditionError, match=r"sequence_length\(0\) <= 8"):
        op.ctc_ext_beam_search_decoder(x, [9], beam_width=4, top_paths=1)
    with pytest.raises(op.InvalidArgumentError):  # rejected here, undefined behaviour in the reference
        op.ctc_ext_beam_search_decoder(x, [8], beam_width=4, top_paths=1, blank_index=3)
    with pytest.raises(op.InvalidArgumentError):
        op.ctc_ext_beam_search_decoder(x, [-1], beam_width=4, top_paths=1)
    with pytest.raises(op.UnsupportedError):
        op.ctc_ext_beam_search_decoder(x, [8], beam_width=5000, top_paths=1)


def test_multi_device_sharding_equals_single(op):
    """Batch cut into blocks (here: three blocks on the same GPU) and merged on the host."""
    x = L.make_logits("peaky", 25, 7, 10, 9, 13)
    sl = L.ragged_lengths(25, 7, 13)
    whole = op.ctc_ext_beam_search_decoder_raw(x, sl, beam_width=6, top_paths=2, merge_repeated=True, blank_index=9)
    import torch
    layouts = [[0, 0, 0]]
    if torch.cuda.device_count() >= 2:  # really different devices where the box has them
        layouts += [[0, 1], [1, 0, 1]]
    for devices in layouts:
        parts = op.decode_multi_device(x, sl, 6, 2, True, 9, -1, devices=devices)
        for g in range(6):
            for p in range(2):
                np.testing.assert_array_equal(parts[g][p], whole[g][p])
        np.testing.assert_array_equal(parts[6], whole[6])
    if torch.cuda.device_count() >= 2:  # a tensor living on the second device is decoded there
        r1 = op.ctc_ext_beam_search_decoder_raw(torch.from_numpy(x).to("cuda:1"), torch.from_numpy(sl).to("cuda:1"),
                                                beam_width=6, top_paths=2, merge_repeated=True, blank_index=9)
        assert r1[6].device == torch.device("cuda", 1)
        np.testing.assert_array_equal(r1[6].cpu().numpy(), np.asarray(whole[6]))
        np.testing.assert_array_equal(r1[4][0].cpu().numpy(), np.asarray(whole[4][0]))


# ------------------------------------------------------------------------------------------------
# BASELINE.json sizes: parity on a subset against the oracle + size-independent properties on all
def _collapse(ali_row, blank_label, merge):
    out, prev = [], None
    for s in ali_row:
        if s != blank_label and s != prev:
            out.append(s)
        prev = s
    if merge:
        out = [v for i, v in enumerate(out) if i == 0 or v != out[i - 1]]
    return out


FULL = [
    # name, T, B, C, W, P, merge, blank, oracle utterances
    ("cfg2", 500, 256, 29, 100, 1, True, 28, 6),
    ("cfg3", 1500, 64, 32, 64, 4, False, 31, 2),
    ("cfg4", 400, 128, 1024, 16, 1, False, 1023, 2),
]


@pytest.mark.parametrize("cfg", FULL, ids=lambda c: c[0])
def test_full_size_properties_and_subset_parity(op, cfg):
    import torch
    name, T, B, C, W, P, merge, blank, n_oracle = cfg
    x = L.make_logits("peaky", T, B, C, blank, seed=31)
    sl = L.ragged_lengths(T, B, 31)
    raw = op.ctc_ext_beam_search_decoder_raw(x, sl, beam_width=W, top_paths=P, merge_repeated=merge,
                                             blank_index=blank, blank_label=-1)
    dec, ali = _dense_from_raw(raw, B, P, T)
    lp = np.asarray(raw[6])
    for b in range(B):
        for p in range(P):
            assert len(ali[b][p]) == sl[b]                       # one alignment symbol per frame
            # the decoded path is the CTC collapse of its own best alignment (blank_label=-1 is no class)
            assert dec[b][p] == _collapse(ali[b][p], -1, merge)
            assert all(0 <= v < C and v != blank for v in dec[b][p])
        assert all(lp[b, p] >= lp[b, p + 1] for p in range(P - 1))  # paths best-first
        assert np.all(lp[b] <= 0)
    for p in range(P):  # shapes = [batch, longest]
        assert raw[2][p].tolist() == [B, max(len(dec[b][p]) for b in range(B))]
        assert raw[5][p].tolist() == [B, int(sl.max())]
    # idempotence / order independence: a permuted batch gives the permuted result
    perm = np.random.default_rng(0).permutation(B)
    raw2 = op.ctc_ext_beam_search_decoder_raw(np.ascontiguousarray(x[:, perm]), sl[perm], beam_width=W,
                                              top_paths=P, merge_repeated=merge, blank_index=blank)
    dec2, ali2 = _dense_from_raw(raw2, B, P, T)
    for i, b in enumerate(perm):
        assert dec2[i] == dec[b] and ali2[i] == ali[b]
    np.testing.assert_array_equal(np.asarray(raw2[6]), lp[perm])
    # bit-exact parity against the oracle on the first utterances
    want = L.oracle_decode(x[:, :n_oracle], sl[:n_oracle], W, P, merge, blank, -1)
    for b in range(n_oracle):
        for p in range(P):
            assert dec[b][p] == want.decoded(b, p) and ali[b][p] == want.alignment(b, p)
            assert np.float32(lp[b, p]).view(np.uint32) == np.float32(want.logp[b, p]).view(np.uint32)
    assert raw.flags == 0 and raw2.flags == 0  # no utterance hit the documented rounding anomaly


# ------------------------------------------------------------------------------------------------
# Streaming: Step / TopPaths / Reset (decoder.h:39-53). Any chunking == one-shot == oracle.
STREAM_CASES = [
    # kind, T, B, C, W, P, merge, blank
    ("peaky", 70, 5, 29, 100, 2, True, 28),    # fast kernel
    ("gauss", 40, 4, 29, 10, 3, False, 28),    # fast kernel, small tier
    ("gauss", 30, 3, 40, 24, 2, False, 7),     # wide kernel, all classes sorted (generic when forced)
    ("peaky", 24, 2, 1024, 16, 1, False, 1023),  # wide kernel (generic: streaming candidate mode)
    ("gauss", 36, 3, 120, 6, 2, True, 0),        # wide kernel, truncated class order
]


@pytest.mark.parametrize("case", STREAM_CASES, ids=lambda c: "%s-T%d-C%d-W%d" % (c[0], c[1], c[3], c[4]))
def test_streaming_equals_one_shot_and_oracle(op, case):
    kind, T, B, C, W, P, merge, blank = case
    rng = np.random.default_rng(17)
    x = L.make_logits(kind, T, B, C, blank, seed=23)
    sl = L.ragged_lengths(T, B, 23)
    dec = op.CTCExtBeamSearchDecoderStream(batch_size=B, num_classes=C, beam_width=W, top_paths=P,
                                           max_time=T, merge_repeated=merge, blank_index=blank, blank_label=-1)
    for rep in range(2):  # the second pass checks reset()
        t = 0
        while t < T:
            ct = int(rng.integers(1, 12))
            ct = min(ct, T - t)
            lens = np.clip(sl - t, 0, ct).astype(np.int32)
            dec.step(x[t:t + ct], lens)
            t += ct
            if t in (ct, T) or rng.random() < 0.3:  # TopPaths mid-stream == oracle on the prefix
                done = np.minimum(sl, t).astype(np.int32)
                if P == 1 or done.min() >= 2:
                    raw = dec.top_paths_raw()
                    want = L.pack_sparse(L.oracle_decode(x[:t], done, W, P, merge, blank, -1))
                    for g in range(6):
                        for p in range(P):
                            np.testing.assert_array_equal(raw[g][p].cpu().numpy(), want[g][p])
                    np.testing.assert_array_equal(raw[6].cpu().numpy().view(np.uint32), want[6].view(np.uint32))
        raw = dec.top_paths_raw()
        one = op.ctc_ext_beam_search_decoder_raw(x, sl, beam_width=W, top_paths=P, merge_repeated=merge,
                                                 blank_index=blank)
        for g in range(6):
            for p in range(P):
                np.testing.assert_array_equal(raw[g][p].cpu().numpy(), one[g][p])
        np.testing.assert_array_equal(raw[6].cpu().numpy().view(np.uint32), np.asarray(one[6]).view(np.uint32))
        dec.reset()


def test_streaming_overflow_and_errors(op):
    x = L.make_logits("peaky", 12, 2, 6, 5, 3)
    dec = op.CTCExtBeamSearchDecoderStream(2, 6, 4, 1, max_time=8, blank_index=5)
    dec.step(x[:6])
    dec.step(x[6:12])  # 12 frames into a stream sized for 8
    with pytest.raises(op.FailedPreconditionError, match=r"sequence_length\(0\) <= 8"):
        dec.top_paths()
    dec.reset()
    dec.step(x[:8])
    d, a, lp = dec.top_paths()
    want = L.pack_sparse(L.oracle_decode(x[:8], np.full(2, 8, np.int32), 4, 1, False, 5, -1))
    np.testing.assert_array_equal(a[0].values.cpu().numpy(), want[4][0])
    with pytest.raises(op.InvalidArgumentError):
        dec.step(x[:, :1])  # wrong batch


def test_reference_import_path(op):
    """The reference test's own import line and call (ops_test.py:12-15, :67-69) work unchanged."""
    from tensorflow_ctc_ext_beam_search_decoder.python.ops.ctc_ext_beam_search_decoder_ops import \
        ctc_ext_beam_search_decoder
    out = ctc_ext_beam_search_decoder(inputs=L.paper_logits(np.float64), sequence_length=[8], beam_width=10,
                                      blank_index=0, top_paths=5, blank_label=0, merge_repeated=False)
    np.testing.assert_allclose(out[1][0], [1, 1, 2])
    np.testing.assert_allclose(out[6], [[-2.0613022, -2.1155741, -2.713197, -2.8770373, -2.9212725]],
                               rtol=1e-6, atol=1e-6)


# ------------------------------------------------------------------------------------------------
# Shape fuzz: small random configurations around the tier / vocabulary boundaries, every kernel.
def _fuzz_cases():
    rng = np.random.default_rng(2024)
    cases = []
    fixed = [(1, 1, 2, 1, 1), (3, 2, 2, 4, 2), (5, 1, 1, 3, 1), (9, 3, 32, 32, 4), (7, 2, 33, 33, 3),
             (6, 2, 31, 128, 5), (6, 2, 32, 129, 2), (5, 2, 17, 256, 3), (4, 1, 9, 257, 2),
             (12, 2, 29, 159, 1), (8, 2, 64, 72, 2), (8, 2, 65, 70, 2), (10, 2, 3, 100, 7)]
    for T, B, C, W, P in fixed:
        cases.append((T, B, C, W, P, int(rng.integers(0, C)), bool(rng.integers(0, 2)),
                      ["gauss", "peaky"][int(rng.integers(0, 2))], float(rng.choice([0.5, 1, 3])), int(rng.integers(0, 9999))))
    for _ in range(40):
        C = int(rng.choice([2, 3, 5, 8, 16, 29, 31, 32, 33, 40, 100]))
        W = int(rng.choice([1, 2, 3, 7, 16, 31, 32, 33, 64, 100, 128, 130, 200]))
        T = int(rng.integers(1, 40))
        B = int(rng.integers(1, 6))
        P = int(rng.integers(1, min(W, 4) + 1))
        cases.append((T, B, C, W, P, int(rng.integers(0, C)), bool(rng.integers(0, 2)),
                      ["gauss", "peaky"][int(rng.integers(0, 2))], float(rng.choice([0.5, 1, 3])), int(rng.integers(0, 9999))))
    return cases


def test_fuzz_shapes(op):
    n_err = 0
    for T, B, C, W, P, blank, merge, kind, sigma, seed in _fuzz_cases():
        if C == 1:
            x = np.random.default_rng(seed).standard_normal((T, B, 1)).astype(np.float32)
        else:
            x = L.make_logits(kind, T, B, C, blank, seed, sigma)
        sl = L.ragged_lengths(T, B, seed)
        try:
            want = L.oracle_decode(x, sl, W, P, merge, blank, -1)
        except L.OracleError as e:
            with pytest.raises(op.CtcxError, match=str(e)[:24]):
                op.ctc_ext_beam_search_decoder_raw(x, sl, beam_width=W, top_paths=P, merge_repeated=merge,
                                                   blank_index=blank)
            n_err += 1
            continue
        raw = op.ctc_ext_beam_search_decoder_raw(x, sl, beam_width=W, top_paths=P, merge_repeated=merge,
                                                 blank_index=blank, blank_label=-1)
        packed = L.pack_sparse(want)
        for g in range(6):
            for p in range(P):
                np.testing.assert_array_equal(np.asarray(raw[g][p]), packed[g][p],
                                              err_msg="T=%d B=%d C=%d W=%d P=%d blank=%d" % (T, B, C, W, P, blank))
        np.testing.assert_array_equal(np.asarray(raw[6]).view(np.uint32), packed[6].view(np.uint32))
    assert n_err < 30


@pytest.mark.parametrize("dt", ["float16", "bfloat16"])
def test_half_precision_logits(op, dt):
    """fp16 / bf16 logits: the result must equal the oracle run on the (exactly) upcast values."""
    import torch
    tdt = getattr(torch, dt)
    x32 = L.make_logits("peaky", 40, 5, 29, 28, 41)
    xh = torch.from_numpy(x32).to(tdt)
    up = xh.to(torch.float32).numpy()
    sl = L.ragged_lengths(40, 5, 41)
    want = L.pack_sparse(L.oracle_decode(up, sl, 20, 2, True, 28, -1))
    for inp in (xh, xh.cuda()):
        raw = op.ctc_ext_beam_search_decoder_raw(inp, sl, beam_width=20, top_paths=2, merge_repeated=True,
                                                 blank_index=28)
        for g in range(6):
            for p in range(2):
                np.testing.assert_array_equal(raw[g][p].cpu().numpy(), want[g][p])
        np.testing.assert_array_equal(raw[6].cpu().numpy().view(np.uint32), want[6].view(np.uint32))


def test_torch_library_op(op):
    """torch.ops.ctcx.ctc_ext_beam_search_decoder == the raw Python entry; opcheck validates the
    schema / fake-tensor registration against the real kernels."""
    import torch
    T, B, C, W, P = 40, 5, 29, 10, 3
    x = torch.from_numpy(L.make_logits("peaky", T, B, C, 28, 7)).cuda()
    sl = torch.from_numpy(L.ragged_lengths(T, B, 7)).cuda()
    flat = torch.ops.ctcx.ctc_ext_beam_search_decoder(x, sl, W, P, True, 28, -1)
    got = op.torch_op.unflatten(flat, P)
    want = op.ctc_ext_beam_search_decoder_raw(x, sl, beam_width=W, top_paths=P, merge_repeated=True, blank_index=28)
    for g in range(6):
        for p in range(P):
            assert torch.equal(got[g][p], want[g][p])
    assert torch.equal(got[6], want[6])
    torch.library.opcheck(torch.ops.ctcx.ctc_ext_beam_search_decoder.default, (x, sl, W, P, True, 28, -1),
                          test_utils=("test_schema", "test_faketensor"))


def test_scorer_extension_point(op):
    """ctcx_decode_scorer_f32: a [C+1, C] expansion-score table plugged into the reference's
    BaseBeamScorer call sites (decoder.h:103,114,171-182). GPU == oracle bit-for-bit for random
    bigram tables; the constant-table case is pinned against the compiled reference in
    tests/test_oracle.py."""
    rng = np.random.default_rng(77)
    for (kind, T, B, C, W, P, merge, blank) in [("gauss", 50, 5, 29, 10, 3, False, 28), ("peaky", 60, 4, 29, 100, 2, True, 28),
                                                ("peaky", 30, 3, 120, 6, 2, False, 0), ("gauss", 25, 2, 40, 200, 2, False, 7),
                                                # the narrow kernel's scorer variant: every beam tier, a full
                                                # 32-class row, blank in the middle, a batch that is time-sliced
                                                ("gauss", 40, 3, 32, 32, 2, True, 31), ("peaky", 80, 4, 12, 256, 1, False, 5),
                                                ("gauss", 45, 3, 17, 130, 2, False, 0), ("gauss", 64, 640, 10, 8, 1, True, 3)]:
        x = L.make_logits(kind, T, B, C, blank, 13)
        sl = L.ragged_lengths(T, B, 13)
        for table in (-np.abs(rng.standard_normal((C + 1, C))).astype(np.float32) * 2,
                      np.full((C + 1, C), -1.25, np.float32)):
            want = L.oracle_decode(x, sl, W, P, merge, blank, -1, lm=table)
            raw = op.ctc_ext_beam_search_decoder_raw(x, sl, beam_width=W, top_paths=P, merge_repeated=merge,
                                                     blank_index=blank, blank_label=-1, expansion_scores=table)
            packed = L.pack_sparse(want)
            for g in range(6):
                for p in range(P):
                    np.testing.assert_array_equal(np.asarray(raw[g][p]), packed[g][p])
            np.testing.assert_array_equal(np.asarray(raw[6]).view(np.uint32), packed[6].view(np.uint32))
        # a zero table is the default scorer
        zero = op.ctc_ext_beam_search_decoder_raw(x, sl, beam_width=W, top_paths=P, merge_repeated=merge,
                                                  blank_index=blank, expansion_scores=np.zeros((C + 1, C), np.float32))
        plain = op.ctc_ext_beam_search_decoder_raw(x, sl, beam_width=W, top_paths=P, merge_repeated=merge, blank_index=blank)
        np.testing.assert_array_equal(np.asarray(zero[6]).view(np.uint32), np.asarray(plain[6]).view(np.uint32))
        assert all(np.array_equal(zero[4][p], plain[4][p]) for p in range(P))
    # positive entries are refused (the gate decoder.h:157 is only redundant for log-probabilities)
    bad = np.zeros((30, 29), np.float32)
    bad[3, 4] = 0.5
    with pytest.raises(op.CtcxError):
        op.ctc_ext_beam_search_decoder_raw(L.make_logits("gauss", 10, 2, 29, 28, 1), [10, 10], beam_width=4, top_paths=1,
                                           blank_index=28, expansion_scores=bad)
    with pytest.raises(op.CtcxError):
        op.ctc_ext_beam_search_decoder_raw(L.make_logits("gauss", 10, 2, 29, 28, 1), [10, 10], beam_width=4, top_paths=1,
                                           blank_index=28, expansion_scores=np.zeros((29, 29), np.float32))


def test_masked_logits_minus_infinity(op):
    """-inf logits (vocabulary masking): probability exactly 0 for those classes. The reference
    handles them through kLogZero (loss_util.h:19-22, decoder.h:151 `total > kLogZero`); oracle ==
    compiled reference on such inputs (checked on the CPU), GPU == oracle here. The blank stays
    finite (a frame with every class at -inf is NaN in the reference as well)."""
    rng = np.random.default_rng(0)
    for (kind, T, B, C, W, P, merge, blank, frac) in [("gauss", 40, 6, 12, 8, 3, False, 11, 0.2),
                                                      ("peaky", 60, 4, 29, 20, 2, True, 28, 0.3),
                                                      ("gauss", 30, 4, 40, 16, 2, False, 0, 0.5),
                                                      ("gauss", 30, 4, 8, 100, 4, False, 7, 0.4),
                                                      ("peaky", 40, 3, 200, 6, 2, False, 199, 0.9),   # wide, few finite classes
                                                      ("gauss", 30, 2, 1024, 16, 1, False, 1023, 0.5),
                                                      ("gauss", 50, 3, 29, 100, 1, True, 28, 0.6)]:
        x = L.make_logits(kind, T, B, C, blank, 5)
        mask = rng.random((T, B, C)) < frac
        mask[..., blank] = False
        x = np.where(mask, -np.inf, x).astype(np.float32)
        check_against_oracle(op, x, L.ragged_lengths(T, B, 5), W, P, merge, blank, -1)
    # a label that is masked in every frame never appears; float64 path too
    x = L.make_logits("gauss", 30, 3, 10, 9, 8).astype(np.float64)
    x[:, :, 4] = -np.inf
    sl = np.full(3, 30, np.int32)
    want = L.oracle_decode(x, sl, 12, 3, False, 9, -1)
    raw = op.ctc_ext_beam_search_decoder_raw(x, sl, beam_width=12, top_paths=3, blank_index=9)
    packed = L.pack_sparse(want)
    for g in range(6):
        for p in range(3):
            np.testing.assert_array_equal(np.asarray(raw[g][p]), packed[g][p])
    np.testing.assert_array_equal(np.asarray(raw[6]).view(np.uint64), packed[6].view(np.uint64))
    assert all(4 not in np.asarray(raw[1][p]).tolist() for p in range(3))


def test_streaming_steps_replayed_from_a_cuda_graph(op):
    """The step call only enqueues kernels (no synchronisation, no allocation), so a chunk step can be
    captured once into a CUDA graph and replayed for every chunk: same result as the one-shot decode."""
    import torch
    for (T, B, C, W, P, blank, Tc) in [(64, 6, 29, 20, 2, 28, 8), (48, 3, 300, 8, 1, 0, 6)]:
        x = L.make_logits("peaky", T, B, C, blank, 19)
        sl = np.full(B, T, np.int32)
        dec = op.CTCExtBeamSearchDecoderStream(batch_size=B, num_classes=C, beam_width=W, top_paths=P,
                                               max_time=T, merge_repeated=True, blank_index=blank)
        x_static = torch.zeros((Tc, B, C), dtype=torch.float32, device="cuda")
        l_static = torch.full((B,), Tc, dtype=torch.int32, device="cuda")
        side = torch.cuda.Stream()
        side.wait_stream(torch.cuda.current_stream())
        with torch.cuda.stream(side):  # warm-up outside the capture (module loading, attributes)
            dec.step_device(x_static, l_static)
        torch.cuda.current_stream().wait_stream(side)
        dec.reset()
        g = torch.cuda.CUDAGraph()
        with torch.cuda.graph(g):
            dec.step_device(x_static, l_static)
        dec.reset()  # the capture itself does not run the step
        xd = torch.from_numpy(x).cuda()
        for t in range(0, T, Tc):
            x_static.copy_(xd[t:t + Tc])
            g.replay()
        raw = dec.top_paths_raw()
        one = op.ctc_ext_beam_search_decoder_raw(x, sl, beam_width=W, top_paths=P, merge_repeated=True,
                                                 blank_index=blank)
        for gi in range(6):
            for p in range(P):
                np.testing.assert_array_equal(raw[gi][p].cpu().numpy(), one[gi][p])
        np.testing.assert_array_equal(raw[6].cpu().numpy().view(np.uint32), np.asarray(one[6]).view(np.uint32))


def test_side_stream_and_non_contiguous_inputs(op):
    """The op runs on the caller's current stream and accepts strided views (host and device)."""
    import torch
    T, B, C, W, P = 40, 6, 29, 12, 2
    big = L.make_logits("peaky", T, 2 * B, C, 28, 29)
    x = big[:, ::2, :]                       # non-contiguous numpy view
    sl = L.ragged_lengths(T, B, 29)
    want = L.pack_sparse(L.oracle_decode(np.ascontiguousarray(x), sl, W, P, True, 28, -1))
    kw = dict(beam_width=W, top_paths=P, merge_repeated=True, blank_index=28)
    for raw in (op.ctc_ext_beam_search_decoder_raw(x, sl, **kw),
                op.ctc_ext_beam_search_decoder_raw(torch.from_numpy(big).cuda()[:, ::2, :], torch.from_numpy(sl).cuda(), **kw)):
        for g in range(6):
            for p in range(P):
                np.testing.assert_array_equal(np.asarray(raw[g][p].cpu() if hasattr(raw[g][p], "cpu") else raw[g][p]), want[g][p])
    side = torch.cuda.Stream()
    xd, sd = torch.from_numpy(np.ascontiguousarray(x)).cuda(), torch.from_numpy(sl).cuda()
    torch.cuda.synchronize()
    with torch.cuda.stream(side):
        xs = xd * 1.0                        # produced on the side stream: the decode must be ordered after it
        raw = op.ctc_ext_beam_search_decoder_raw(xs, sd, **kw)
        lp = raw[6].clone()
    side.synchronize()
    np.testing.assert_array_equal(lp.cpu().numpy().view(np.uint32), want[6].view(np.uint32))
    np.testing.assert_array_equal(raw[4][0].cpu().numpy(), want[4][0])


# ------------------------------------------------------------------------------------------------
# Round 2: host-input decode with the copy overlapped, views decoded in place, flags in the result
@pytest.mark.parametrize("dt", ["float32", "bfloat16"])
def test_pinned_host_logits_of_a_wide_vocabulary_are_decoded_slab_by_slab(op, dt):
    """Wide vocabularies from page-locked host memory: the copy is cut into time slabs and the decode
    follows it chunk by chunk (one event per slab; the beam crosses chunks through the state block).
    Ragged lengths -- utterances that end inside the first slab, at a slab boundary, empty ones -- and
    top_paths > 1 must give the oracle's result, as the one-shot decode of the device copy does."""
    import torch
    T, B, C, W, P, blank = 130, 9, 300, 16, 3, 299
    x32 = L.make_logits("peaky", T, B, C, blank, 61)
    xh = torch.from_numpy(x32).to(getattr(torch, dt)).pin_memory()
    up = xh.to(torch.float32).numpy()
    sl = np.array([130, 1, 5, 16, 17, 65, 129, 32, 100], np.int32)
    want = L.oracle_decode(up, sl, W, P, False, blank, -1)
    for _ in range(2):
        raw = op.ctc_ext_beam_search_decoder_raw(xh, sl, beam_width=W, top_paths=P, blank_index=blank)
        assert not raw[6].is_cuda
        assert not L.raw_mismatches(raw, want)
    # empty utterances (one leaf: top_paths 1), merge_repeated
    sl0 = np.array([0, 130, 0, 48, 49, 0, 2, 97, 0], np.int32)
    raw0 = op.ctc_ext_beam_search_decoder_raw(xh, sl0, beam_width=W, top_paths=1, merge_repeated=True, blank_index=blank)
    assert not L.raw_mismatches(raw0, L.oracle_decode(up, sl0, W, 1, True, blank, -1))
    dev = op.ctc_ext_beam_search_decoder_raw(xh.cuda(), torch.from_numpy(sl).cuda(), beam_width=W, top_paths=P,
                                             blank_index=blank)
    assert not L.raw_mismatches(dev, want)
    # a batch shard of the pinned tensor (pitched slab copies)
    part = op.ctc_ext_beam_search_decoder_raw(xh[:, 2:8, :], sl[2:8], beam_width=W, top_paths=P, blank_index=blank)
    assert not L.raw_mismatches(part, L.oracle_decode(np.ascontiguousarray(up[:, 2:8]), sl[2:8], W, P, False, blank, -1))
    # an out-of-range length is still reported as the reference reports it
    bad = sl.copy()
    bad[4] = T + 1
    with pytest.raises(op.CtcxError, match=r"sequence_length\(4\) <= %d" % T):
        op.ctc_ext_beam_search_decoder_raw(xh, bad, beam_width=W, top_paths=P, blank_index=blank)


@pytest.mark.parametrize("dt", ["float32", "float16", "bfloat16", "float64"])
def test_pinned_host_logits_are_fed_while_the_kernel_runs(op, dt):
    """ctcx_decode_hostin: page-locked host logits are copied in time slabs on a side stream while the
    beam kernel already consumes the frames that have landed (char-CTC shapes). The result must be
    the oracle's on the (exactly widened) values, for contiguous tensors and for a batch shard view."""
    import torch
    T, B, C, W, P = 300, 48, 29, 100, 1
    x32 = L.make_logits("gauss", T, B, C, 28, 51)
    xh = torch.from_numpy(x32).to(getattr(torch, dt)).pin_memory()
    up = xh.numpy() if dt == "float64" else xh.to(torch.float32).numpy()  # float64 is decoded in double
    sl = L.ragged_lengths(T, B, 51)
    want = L.oracle_decode_threaded(up, sl, W, P, True, 28, -1)
    for _ in range(3):  # repeated calls reuse the side stream and the staging memory
        raw = op.ctc_ext_beam_search_decoder_raw(xh, sl, beam_width=W, top_paths=P, merge_repeated=True,
                                                 blank_index=28)
        assert not raw[6].is_cuda  # host in -> host out
        assert not L.raw_mismatches(raw, want)
    # a shard view [:, b0:b1, :] of the pinned tensor: pitched copy, no repack
    b0, b1 = 7, 39
    part = op.ctc_ext_beam_search_decoder_raw(xh[:, b0:b1, :], sl[b0:b1], beam_width=W, top_paths=P,
                                              merge_repeated=True, blank_index=28)
    want_part = L.oracle_decode(np.ascontiguousarray(up[:, b0:b1]), sl[b0:b1], W, P, True, 28, -1)
    assert not L.raw_mismatches(part, want_part)
    # the same view on the device is decoded in place (time stride = whole batch)
    xd = xh.cuda()
    view = xd[:, b0:b1, :]
    assert not view.is_contiguous()
    partd = op.ctc_ext_beam_search_decoder_raw(view, torch.from_numpy(sl[b0:b1]).cuda(), beam_width=W, top_paths=P,
                                               merge_repeated=True, blank_index=28)
    assert partd[6].is_cuda and not L.raw_mismatches(partd, want_part)


def test_views_of_wide_and_float64_tensors(op):
    """Time-strided views through the wide kernel (C > 32) and the float64 path."""
    import torch
    T, B, C, W, P = 40, 9, 200, 8, 2
    x = L.make_logits("peaky", T, B, C, 0, 61)
    sl = L.ragged_lengths(T, B, 61)
    for arr in (x, x.astype(np.float64) + 1e-9):
        want = L.oracle_decode(np.ascontiguousarray(arr[:, 2:7]), sl[2:7], W, P, False, 0, -1)
        for inp in (torch.from_numpy(arr).cuda()[:, 2:7, :], arr[:, 2:7, :], torch.from_numpy(arr).pin_memory()[:, 2:7, :]):
            raw = op.ctc_ext_beam_search_decoder_raw(inp, sl[2:7], beam_width=W, top_paths=P, blank_index=0)
            assert not L.raw_mismatches(raw, want)
    # half precision through the wide kernel (read directly, no fp32 scratch)
    xh = torch.from_numpy(x).to(torch.bfloat16)
    want = L.oracle_decode(xh.float().numpy(), sl, W, P, False, 0, -1)
    raw = op.ctc_ext_beam_search_decoder_raw(xh.cuda(), sl, beam_width=W, top_paths=P, blank_index=0)
    assert not L.raw_mismatches(raw, want)
    # ... and through the generic path of a shape no fast kernel serves (beam_width > 256)
    T, B, C, W, P = 12, 2, 12, 300, 2
    xh = torch.from_numpy(L.make_logits("gauss", T, B, C, 0, 62)).to(torch.float16)
    want = L.oracle_decode(xh.float().numpy(), np.full(B, T, np.int32), W, P, False, 0, -1)
    raw = op.ctc_ext_beam_search_decoder_raw(xh.cuda(), np.full(B, T, np.int32), beam_width=W, top_paths=P, blank_index=0)
    assert not L.raw_mismatches(raw, want)


def test_flags_travel_with_the_result(op):
    x = L.make_logits("peaky", 30, 4, 29, 28, 3)
    sl = np.full(4, 30, np.int32)
    raw = op.ctc_ext_beam_search_decoder_raw(x, sl, beam_width=10, top_paths=2, blank_index=28)
    assert raw.flags == 0 and len(raw) == 7
    out = op.ctc_ext_beam_search_decoder(x, sl, beam_width=10, top_paths=2, blank_index=28)
    dec, ali, lp = out
    assert out.flags == 0 and len(out) == 3 and lp.shape == (4, 2)


def test_stream_top_paths_before_the_first_step(op):
    """TopPaths right after construction / Reset (decoder.h:212-261): the root alone -- log-prob 0 and
    empty sequences for one path, "Less leaves" for more."""
    import torch
    dec = op.CTCExtBeamSearchDecoderStream(batch_size=3, num_classes=29, beam_width=10, top_paths=1, max_time=40,
                                           blank_index=28)
    d, a, lp = dec.top_paths()
    assert lp.cpu().numpy().tolist() == [[0.0]] * 3 and d[0].values.numel() == 0 and a[0].values.numel() == 0
    assert d[0].dense_shape.tolist() == [3, 0]
    x = L.make_logits("peaky", 25, 3, 29, 28, 9)
    dec.step(x)
    want = L.oracle_decode(x, np.full(3, 25, np.int32), 10, 1, False, 28, -1)
    assert not L.raw_mismatches(dec.top_paths_raw(), want)
    dec.reset()  # ... and again after a decode
    d, a, lp = dec.top_paths()
    assert lp.cpu().numpy().tolist() == [[0.0]] * 3 and a[0].values.numel() == 0
    dec2 = op.CTCExtBeamSearchDecoderStream(batch_size=2, num_classes=29, beam_width=10, top_paths=3, max_time=40,
                                            blank_index=28)
    with pytest.raises(op.InvalidArgumentError, match="Less leaves"):
        dec2.top_paths()
    with pytest.raises(TypeError):
        dec2.step(np.zeros((4, 2, 29), np.float64))


def test_shard_errors_name_the_utterance_in_the_whole_batch(op):
    x = L.make_logits("gauss", 20, 6, 8, 7, 2)
    sl = np.full(6, 20, np.int32)
    sl[4] = 23
    with pytest.raises(op.FailedPreconditionError, match=r"sequence_length\(4\) <= 20"):
        op.decode_multi_device(x, sl, 4, 1, False, 7, -1, devices=[0, 0, 0])


def test_rescore_acceptance_cases_are_flagged(op):
    """The utterances of tests/golden/rescore_cases.npz make the reference accept the re-score of an
    evicted member (decoder.h:189-199) -- possible only at an exact tie with the beam bottom, see
    tests/test_oracle.py. The kernels do not model the event; they must REPORT it: the result's flags
    carry FLAG_ROUNDING_ANOMALY, so a caller can tell that this utterance left the bit-exact contract
    (it is a tie case, where the reference's own answer depends on heap order)."""
    import os
    arr = np.load(os.path.join(L.ROOT, "tests", "golden", "rescore_cases.npz"))
    n = int(arr["n"][0])
    flagged = same = 0
    for k in range(n):
        W, P, merge, blank = (int(v) for v in arr["c%d/attrs" % k])
        x = arr["c%d/x" % k][:, None, :]
        sl = np.asarray([x.shape[0]], np.int32)
        raw = op.ctc_ext_beam_search_decoder_raw(x, sl, beam_width=W, top_paths=P, merge_repeated=bool(merge),
                                                 blank_index=blank, blank_label=-1)
        flagged += int(bool(raw.flags & op.FLAG_ROUNDING_ANOMALY))
        same += int(not L.raw_mismatches(raw, L.oracle_decode(x, sl, W, P, bool(merge), blank, -1)))
    assert flagged == n, (flagged, n)   # every one of them is reported
    assert same >= 0                    # (most still decode like the oracle; not required)
    # ... and ordinary inputs never raise the flag
    x = L.make_logits("gauss", 120, 8, 29, 28, 77)
    raw = op.ctc_ext_beam_search_decoder_raw(x, np.full(8, 120, np.int32), beam_width=100, top_paths=1, blank_index=28)
    assert raw.flags == 0


def test_host_input_and_view_entries_reject_bad_arguments(op):
    """Error behaviour of the two round-2 C-ABI entries, straight through ctypes."""
    import ctypes
    import torch
    from ctc_beam_search_op_b200 import _lib
    lib = _lib.load()
    T, B, C, W, P = 12, 3, 8, 4, 2
    x = torch.from_numpy(L.make_logits("gauss", T, B, C, 7, 1)).pin_memory()
    sl = torch.tensor([12, 5, 3], dtype=torch.int32)
    ws_bytes = lib.ctcx_workspace_bytes(T, B, C, W, W + 1)  # (room for the top_paths > beam_width call below)
    ws = torch.empty(ws_bytes, dtype=torch.uint8, device="cuda")
    staging = torch.empty(lib.ctcx_hostin_staging_bytes(_lib.F32, T, B, C), dtype=torch.uint8, device="cuda")
    side = torch.cuda.Stream()
    main = torch.cuda.Stream()
    arr = ctypes.c_int64 * (W + 1)
    sizes = _lib.CtcxSizes(arr(), arr(), arr(), arr())
    flags = ctypes.c_int32(0)

    def hostin(**kw):
        a = dict(x=x.data_ptr(), dtype=_lib.F32, stride=0, T=T, B=B, C=C, sl=sl.data_ptr(), W=W, P=P, blank=7,
                 staging=staging.data_ptr(), st_bytes=staging.numel(), ws=ws.data_ptr(), ws_bytes=ws_bytes,
                 stream=main.cuda_stream, copy=side.cuda_stream)
        a.update(kw)
        return lib.ctcx_decode_hostin(a["x"], a["dtype"], a["stride"], a["T"], a["B"], a["C"], a["sl"], a["W"], a["P"], 0,
                                      a["blank"], -1, a["staging"], a["st_bytes"], a["ws"], a["ws_bytes"], a["stream"],
                                      a["copy"], ctypes.byref(sizes), ctypes.byref(flags))

    assert hostin() == 0 and sizes.n_alignment[0] == 20                      # 12 + 5 + 3 frames
    assert hostin(T=0) == 2                                                   # "max_time is 0"
    assert hostin(copy=main.cuda_stream) == 8                                 # the copy stream must differ
    assert hostin(st_bytes=16) == 8 and hostin(ws_bytes=256) == 10
    assert hostin(stride=B * C - 1) == 8 and hostin(dtype=9) == 8 and hostin(blank=C) == 8
    assert hostin(P=W + 1) == 6                                               # more paths than the beam width
    bad = torch.tensor([12, 13, 3], dtype=torch.int32)
    assert hostin(sl=bad.data_ptr()) == 5 and lib.ctcx_error_batch_index() == 1
    assert b"sequence_length(1) <= 12" in lib.ctcx_strerror(5)
    assert hostin(B=0) == 0 and sizes.n_alignment[0] == 0                     # empty batch
    torch.cuda.synchronize()
    xd = x.cuda()
    sd = sl.cuda()

    def view(dtype=_lib.F32, stride=0):
        return lib.ctcx_decode_view(xd.data_ptr(), dtype, stride, T, B, C, sd.data_ptr(), W, P, 0, 7, -1, ws.data_ptr(),
                                    ws_bytes, None, ctypes.byref(sizes), ctypes.byref(flags))

    assert view() == 0 and view(stride=B * C) == 0
    assert view(stride=B * C - 1) == 8 and view(stride=-5) == 8 and view(dtype=4) == 8
    # the Python host: empty batch and zero-length utterances through the host-input path
    raw = op.ctc_ext_beam_search_decoder_raw(np.zeros((5, 0, 4), np.float32), np.zeros((0,), np.int32), beam_width=4, top_paths=1)
    assert raw[0][0].shape == (0, 2) and raw[6].shape == (0, 1)
    sl0 = torch.tensor([12, 0, 3], dtype=torch.int32)  # a zero-length utterance: the root, one path only
    raw = op.ctc_ext_beam_search_decoder_raw(x, sl0, beam_width=W, top_paths=1, blank_index=7)
    assert not L.raw_mismatches(raw, L.oracle_decode(x.numpy(), sl0.numpy(), W, 1, False, 7, -1))
    with pytest.raises(op.InvalidArgumentError, match="Less leaves"):
        op.ctc_ext_beam_search_decoder_raw(x, sl0, beam_width=W, top_paths=2, blank_index=7)


def test_single_synchronisation_route_equals_the_two_phase_route(op):
    """Small results are decoded and packed back to back into a buffer sized from an upper bound, with
    one synchronisation (sizes == NULL, ctcx_pack_compact, ctcx_finish); large ones get their sizes
    first and exactly sized outputs. Both routes must return identical tensors, the same `.packed`
    layout and the same errors."""
    import torch
    from ctc_beam_search_op_b200 import decoder as D
    cases = [("gauss", 60, 7, 29, 100, 1, True, 28, np.float32), ("peaky", 40, 5, 32, 16, 3, False, 31, np.float32),
             ("peaky", 50, 4, 300, 16, 2, False, 299, np.float32), ("gauss", 30, 3, 12, 40, 2, True, 0, np.float64),
             ("gauss", 20, 3, 40, 300, 2, False, 7, np.float32)]
    saved = (D.DEFER_MAX_BYTES_DEVICE, D.DEFER_MAX_BYTES_HOST)
    try:
        for kind, T, B, C, W, P, merge, blank, dt in cases:
            x = L.make_logits(kind, T, B, C, blank, 71).astype(dt)
            sl = L.ragged_lengths(T, B, 71)
            kw = dict(beam_width=W, top_paths=P, merge_repeated=merge, blank_index=blank)
            got = {}
            for route, limit in (("deferred", 1 << 30), ("two-phase", 0)):
                D.DEFER_MAX_BYTES_DEVICE = D.DEFER_MAX_BYTES_HOST = limit
                got[route] = [op.ctc_ext_beam_search_decoder_raw(x, sl, **kw),                       # host in, host out
                              op.ctc_ext_beam_search_decoder_raw(torch.from_numpy(x).cuda(),         # device in / out
                                                                 torch.from_numpy(sl).cuda(), **kw),
                              op.ctc_ext_beam_search_decoder_raw(torch.from_numpy(x).pin_memory(), sl, **kw)]
            for a, b in zip(got["deferred"], got["two-phase"]):
                for g in range(6):
                    for p in range(P):
                        np.testing.assert_array_equal(np.asarray(torch.as_tensor(a[g][p]).cpu()), np.asarray(torch.as_tensor(b[g][p]).cpu()))
                np.testing.assert_array_equal(np.asarray(torch.as_tensor(a[6]).cpu()), np.asarray(torch.as_tensor(b[6]).cpu()))
                pa, pb = a.packed.cpu().numpy(), b.packed.cpu().numpy()
                assert pa.shape == pb.shape
                n_cmp = len(pa) - (1 if (dt == np.float32 and (B * P) % 2) else 0)  # (half of the last slot is padding)
                np.testing.assert_array_equal(pa[:n_cmp], pb[:n_cmp])
                assert a.flags == b.flags and a.max_lengths == b.max_lengths
            want = L.oracle_decode(x, sl, W, P, merge, blank, -1)
            assert not L.raw_mismatches(got["deferred"][0], want)
        # errors surface identically (at ctcx_finish on the deferred route)
        x = L.make_logits("gauss", 12, 3, 29, 28, 5)
        for limit in (1 << 30, 0):
            D.DEFER_MAX_BYTES_DEVICE = D.DEFER_MAX_BYTES_HOST = limit
            with pytest.raises(op.FailedPreconditionError, match=r"sequence_length\(1\) <= 12") as e:
                op.ctc_ext_beam_search_decoder_raw(x, [12, 13, 3], beam_width=8, top_paths=1, blank_index=28)
            assert e.value.batch_index == 1
            with pytest.raises(op.InvalidArgumentError, match="Less leaves"):
                op.ctc_ext_beam_search_decoder_raw(x, [12, 0, 3], beam_width=8, top_paths=2, blank_index=28)
            with pytest.raises(op.InvalidArgumentError, match="requested more paths"):
                op.ctc_ext_beam_search_decoder_raw(x, [12, 5, 3], beam_width=2, top_paths=3, blank_index=28)
            with pytest.raises(op.InvalidArgumentError):
                op.ctc_ext_beam_search_decoder_raw(x, [12, -1, 3], beam_width=8, top_paths=1, blank_index=28)
            empty = op.ctc_ext_beam_search_decoder_raw(np.zeros((4, 0, 5), np.float32), np.zeros((0,), np.int32),
                                                       beam_width=3, top_paths=1, blank_index=4)
            assert tuple(np.asarray(empty[2][0])) == (0, 0)
    finally:
        D.DEFER_MAX_BYTES_DEVICE, D.DEFER_MAX_BYTES_HOST = saved


def test_pending_decodes_in_flight(op):
    """wait=False: several decodes enqueued before any result is read (device and pinned-host inputs,
    different shapes), resolved out of order; each equals its blocking twin, errors are raised by
    .result() -- every time it is called."""
    import torch
    jobs = []
    for k, (T, B, C, W, P, blank) in enumerate([(80, 6, 29, 100, 1, 28), (50, 4, 300, 16, 2, 299), (60, 5, 32, 20, 3, 31),
                                               (80, 6, 29, 100, 1, 28)]):
        x = L.make_logits("gauss" if k % 2 else "peaky", T, B, C, blank, 80 + k)
        sl = L.ragged_lengths(T, B, 80 + k)
        kw = dict(beam_width=W, top_paths=P, merge_repeated=bool(k % 2), blank_index=blank)
        xin = torch.from_numpy(x).pin_memory() if k % 2 else torch.from_numpy(x).cuda()
        sin = sl if k % 2 else torch.from_numpy(sl).cuda()
        jobs.append((x, sl, kw, op.ctc_ext_beam_search_decoder_raw(xin, sin, wait=False, **kw)))
    bad = op.ctc_ext_beam_search_decoder_raw(torch.from_numpy(jobs[0][0]).cuda(), [81, 3, 3, 3, 3, 3], beam_width=4,
                                             top_paths=1, blank_index=28, wait=False)
    assert all(isinstance(j[3], op.PendingDecode) for j in jobs)
    for x, sl, kw, pending in reversed(jobs):
        got = pending.result()
        assert pending.result() is got
        want = L.oracle_decode(x, sl, kw["beam_width"], kw["top_paths"], kw["merge_repeated"], kw["blank_index"], -1)
        assert not L.raw_mismatches(got, want)
    for _ in range(2):
        with pytest.raises(op.FailedPreconditionError, match=r"sequence_length\(0\) <= 80"):
            bad.result()
