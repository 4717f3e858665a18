"""Every beam-kernel variant the dispatcher can choose, against the oracle and against exact CTC.

* Exact regime: with a beam at least as wide as the number of labelings that can have non-zero
  probability nothing is pruned, and the result is fixed by the definition of CTC alone
  (tests/ctcx_exact.py, float64): the returned labelings are the most probable ones, log_probability
  is log p(l|x) (+ S(l) with a scorer table) and the alignment scores the Viterbi value. Each case
  also equals the oracle bit for bit where the oracle is cheap.
* Dispatch matrix: one case per kernel variant (element type, beam tier, CTAs per SM, time-sliced
  queue, host feed, route, trace kernel and record size), compared with the oracle bit for bit. The
  preconditions of each variant are asserted from the device properties, not assumed.
* Value edges at length: half-precision logits at the BASELINE shapes, sharp and offset logits, very
  long utterances.

Every returned path in this file is also checked against the bounds that hold with pruning:
log_probability <= log p(l|x) + tol and alignment score <= log_probability + tol, with the float32
tolerance of ctcx_exact.float32_tolerance (4 ulps of |total| + max |logit| per frame), and the
alignment must collapse to the decoded labels.
"""
import zlib

import numpy as np
import pytest

import ctcx_exact as X
import ctcx_testlib as L

pytestmark = pytest.mark.gpu

_oracle_cache = {}
MAX_DISTINCT = 64  # large batches: distinct utterances, replicated


@pytest.fixture(scope="module", params=["fast", "generic"])
def op(request):
    """The default dispatch (fast kernels where they apply) and the generic kernel forced through the
    test hook, as in tests/test_gpu_parity.py."""
    import torch
    if not torch.cuda.is_available():
        pytest.skip("no CUDA device")
    import ctc_beam_search_op_b200 as m
    m.set_beam_impl(request.param)
    yield m
    m.set_beam_impl(None)


@pytest.fixture(scope="module")
def dev():
    """SM count and the most 256-thread CTAs an SM can hold: what the dispatch thresholds depend on."""
    import torch
    if not torch.cuda.is_available():
        pytest.skip("no CUDA device")
    p = torch.cuda.get_device_properties(torch.cuda.current_device())
    sms = int(p.multi_processor_count)
    return {"sms": sms, "minb4": 2 * sms + 1, "sliced": sms * (int(p.max_threads_per_multi_processor) // 256) + 1}


# ------------------------------------------------------------------------------------------------
# helpers
def _np(a):
    return a.detach().cpu().numpy() if hasattr(a, "detach") else np.asarray(a)


def _dense(raw, B, P):
    """Raw sparse outputs -> per (utterance, path) lists of decoded labels and alignments + log-probs."""
    out = []
    for g in (0, 3):
        per = []
        for p in range(P):
            idx, val = _np(raw[g][p]), _np(raw[g + 1][p])
            cnt = np.bincount(idx[:, 0], minlength=B) if len(idx) else np.zeros(B, np.int64)
            per.append(np.split(val, np.cumsum(cnt)[:-1]))
        out.append(per)
    return out[0], out[1], _np(raw[6]).astype(np.float64)


def _paths(d, b, P):
    dec, ali, lp = d
    return [(dec[p][b].tolist(), ali[p][b].tolist(), lp[b, p]) for p in range(P)]


def _check_paths(raw, x, sl, P, merge, blank, utts=None, exact=False, table=None):
    """Exact-CTC checks (exact=True) or the pruning bounds on every returned path of the utterances."""
    B = x.shape[1]
    d = _dense(raw, B, P)
    utts = list(range(B) if utts is None else utts)
    lps = {b: X.log_softmax(np.asarray(x[:sl[b], b], np.float64)) for b in utts}
    if exact:
        labs = {b: X.enumerate_labelings(lps[b], blank) for b in utts}
    else:  # the forward and Viterbi scores of the returned labelings, all at once
        keys = [(b, X.collapse(d[1][p][b].tolist(), -1)) for b in utts for p in range(P)]
        scores = X.ctc_scores_many([lps[b] for b, _ in keys], [l for _, l in keys], blank)
        labs = {b: {} for b in utts}
        for (b, l), v in zip(keys, scores):
            labs[b][l] = v
    for b in utts:
        bad = X.check_paths(_paths(d, b, P), lps[b], blank, -1, merge, exact=exact, table=table,
                            logits=np.asarray(x[:sl[b], b]), labelings=labs[b])
        assert not bad, "utterance %d: %s" % (b, bad[:4])


def _oracle(key, x, sl, W, P, merge, blank, lm=None):
    """Oracle result over the host threads, cached across the two kernel families."""
    if key is None or key not in _oracle_cache:
        res = L.oracle_decode_threaded(x, sl, W, P, merge, blank, -1, lm=lm)
        if key is None:
            return res
        _oracle_cache[key] = res
    return _oracle_cache[key]


def _decode(op, x, sl, W, P, merge, blank, **kw):
    return op.ctc_ext_beam_search_decoder_raw(x, sl, beam_width=W, top_paths=P, merge_repeated=merge,
                                              blank_index=blank, blank_label=-1, **kw)


def _assert_oracle(raw, want, what=""):
    bad = L.raw_mismatches(raw, want)
    assert not bad, "%s: %d utterances differ from the oracle, first %s" % (what, len(bad), bad[:8])


def _replicated(n, B, seed):
    """Sources of a batch of B utterances made of n distinct ones: the n first, then random copies."""
    rng = np.random.default_rng(seed)
    src = np.concatenate([np.arange(n), rng.integers(0, n, B - n)]) if B > n else np.arange(B)
    return src


def _check_replicated(raw, src, sl_full, P, want_distinct):
    """Every copy equals its original bit for bit; the originals equal the oracle."""
    n = want_distinct.B
    d = _dense(raw, len(src), P)
    dec, ali, lp = d
    for p in range(P):  # (float32 and float64 values are exact in float64: compare those bits)
        np.testing.assert_array_equal(lp[:, p].view(np.uint64), lp[src, p].view(np.uint64))
        for b in range(len(src)):
            o = src[b]
            assert np.array_equal(ali[p][b], ali[p][o]) and np.array_equal(dec[p][b], dec[p][o]), (b, o)
    for b in range(n):
        for p in range(P):
            assert dec[p][b].tolist() == want_distinct.decoded(b, p), (b, p)
            assert ali[p][b].tolist() == want_distinct.alignment(b, p), (b, p)
            assert np.float64(lp[b, p]).view(np.uint64) == np.float64(want_distinct.logp[b, p]).view(np.uint64), (b, p)


# ------------------------------------------------------------------------------------------------
# Exact regime on every kernel family
EXACT = [
    # T, C, W, P, merge, blank, dtype      (3 utterances, lengths T, T, T - 1)
    (4, 3, 31, 6, False, 0, "float32"),      # narrow, 32-slot tier
    (4, 3, 15, 9, True, 2, "float32"),       # W = the labeling count: the beam just fills
    (6, 3, 127, 8, False, 1, "float32"),     # 128-slot tier
    (6, 3, 41, 20, True, 0, "float32"),      # (beam just fills; top_paths above 7)
    (7, 3, 255, 5, False, 2, "float32"),     # 256-slot tier
    (7, 3, 67, 4, True, 1, "float32"),
    (6, 3, 127, 6, False, 1, "float16"),     # half inputs: exact CTC of the upcast values
    (7, 3, 255, 6, True, 0, "bfloat16"),
    (6, 3, 127, 4, False, 2, "float64"),     # narrow kernel computing in double
    (2, 29, 813, 6, False, 28, "float32"),   # generic (W > 256)
    (2, 29, 813, 4, True, 0, "float16"),
    (8, 3, 511, 5, False, 1, "float64"),     # generic in double
    (127, 2, 128, 3, True, 1, "float32"),    # one label: chains of ~T LogSumExps per labeling
    (255, 2, 256, 3, False, 0, "float32"),   # narrow, the widest tier
    (1023, 2, 1024, 3, True, 1, "float32"),  # generic, the widest beam; TraceWarpKernel with rows_log2 = 1
]


def _cast(x32, dt):
    """(values handed to the decoder, their exact float64 upcast)."""
    import torch
    if dt == "float64":
        x = x32.astype(np.float64)
        return x, x
    if dt == "float32":
        return x32, x32.astype(np.float64)
    xh = torch.from_numpy(x32).to(getattr(torch, dt))
    return xh, xh.to(torch.float64).numpy()


@pytest.mark.parametrize("case", EXACT, ids=lambda c: "T%d-C%d-W%d-P%d-%s" % (c[0], c[1], c[2], c[3], c[6]))
def test_exact_regime(op, case):
    T, C, W, P, merge, blank, dt = case
    rng = np.random.default_rng(T * 7 + C + W)
    x32 = (rng.standard_normal((T, 3, C)) * 1.5).astype(np.float32)
    xin, up = _cast(x32, dt)
    sl = np.array([T, T, T - 1], np.int32)
    assert X.max_labelings(up, sl, blank) <= W  # nothing can be pruned
    raw = _decode(op, xin, sl, W, P, merge, blank)
    _check_paths(raw, up, sl, P, merge, blank, exact=True)
    if T * W * C <= 3e6:  # the oracle is cheap: bit for bit
        want = L.oracle_decode(up if dt == "float64" else up.astype(np.float32), sl, W, P, merge, blank, -1)
        _assert_oracle(raw, want)


@pytest.mark.parametrize("merge", [False, True])
def test_exact_regime_with_a_scorer_table(op, merge):
    """log_probability = log p(l|x) + S(l): narrow scorer variant (128-slot tier) and generic."""
    rng = np.random.default_rng(5)
    for T, C, W, P, blank in ((6, 3, 127, 6, 0), (5, 4, 200, 5, 2), (2, 29, 813, 5, 28)):
        x = (rng.standard_normal((T, 3, C)) * 1.5).astype(np.float32)
        table = (-np.abs(rng.standard_normal((C + 1, C))) * 1.5).astype(np.float32)
        sl = np.array([T, T, T - 1], np.int32)
        assert X.max_labelings(x, sl, blank) <= W
        raw = _decode(op, x, sl, W, P, merge, blank, expansion_scores=table)
        _check_paths(raw, x, sl, P, merge, blank, exact=True, table=table)
        _assert_oracle(raw, L.oracle_decode(x, sl, W, P, merge, blank, -1, lm=table))


MASKED = [
    # T, C, blank, dtype: 2-3 finite non-blank classes per frame at high label ids
    (4, 300, 0, "float32"),     # wide kernel
    (4, 300, 299, "float16"),   # wide kernel, half inputs
    (3, 4096, 4095, "float32"),  # C > 2048: generic
    (3, 4096, 17, "bfloat16"),
    (5, 8192, 8191, "float32"),
    (5, 32000, 0, "float32"),
    (5, 65535, 65534, "float32"),  # the largest vocabulary the API accepts
]


@pytest.mark.parametrize("case", MASKED, ids=lambda c: "T%d-C%d-%s" % (c[0], c[1], c[3]))
def test_exact_regime_masked_vocabulary(op, case):
    """-inf masking leaves a few labelings in a wide vocabulary: exact CTC at W = their count (the beam
    just fills) and at W = 1024. A shape the kernels cannot hold must say so (UnsupportedError)."""
    T, C, blank, dt = case
    rng = np.random.default_rng(C + T)
    x32 = X.masked_logits(T, 3, C, blank, rng)
    xin, up = _cast(x32, dt)
    sl = np.array([T, T, T - 1], np.int32)
    n = X.max_labelings(up, sl, blank)
    for W in sorted({n, 1024}):
        try:
            raw = _decode(op, xin, sl, W, 4, False, blank)
        except op.UnsupportedError:
            assert C > 2048, "(W=%d, C=%d) must be supported" % (W, C)
            continue
        _check_paths(raw, up, sl, 4, False, blank, exact=True)
        if W * C * T <= 2e6:
            _assert_oracle(raw, L.oracle_decode(up.astype(np.float32), sl, W, 4, False, blank, -1))


def test_streaming_exact_after_every_chunk(op):
    """TopPaths after each chunk = exact CTC of the frames each utterance consumed so far; utterance 1
    takes no frame in some chunks and frames again later."""
    T, B, C, W, P, blank = 7, 3, 3, 127, 3, 2
    rng = np.random.default_rng(8)
    chunks = [(rng.standard_normal((2, B, C)) * 1.5).astype(np.float32) for _ in range(5)]
    lens = [np.array([2, 0, 1]), np.array([1, 2, 2]), np.array([2, 0, 1]), np.array([0, 2, 2]), np.array([2, 1, 0])]
    dec = op.CTCExtBeamSearchDecoderStream(batch_size=B, num_classes=C, beam_width=W, top_paths=P, max_time=T,
                                           blank_index=blank)
    frames = [[] for _ in range(B)]
    for ch, ln in zip(chunks, lens):
        dec.step(ch, ln.astype(np.int32))
        for b in range(B):
            frames[b].extend(ch[:ln[b], b])
        done = np.array([len(f) for f in frames], np.int32)
        x = np.zeros((max(done.max(), 1), B, C), np.float32)
        for b in range(B):
            if done[b]:
                x[:done[b], b] = np.stack(frames[b])
        if X.labeling_count(int(done.min()), C - 1) < P:
            continue  # fewer leaves than paths
        raw = dec.top_paths_raw()
        _check_paths(raw, x, done, P, False, blank, exact=True)
        _assert_oracle(raw, L.oracle_decode(x, done, W, P, False, blank, -1))


# ------------------------------------------------------------------------------------------------
# Dispatch matrix: one case per variant, bit for bit against the oracle
def _lengths_over_slices(B, T):
    """Every length 0..T (so every slice boundary, whatever the slice size), then full ones."""
    return (np.arange(B) % (T + 1)).astype(np.int32)


MATRIX = [
    # name, T, C, W, P, dtype, B (or "minb4" / "sliced"), lengths ("full" / "ragged" / "slices"), kind
    ("narrow-f32-minb4-t32", 80, 29, 20, 2, "float32", "minb4", "ragged", "gauss"),
    ("narrow-f32-minb4-t256-sliced", 96, 18, 200, 1, "float32", "sliced", "slices", "peaky"),
    ("narrow-f16-minb4-t32-sliced", 96, 29, 16, 1, "float16", "sliced", "slices", "gauss"),
    ("narrow-bf16-minb4-t128-sliced", 80, 29, 100, 1, "bfloat16", "sliced", "slices", "peaky"),
    ("narrow-f16-minb4-t256-sliced", 70, 12, 256, 1, "float16", "sliced", "slices", "gauss"),
    ("narrow-bf16-minb2-t256", 60, 20, 200, 3, "bfloat16", 40, "ragged", "gauss"),
    ("narrow-f16-minb4-t128", 60, 29, 64, 2, "float16", "minb4", "ragged", "peaky"),
    ("narrow-f64-bigbatch-t128", 60, 29, 100, 2, "float64", "minb4", "ragged", "peaky"),
    ("narrow-f64-bigbatch-t256", 40, 12, 200, 1, "float64", "minb4", "ragged", "gauss"),
    ("narrow-f32-topk12", 50, 29, 16, 12, "float32", 6, "full", "gauss"),
    ("narrow-f32-topk40", 40, 16, 64, 40, "float32", 4, "full", "peaky"),
    ("wide-f16-t32", 60, 300, 16, 2, "float16", 8, "ragged", "peaky"),
    ("wide-bf16-t128", 40, 700, 40, 2, "bfloat16", 4, "ragged", "gauss"),
    ("wide-f16-t256", 25, 40, 200, 2, "float16", 4, "ragged", "gauss"),
    ("generic-wide-too-big-smem", 30, 500, 200, 2, "float32", 3, "ragged", "peaky"),
    ("generic-wide-too-big-smem-f16", 20, 2048, 120, 2, "float16", 2, "ragged", "gauss"),
    ("generic-c4096-w16", 30, 4096, 16, 2, "float32", 3, "ragged", "peaky"),
    ("generic-c8192-w8", 10, 8192, 8, 1, "float32", 2, "full", "peaky"),
    ("generic-w1024-trace-warp", 40, 5, 1024, 3, "float32", 2, "ragged", "gauss"),
    ("trace-thread-rec8", 30, 300, 8, 4, "float32", 1024, "ragged", "peaky"),
    ("trace-thread-rec4", 40, 29, 10, 8, "float32", 512, "ragged", "gauss"),
]


def _batch(spec, dev):
    return dev[spec] if isinstance(spec, str) else spec


@pytest.mark.parametrize("case", MATRIX, ids=lambda c: c[0])
def test_dispatch_matrix(op, dev, case):
    import torch
    name, T, C, W, P, dt, bspec, lspec, kind = case
    B = _batch(bspec, dev)
    blank = C - 1 if C <= 32 else 3
    # preconditions of the variant, from the device properties
    if bspec == "minb4":
        assert B > 2 * dev["sms"]
    if bspec == "sliced":
        assert B > 2 * dev["sms"] and B >= dev["sliced"] and T >= 64
    if name.startswith("generic-wide-too-big"):  # the candidate list alone is over the wide kernel's 200 KB
        assert C <= 2048 and W <= 256 and 8 * W * min(C - 1, 2 * W + 2) > 200 * 1024
    if name.startswith("trace-thread"):
        assert B * P >= 4096
    if name == "trace-thread-rec8":
        assert C > 256  # 8-byte back-pointer records
    seed = zlib.crc32(name.encode()) % 10007
    if lspec == "slices":
        # lengths b % (T + 1): every length 0..T, so every slice boundary whatever the slice size; the
        # T + 1 distinct utterances each come with their own length
        n = T + 1
        sl_n = np.arange(n, dtype=np.int32)
        src = np.arange(B) % n
    else:
        n = min(B, MAX_DISTINCT)
        sl_n = L.ragged_lengths(T, n, seed) if lspec == "ragged" else np.full(n, T, np.int32)
        src = _replicated(n, B, seed)
    x32 = L.make_logits(kind, T, n, C, blank, seed)
    xin, up = _cast(x32, dt)
    up32 = up if dt == "float64" else up.astype(np.float32)
    xd = (xin if isinstance(xin, torch.Tensor) else torch.from_numpy(xin)).cuda()
    xb = xd.index_select(1, torch.from_numpy(src).cuda()).contiguous()
    raw = _decode(op, xb, torch.from_numpy(sl_n[src]).cuda(), W, P, True, blank)
    want = _oracle((name,), np.ascontiguousarray(up32), sl_n, W, P, True, blank)
    _check_replicated(raw, src, sl_n[src], P, want)
    _check_paths(raw, up[:, src], sl_n[src], P, True, blank, utts=range(n))
    assert raw.flags == 0


@pytest.mark.parametrize("tier", [(128, 64, 29), (256, 150, 20)], ids=lambda t: "t%d" % t[0])
def test_scorer_variant_with_four_ctas_per_sm(op, dev, tier):
    """The narrow kernel's scorer-table variant in the throughput regime (B > 2 x SMs)."""
    import torch
    _, W, C = tier
    T, P, blank = 50, 2, C - 1
    B = dev["minb4"]
    assert B > 2 * dev["sms"]
    n = MAX_DISTINCT
    x = L.make_logits("gauss", T, n, C, blank, W)
    sl_n = L.ragged_lengths(T, n, W)
    table = (-np.abs(np.random.default_rng(W).standard_normal((C + 1, C))) * 1.5).astype(np.float32)
    src = _replicated(n, B, W)
    want = _oracle(("scorer", W), x, sl_n, W, P, False, blank, lm=table)
    raw = _decode(op, np.ascontiguousarray(x[:, src]), sl_n[src], W, P, False, blank, expansion_scores=table)
    _check_replicated(raw, src, sl_n[src], P, want)
    _check_paths(raw, x, sl_n, P, False, blank, table=table)


@pytest.mark.parametrize("dt", ["float32", "bfloat16"])
def test_pinned_host_feed_with_the_time_sliced_queue(op, dev, dt):
    """Page-locked host logits (the kernel polls the "frames landed" word) in a batch large enough for
    the time-sliced queue, lengths over every slice boundary, P = 1 (length 0 occurs)."""
    import torch
    T, C, W, P, blank = 96, 29, 32, 1, 28
    B = dev["sliced"]
    assert B > 2 * dev["sms"] and T >= 64
    n = T + 1  # distinct utterance b % n has length b % (T + 1) = its own index
    x32 = L.make_logits("peaky", T, n, C, blank, 91)
    src = np.arange(B) % n
    sl = _lengths_over_slices(B, T)
    xh = torch.from_numpy(np.ascontiguousarray(x32[:, src])).to(getattr(torch, dt)).pin_memory()
    up = xh[:, :n].to(torch.float32).numpy()
    want = _oracle(("pinned", dt), up, sl[:n], W, P, False, blank)
    full = L.DenseResult.__new__(L.DenseResult)  # the whole batch's expected result: copies of the distinct ones
    full.B, full.P, full.T = B, P, T
    full.dec_len, full.ali_len = want.dec_len[src], want.ali_len[src]
    full.dec, full.ali, full.logp = want.dec[src], want.ali[src], want.logp[src]
    for _ in range(2):
        raw = _decode(op, xh, sl, W, P, False, blank)
        assert not raw[6].is_cuda
        _assert_oracle(raw, full, "pinned %s" % dt)
    _check_paths(raw, xh.to(torch.float64).numpy(), sl, P, False, blank, utts=range(n))


def test_large_vocabularies_are_decoded_or_refused(op):
    """C > 2048 on the default dispatch, beam widths up to 1024: each (W, C) either equals exact CTC (and
    the oracle where it is cheap) or raises UnsupportedError -- never a CUDA error."""
    rng = np.random.default_rng(12)
    T, B, P = 4, 2, 2
    decoded = refused = 0
    for C in (2049, 4096, 8192, 32000, 65535):
        blank = C - 1 if C % 2 else 1
        x = X.masked_logits(T, B, C, blank, rng)
        sl = np.full(B, T, np.int32)
        n = X.max_labelings(x, sl, blank)
        for W in (1, 8, 64, 256, 1024):
            try:
                raw = _decode(op, x, sl, W, min(P, W), False, blank)
            except op.UnsupportedError:
                # the generic kernel keeps a logit row and a [beam, classes] bitmap in shared memory
                assert not ((C <= 8192 and W <= 64) or (C <= 4096 and W <= 256)), (C, W)
                refused += 1
                continue
            decoded += 1
            _check_paths(raw, x, sl, min(P, W), False, blank, exact=W >= n)
            if W * C * T <= 4e7:
                _assert_oracle(raw, L.oracle_decode(x, sl, W, min(P, W), False, blank, -1), "C=%d W=%d" % (C, W))
    assert decoded >= 11, (decoded, refused)


def test_streaming_large_batch_with_idle_chunks(op, dev):
    """Streaming with more utterances than 2 x SMs; some utterances take no frame in a chunk and frames
    again in a later one (the step docstring allows it)."""
    T, C, W, P, blank = 48, 29, 16, 1, 28
    B = dev["minb4"] + 7
    rng = np.random.default_rng(21)
    dec = op.CTCExtBeamSearchDecoderStream(batch_size=B, num_classes=C, beam_width=W, top_paths=P, max_time=T,
                                           merge_repeated=True, blank_index=blank)
    n = MAX_DISTINCT
    base = L.make_logits("peaky", T, n, C, blank, 22)
    frames = np.zeros((T, B, C), np.float32)
    used = np.zeros(B, np.int32)
    while used.min() < T - 8:
        ct = int(rng.integers(1, 9))
        ln = np.where(rng.random(B) < 0.3, 0, rng.integers(1, ct + 1, B)).astype(np.int32)
        ln = np.minimum(ln, T - used)
        chunk = np.zeros((ct, B, C), np.float32)
        for b in range(B):
            chunk[:ln[b], b] = base[used[b]:used[b] + ln[b], b % n]
            frames[used[b]:used[b] + ln[b], b] = chunk[:ln[b], b]
        dec.step(chunk, ln)
        used += ln
    raw = dec.top_paths_raw()
    # utterance b consumed the first used[b] frames of distinct b % n
    pairs = sorted(set(zip((np.arange(B) % n).tolist(), used.tolist())))
    xs = np.ascontiguousarray(base[:, [s for s, _ in pairs]])
    ls = np.array([l for _, l in pairs], np.int32)
    want = L.oracle_decode_threaded(xs, ls, W, P, True, blank)
    ix = {pr: i for i, pr in enumerate(pairs)}
    d = _dense(raw, B, P)
    for b in range(B):
        i = ix[(b % n, int(used[b]))]
        assert d[1][0][b].tolist() == want.alignment(i, 0) and d[0][0][b].tolist() == want.decoded(i, 0), b
        assert np.float32(d[2][b, 0]).view(np.uint32) == np.float32(want.logp[i, 0]).view(np.uint32), b
    _check_paths(raw, frames, used, P, True, blank, utts=range(n))


# ------------------------------------------------------------------------------------------------
# Value edges at length
HALF_FULL = [
    # name, T, B, C, W, P, merge, blank, utterances decoded
    ("cfg2", 500, 256, 29, 100, 1, True, 28, 256),
    ("cfg3", 1500, 64, 32, 64, 4, False, 31, 64),
    ("cfg4", 400, 128, 1024, 16, 1, False, 1023, 32),
]


@pytest.mark.parametrize("dt", ["bfloat16", "float16"])
@pytest.mark.parametrize("cfg", HALF_FULL, ids=lambda c: c[0])
def test_half_precision_at_the_baseline_shapes(op, cfg, dt):
    """Quantised logits tie exactly far more often: every utterance against the oracle on the upcast values."""
    import torch
    name, T, B, C, W, P, merge, blank, nb = cfg
    seed = {"cfg2": 61, "cfg3": 62, "cfg4": 63}[name]
    x32 = np.concatenate([L.make_logits("gauss", T, nb // 2, C, blank, seed),
                          L.make_logits("peaky", T, nb - nb // 2, C, blank, seed + 1)], axis=1)
    sl = L.ragged_lengths(T, nb, seed)
    sl[0] = T
    xh = torch.from_numpy(x32).to(getattr(torch, dt))
    up = xh.to(torch.float32).numpy()
    want = _oracle((name, dt), up, sl, W, P, merge, blank)
    raw = _decode(op, xh.cuda(), torch.from_numpy(sl).cuda(), W, P, merge, blank)
    _assert_oracle(raw, want, "%s %s" % (name, dt))
    _check_paths(raw, up, sl, P, merge, blank)


def test_bf16_beyond_the_resident_ctas(op, dev):
    import torch
    T, C, W, P, blank = 200, 29, 100, 1, 28
    B = dev["sliced"]
    x32 = L.make_logits("gauss", T, MAX_DISTINCT, C, blank, 71)
    sl_n = L.ragged_lengths(T, MAX_DISTINCT, 71)
    src = _replicated(MAX_DISTINCT, B, 71)
    xh = torch.from_numpy(x32).to(torch.bfloat16).cuda()
    up = xh.float().cpu().numpy()
    want = _oracle(("bf16-large",), up, sl_n, W, P, True, blank)
    raw = _decode(op, xh.index_select(1, torch.from_numpy(src).cuda()).contiguous(),
                  torch.from_numpy(sl_n[src]).cuda(), W, P, True, blank)
    _check_replicated(raw, src, sl_n[src], P, want)


SHARP = [("x20", 20.0, 0.0), ("x100", 100.0, 0.0), ("plus1e4", 1.0, 1e4)]


@pytest.mark.parametrize("edge", SHARP, ids=lambda e: e[0])
def test_sharp_and_offset_logits_at_cfg2_size(op, edge):
    """Scaled or offset logits drive the narrow kernel's range prediction (1.25 gap - 64) and its second,
    full-range pass; an offset of 1e4 leaves ~1e-3 of float32 resolution in every logit."""
    name, scale, shift = edge
    T, B, C, W, P, merge, blank = 500, 64, 29, 100, 1, True, 28
    x = L.make_logits("gauss", T, B, C, blank, 81)
    x = (x.astype(np.float64) * scale + shift).astype(np.float32)
    sl = L.ragged_lengths(T, B, 81)
    want = _oracle(("sharp", name), x, sl, W, P, merge, blank)
    raw = _decode(op, x, sl, W, P, merge, blank)
    _assert_oracle(raw, want, name)
    _check_paths(raw, x, sl, P, merge, blank)


def test_very_long_utterances(op):
    """T = 8000: totals near -1e4, where float32 spacing is ~1e-3 and exact ties are everywhere."""
    T, B, C, W, P, merge, blank = 8000, 16, 29, 100, 2, True, 28
    x = np.concatenate([L.make_logits("gauss", T, B // 2, C, blank, 83),
                        L.make_logits("peaky", T, B // 2, C, blank, 84)], axis=1)
    sl = np.full(B, T, np.int32)
    sl[1::2] = L.ragged_lengths(T, B // 2, 83)
    want = _oracle(("long",), x, sl, W, P, merge, blank)
    raw = _decode(op, x, sl, W, P, merge, blank)
    _assert_oracle(raw, want, "T=8000")
    _check_paths(raw, x, sl, P, merge, blank)


def test_long_utterances_beyond_the_resident_ctas(op, dev):
    """T = 4000 with more utterances than resident CTAs: the queue cuts every utterance into up to 16
    time slices."""
    import torch
    T, C, W, P, merge, blank = 4000, 29, 100, 1, True, 28
    B = dev["sliced"]
    n = 16
    x32 = L.make_logits("peaky", T, n, C, blank, 85)
    sl_n = np.full(n, T, np.int32)
    sl_n[1::2] = L.ragged_lengths(T, n // 2, 85)
    src = _replicated(n, B, 85)
    want = _oracle(("long-large",), x32, sl_n, W, P, merge, blank)
    xd = torch.from_numpy(x32).cuda()
    raw = _decode(op, xd.index_select(1, torch.from_numpy(src).cuda()).contiguous(),
                  torch.from_numpy(sl_n[src]).cuda(), W, P, merge, blank)
    _check_replicated(raw, src, sl_n[src], P, want)
    _check_paths(raw, x32[:, src], sl_n[src], P, merge, blank, utts=range(n))
