"""The table-driven beam kernels (a scorer table through `expansion_scores=`, ctcx_decode_scorer_f32 and the
float32 stream) on the tables users actually write: -inf entries as label constraints, entries far below
the logits, subnormal and -0.0 entries, quantised entries that tie. Every decode is compared with the
oracle bit for bit, and with exact CTC (tests/ctcx_exact.py) where nothing can be pruned.

* Constrained exact regime: with -inf entries forming a DAG over the labels the number of allowed
  labelings is finite whatever T is, so at a beam at least that wide nothing is pruned even at T = 500:
  the returned labelings are the best by log p(l|x) + S(l), each with its exact score. W = the count
  (the beam just fills) and W = the tier's maximum (it never fills, so nothing is evicted and no flag may
  be set); the narrow scorer variant at every tier (32/128/256 slots) in the latency and throughput
  regimes and the time-sliced queue; the generic kernel forced on the same cases, and at C = 40 and 300,
  where it is the only route for a table.
* Extreme entries: -1e3 / -1e4 entries put children far below the narrow kernel's range bound of a beam
  that is not full; subnormal entries in row 0 are the child's whole base at the root; an all -0.0 table
  is the default scorer; quantised entries tie children exactly; row 0 all -inf leaves only the root;
  rows with no successor.
* Errors on every kernel family: more paths than allowed labelings is "Less leaves"; a NaN entry is
  refused by the one-shot decode, ctcx_decode_scorer_f32 itself, the stream constructor and the stream's
  TopPaths; -inf is accepted at each of them.
* The revisit-wipe fixed point with a table: the cases of tests/golden/wipe_table_cases.npz (as deep as
  the zero-table cases, with cases that expose a fixed point that counts wiped rows or stops after 4
  rounds) on the narrow variant at two and four CTAs per SM, the time-sliced queue, the generic kernel's
  list and sweep forms, streaming cut at the deepest frames and page-locked host logits; the tier-128
  timing build's at-risk, wiped and frames-with-at-risk counts equal the model's.
* Shapes that only the generic kernel takes with a table run once, under the forced generic setting.
* Streaming: exact CTC after every chunk with a DAG table and idle utterances; reset / TopPaths of
  single slots with a constraint table.
"""
import ctypes
import zlib

import numpy as np
import pytest

import ctcx_exact as X
import ctcx_testlib as L

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module", params=["fast", "generic"])
def op(request):
    """The default dispatch (the narrow scorer variant where C <= 32) and the generic kernel forced."""
    import torch
    if not torch.cuda.is_available():
        pytest.skip("no CUDA device")
    import ctc_beam_search_op_b200 as m
    m.set_beam_impl(request.param)
    yield m
    m.set_beam_impl(None)


@pytest.fixture(scope="module")
def dev():
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
    out = []
    for g in (0, 3):
        per = []
        for p in range(P):
            idx, val = _np(raw[g][p]), _np(raw[g + 1][p])
            cnt = np.bincount(idx[:, 0], minlength=B) if len(idx) else np.zeros(B, np.int64)
            per.append(np.split(val, np.cumsum(cnt)[:-1]))
        out.append(per)
    return out[0], out[1], _np(raw[6]).astype(np.float64)


def _check_paths(raw, x, sl, P, merge, blank, table, utts, exact, labelings=None):
    """Exact CTC with the table's constraints (exact=True) or the pruning bounds, utterance by utterance.
    labelings: {utterance: enumerate_labelings(...)} already computed, or None."""
    d = _dense(raw, x.shape[1], P)
    for b in utts:
        lp = X.log_softmax(np.asarray(x[:sl[b], b], np.float64))
        labs = None
        if exact:
            labs = labelings[b] if labelings is not None else X.enumerate_labelings(lp, blank, table=table)
        paths = [(d[0][p][b].tolist(), d[1][p][b].tolist(), d[2][b, p]) for p in range(P)]
        bad = X.check_paths(paths, lp, blank, -1, merge, exact=exact, table=table, logits=x[:sl[b], b],
                            labelings=labs)
        assert not bad, "utterance %d: %s" % (b, bad[:4])


def _decode(op, x, sl, W, P, merge, blank, table):
    return op.ctc_ext_beam_search_decoder_raw(x, sl, beam_width=W, top_paths=P, merge_repeated=merge,
                                              blank_index=blank, blank_label=-1, expansion_scores=table)


def _assert_oracle(raw, want, what=""):
    bad = L.raw_mismatches(raw, want)
    assert not bad, "%s: %d utterances differ from the oracle, first %s" % (what, len(bad), bad[:8])


def _rows(r, src):
    """DenseResult r with its utterances picked by src (a replicated batch's expected result)."""
    t = L.DenseResult.__new__(L.DenseResult)
    t.B, t.P, t.T = len(src), r.P, r.T
    t.dec_len, t.ali_len, t.dec, t.ali, t.logp = r.dec_len[src], r.ali_len[src], r.dec[src], r.ali[src], r.logp[src]
    return t


def _batch(spec, n, T, dev, seed):
    """(B, src, lengths of the distinct utterances): n distinct utterances replicated to the batch size of
    the regime; "sliced" gives the T + 1 distinct lengths 0..T so that every slice boundary is met."""
    if spec == "sliced":
        B = dev["sliced"]
        assert B > 2 * dev["sms"] and T >= 64
        return B, np.arange(B) % (T + 1), np.arange(T + 1, dtype=np.int32)
    B = dev["minb4"] if spec == "minb4" else n
    assert spec != "minb4" or B > 2 * dev["sms"]
    rng = np.random.default_rng(seed)
    src = np.concatenate([np.arange(n), rng.integers(0, n, B - n)]) if B > n else np.arange(B)
    sl = np.full(n, T, np.int32)
    sl[1::2] = rng.integers(T // 2, T + 1, len(sl[1::2]))
    return B, src, sl


# ------------------------------------------------------------------------------------------------
# Constrained exact regime
CONSTRAINED = [
    # name, T, C, blank, most allowed labelings, self-transition, merge, batch ("latency" / "minb4" / "sliced")
    ("c12-t32", 50, 12, 0, 30, False, False, "latency"),
    ("c12-t32-loop", 60, 12, 5, 31, True, True, "minb4"),
    ("c29-t128", 200, 29, 28, 120, False, True, "minb4"),
    ("c29-t128-sliced", 96, 29, 28, 127, False, False, "sliced"),
    ("c18-t256", 120, 18, 17, 250, False, False, "latency"),  # (W x C <= 4608: the narrow kernel's list)
    ("c16-t256-sliced", 80, 16, 0, 255, False, True, "sliced"),
    ("c32-t32-long", 500, 32, 31, 32, False, True, "latency"),
    ("c18-t256-long", 500, 18, 0, 200, False, False, "minb4"),
    ("c32-t256-generic", 120, 32, 31, 250, False, False, "latency"),  # (W x C past the list: generic)
    ("c29-t128-loop", 80, 29, 0, 127, True, False, "latency"),
    ("c40-generic", 100, 40, 3, 200, False, False, "latency"),
    ("c300-generic", 60, 300, 3, 180, False, True, "minb4"),
]


def _tier(W):
    return 32 if W <= 32 else (128 if W <= 128 else 256)


def _impl(request):
    return request.node.callspec.params["op"]


def _once(request, C, W=0):
    """A shape that only the generic kernel takes with a table (C > 32, W > 256 or W x C past the narrow
    candidate list) decodes the same way under both settings of the test hook: run it under one."""
    if _impl(request) == "fast" and (C > 32 or W > 256 or W * C > 4608):
        pytest.skip("the generic kernel on either setting: run under the forced one")


@pytest.mark.parametrize("case", CONSTRAINED, ids=lambda c: c[0])
def test_constrained_exact_regime(op, dev, request, case):
    import torch
    name, T, C, blank, most, loop, merge, spec = case
    _once(request, C, most)
    seed = zlib.crc32(name.encode()) % 10007
    table, n = X.dag_table(C, blank, seed, most, T=T if loop else None, self_loop=loop)
    B, src, sl_n = _batch(spec, 8, T, dev, seed)
    nd = len(sl_n)
    x = (np.random.default_rng(seed).standard_normal((T, nd, C)) * 1.5).astype(np.float32)
    # exact CTC on the distinct utterances (on a few of the T + 1 lengths of the sliced batch: 0, 1, 2, a
    # middle one and T), the oracle on all; batch index b < nd is distinct utterance b
    check = [0, 1, 2, nd // 2, nd - 1] if spec == "sliced" else list(range(nd))
    labs = {b: X.enumerate_labelings(X.log_softmax(x[:sl_n[b], b]), blank, table=table) for b in check}
    assert max(len(v) for v in labs.values()) == n  # (an utterance of full length is among them)
    P_most = 1 if spec == "sliced" else min(len(v) for v in labs.values())  # (length 0: the root alone)
    xb = torch.from_numpy(np.ascontiguousarray(x[:, src])).cuda()
    slb = torch.from_numpy(sl_n[src]).cuda()
    full = _tier(n) if C <= 32 else (1024 if C <= 64 else 256)
    for W, P in ((n, min(P_most, 24)), (full, min(P_most, 40))):
        raw = _decode(op, xb, slb, W, P, merge, blank, table)
        _assert_oracle(raw, _rows(L.oracle_decode_threaded(x, sl_n, W, P, merge, blank, lm=table), src),
                       "%s W=%d" % (name, W))
        _check_paths(raw, x[:, src], sl_n[src], P, merge, blank, table, check, exact=True, labelings=labs)
        assert raw.flags == 0, (W, raw.flags)  # nothing is ever evicted: no anomaly can be reported


@pytest.mark.parametrize("C,blank", [(12, 0), (32, 31), (40, 3)])
def test_every_allowed_labeling_and_one_more(op, request, C, blank):
    """P = the allowed count returns every allowed labeling once (exactly scored); P = count + 1 is the
    reference's "Less leaves" error, as the oracle says."""
    _once(request, C)
    T = 64
    table, n = X.dag_table(C, blank, C, 24)
    x = (np.random.default_rng(C).standard_normal((T, 2, C)) * 1.5).astype(np.float32)
    sl = np.array([T, T], np.int32)
    raw = _decode(op, x, sl, n, n, False, blank, table)
    _assert_oracle(raw, L.oracle_decode(x, sl, n, n, False, blank, -1, lm=table))
    _check_paths(raw, x, sl, n, False, blank, table, [0, 1], exact=True)
    with pytest.raises(L.OracleError, match="Less leaves"):
        L.oracle_decode(x, sl, n + 1, n + 1, False, blank, -1, lm=table)
    with pytest.raises(op.InvalidArgumentError, match="Less leaves"):
        _decode(op, x, sl, n + 1, n + 1, False, blank, table)


# ------------------------------------------------------------------------------------------------
# Extreme entries
def _far_table(C, blank, rng, far, frac):
    t = (-np.abs(rng.standard_normal((C + 1, C))) * 1.5).astype(np.float32)
    return np.where(rng.random((C + 1, C)) < frac, rng.choice(far, (C + 1, C)), t).astype(np.float32)


FAR = [
    # T, C, W, P, merge: the beam of W = 16 at C = 32 overflows in the first frame (bin 0 decides), W = 200
    # stays below full for many frames
    (60, 32, 16, 3, False), (100, 29, 100, 2, True), (80, 32, 200, 4, False), (60, 12, 256, 6, True),
    (50, 40, 64, 2, False),
]


@pytest.mark.parametrize("far", [(-1e3,), (-1e4,), (-1e3, -1e4)], ids=["1e3", "1e4", "mixed"])
@pytest.mark.parametrize("case", FAR, ids=lambda c: "T%d-C%d-W%d" % c[:3])
def test_far_negative_entries(op, request, case, far):
    """Children far below the lowest base + lowest log-prob of a beam that is not full, and in a full one."""
    _once(request, case[1], case[2])
    T, C, W, P, merge = case
    rng = np.random.default_rng(T + C + W + int(-far[0]))
    blank = C - 1
    table = _far_table(C, blank, rng, far, 0.4)
    x = L.make_logits("gauss", T, 4, C, blank, W)
    sl = L.ragged_lengths(T, 4, W)
    raw = _decode(op, x, sl, W, P, merge, blank, table)
    _assert_oracle(raw, L.oracle_decode(x, sl, W, P, merge, blank, -1, lm=table))
    _check_paths(raw, x, sl, P, merge, blank, table, range(4), exact=False)


@pytest.mark.parametrize("C,W", [(12, 20), (32, 100), (29, 200), (40, 64)])
def test_far_negative_constraint_dag_never_fills(op, request, C, W):
    """A DAG table whose allowed entries are all around -1e3 .. -1e4: exact CTC, beam never full."""
    _once(request, C, W)
    T, blank = 80, 1
    table, n = X.dag_table(C, blank, C + W, min(W - 1, 120))
    rng = np.random.default_rng(C)
    table = np.where(np.isfinite(table), -(1e3 + rng.random(table.shape) * 9e3), -np.inf).astype(np.float32)
    x = (rng.standard_normal((T, 3, C)) * 1.5).astype(np.float32)
    sl = np.array([T, T - 3, T // 2], np.int32)
    P = min(n, 5)
    raw = _decode(op, x, sl, W, P, True, blank, table)
    _assert_oracle(raw, L.oracle_decode(x, sl, W, P, True, blank, -1, lm=table))
    _check_paths(raw, x, sl, P, True, blank, table, range(3), exact=True)
    assert raw.flags == 0


@pytest.mark.parametrize("C,W", [(12, 16), (29, 100), (32, 256), (40, 16)])
def test_subnormal_entries_in_row_zero(op, request, C, W):
    """Row 0 entries are subnormal: at the root (total 0) the child's base IS the entry. With logits that
    leave one finite class in frame 0 (log-prob exactly 0) and only the blank afterwards, the best path's
    log_probability is the entry itself, which flushing subnormals to zero would turn into -0.0."""
    _once(request, C, W)
    blank = C - 1
    T, B = 3, C - 1
    rng = np.random.default_rng(C)
    table = (-np.abs(rng.standard_normal((C + 1, C)))).astype(np.float32)
    sub = -(np.arange(1, C + 1, dtype=np.float64) * 1.7e-41)  # (1.4e-45 is the smallest subnormal)
    table[0] = sub.astype(np.float32)
    table[0, 0] = -np.float32(1.4e-45)
    assert all(0 < abs(v) < np.finfo(np.float32).tiny for v in table[0])
    x = np.full((T, B, C), -np.inf, np.float32)
    for b in range(B):
        x[0, b, b] = 0.0  # utterance b: class b in frame 0, then blank
        x[1:, b, blank] = 0.0
    sl = np.array([1 + b % T for b in range(B)], np.int32)
    raw = _decode(op, x, sl, W, 1, False, blank, table)
    _assert_oracle(raw, L.oracle_decode(x, sl, W, 1, False, blank, -1, lm=table))
    np.testing.assert_array_equal(_np(raw[6])[:, 0].view(np.uint32), table[0, :B].view(np.uint32))
    # and mixed into ordinary logits
    x = L.make_logits("gauss", 40, 4, C, blank, C)
    sl = np.full(4, 40, np.int32)
    raw = _decode(op, x, sl, W, 2, False, blank, table)
    _assert_oracle(raw, L.oracle_decode(x, sl, W, 2, False, blank, -1, lm=table))


@pytest.mark.parametrize("C,W", [(29, 16), (29, 100), (32, 256), (40, 64)])
def test_negative_zero_table_is_the_default_scorer(op, request, C, W):
    """Adding -0.0 changes no score: the table decode equals the decode without a table bit for bit."""
    _once(request, C, W)
    T, blank = 120, C - 1
    x = L.make_logits("peaky", T, 6, C, blank, W)
    sl = L.ragged_lengths(T, 6, W)
    table = np.full((C + 1, C), -0.0, np.float32)
    want = L.oracle_decode(x, sl, W, 3, True, blank, -1)
    _assert_oracle(_decode(op, x, sl, W, 3, True, blank, table), want, "-0.0 table")
    _assert_oracle(_decode(op, x, sl, W, 3, True, blank, None), want, "no table")


@pytest.mark.parametrize("C,W", [(12, 8), (29, 32), (29, 128), (32, 256), (40, 100)])
def test_quantised_entries_tie_children(op, request, C, W):
    """Logits k/8 and entries k/4: child scores are short dyadic sums, so they tie exactly and often."""
    _once(request, C, W)
    T, blank = 100, 0
    rng = np.random.default_rng(C * W)
    x = (np.round(rng.standard_normal((T, 4, C)) * 8) / 8).astype(np.float32)
    table = (-np.floor(rng.random((C + 1, C)) * 8) / 4).astype(np.float32)
    sl = np.array([T, T, T - 9, T // 3], np.int32)
    P = min(W, 4)
    raw = _decode(op, x, sl, W, P, False, blank, table)
    _assert_oracle(raw, L.oracle_decode(x, sl, W, P, False, blank, -1, lm=table))
    _check_paths(raw, x, sl, P, False, blank, table, range(4), exact=False)


@pytest.mark.parametrize("C,W", [(12, 16), (29, 100), (32, 200), (40, 64)])
def test_row_zero_all_minus_inf_keeps_only_the_root(op, request, C, W):
    """No label may start: the beam holds the root alone for all T frames, and its path is all blanks with
    the sum of the blank log-probabilities; a second path is "Less leaves"."""
    _once(request, C, W)
    T, blank = 90, 2
    rng = np.random.default_rng(C + W)
    table = (-np.abs(rng.standard_normal((C + 1, C)))).astype(np.float32)
    table[0] = -np.inf
    x = L.make_logits("gauss", T, 3, C, blank, C)
    sl = np.array([T, 1, T // 2], np.int32)
    raw = _decode(op, x, sl, W, 1, False, blank, table)
    _assert_oracle(raw, L.oracle_decode(x, sl, W, 1, False, blank, -1, lm=table))
    d = _dense(raw, 3, 1)
    for b in range(3):
        assert d[0][0][b].tolist() == [] and d[1][0][b].tolist() == [-1] * int(sl[b])
    _check_paths(raw, x, sl, 1, False, blank, table, range(3), exact=True)
    assert raw.flags == 0
    with pytest.raises(op.InvalidArgumentError, match="Less leaves"):
        _decode(op, x, sl, W, 2, False, blank, table)


@pytest.mark.parametrize("C,W", [(12, 32), (29, 128), (32, 256), (40, 100)])
def test_rows_with_no_successor(op, request, C, W):
    """Half of the labels end every labeling (their rows are all -inf); the others are unconstrained."""
    _once(request, C, W)
    T, blank = 80, C - 1
    rng = np.random.default_rng(3 * C + W)
    table = (-np.abs(rng.standard_normal((C + 1, C))) * 1.5).astype(np.float32)
    dead = rng.choice(C, C // 2, replace=False)
    table[dead + 1] = -np.inf
    x = L.make_logits("peaky", T, 4, C, blank, W)
    sl = L.ragged_lengths(T, 4, W)
    raw = _decode(op, x, sl, W, 3, True, blank, table)
    _assert_oracle(raw, L.oracle_decode(x, sl, W, 3, True, blank, -1, lm=table))
    _check_paths(raw, x, sl, 3, True, blank, table, range(4), exact=False)


# ------------------------------------------------------------------------------------------------
# Errors
def _scorer_direct(op, x, sl, W, P, blank, table):
    """ctcx_decode_scorer_f32 called as a C caller would: its return code."""
    import torch
    from ctc_beam_search_op_b200 import _lib
    lib = _lib.load()
    T, B, C = x.shape
    xd = torch.from_numpy(x).cuda()
    sd = torch.from_numpy(sl).cuda()
    td = torch.from_numpy(table).cuda()
    nbytes = lib.ctcx_workspace_bytes(T, B, C, W, P)
    ws = torch.empty(max(nbytes, 256), dtype=torch.uint8, device="cuda")
    arr = ctypes.c_int64 * P
    sizes = _lib.CtcxSizes(arr(), arr(), arr(), arr())
    flags = ctypes.c_int32(0)
    rc = lib.ctcx_decode_scorer_f32(xd.data_ptr(), T, B, C, sd.data_ptr(), W, P, 0, blank, -1, td.data_ptr(),
                                    ws.data_ptr(), nbytes, torch.cuda.current_stream().cuda_stream,
                                    ctypes.byref(sizes), ctypes.byref(flags))
    torch.cuda.synchronize()
    return rc


@pytest.mark.parametrize("C,W", [(12, 16), (29, 100), (32, 256), (40, 64)])
def test_nan_refused_and_minus_inf_accepted_everywhere(op, request, C, W):
    _once(request, C, W)
    import torch
    T, blank, P = 20, 0, 1
    x = L.make_logits("gauss", T, 2, C, blank, C)
    sl = np.full(2, T, np.int32)
    ok = (-np.abs(np.random.default_rng(C).standard_normal((C + 1, C)))).astype(np.float32)
    ok[1::3, ::2] = -np.inf
    bad = ok.copy()
    bad[C // 2, C - 1] = np.nan
    want = L.oracle_decode(x, sl, W, P, False, blank, -1, lm=ok)
    # one-shot decode (the C-ABI's device check), and ctcx_decode_scorer_f32 itself
    with pytest.raises(op.InvalidArgumentError):
        _decode(op, x, sl, W, P, False, blank, bad)
    _assert_oracle(_decode(op, x, sl, W, P, False, blank, ok), want, "-inf table")
    assert _scorer_direct(op, x, sl, W, P, blank, bad) == 8
    assert _scorer_direct(op, x, sl, W, P, blank, ok) == 0
    # stream: the constructor's check ...
    kw = dict(batch_size=2, num_classes=C, beam_width=W, top_paths=P, max_time=T, blank_index=blank)
    with pytest.raises(op.InvalidArgumentError):
        op.CTCExtBeamSearchDecoderStream(expansion_scores=bad, **kw)
    dec = op.CTCExtBeamSearchDecoderStream(expansion_scores=ok, **kw)
    dec.step(x)
    _assert_oracle(dec.top_paths_raw(), want, "stream -inf table")
    # ... and TopPaths after a step with a NaN entry (the stream-wide device check of ctcx_stream_step_v)
    dec.reset()
    dec._esd.copy_(torch.from_numpy(bad).cuda())
    dec.step(x)
    with pytest.raises(op.InvalidArgumentError):
        dec.top_paths_raw()


# ------------------------------------------------------------------------------------------------
# The revisit-wipe fixed point with a table: tests/golden/wipe_table_cases.npz (tests/test_wipe_table_cases.py
# checks the cases on the CPU: depths per tier at or above the zero-table fixture's, verdicts that flip
# back, wiped parents, and cases that decode differently under a fixed point that counts the candidates
# of wiped rows or stops after 4 rounds)
DEEP = L.wipe_table_cases()
_want = {}


def _want_deep(c, B=1):
    if c.name not in _want:
        _want[c.name] = L.oracle_decode(c.x, c.sl, c.W, c.P, c.merge, c.blank, -1, lm=c.lm)
    return _rows(_want[c.name], np.zeros(B, np.int64))


def _decode_deep(op, c, x, sl, lm=None):
    return _decode(op, x, sl, c.W, c.P, c.merge, c.blank, c.lm if lm is None else lm)


@pytest.mark.parametrize("c", DEEP, ids=lambda c: c.name)
def test_deep_fixed_points_on_every_route(op, dev, request, c):
    """Two CTAs per SM (one utterance), four (replicated past 2 x SMs), more utterances than resident CTAs
    (at T = 128 the time-sliced queue, its boundaries at deep frames), page-locked host logits. The
    generic range (W > 256) has one route whatever the test hook says: it runs under the forced generic
    kernel only."""
    import torch
    if c.W > 256 and _impl(request) == "fast":
        pytest.skip("W > 256 takes the generic kernel on either setting")
    tab = torch.from_numpy(c.lm).cuda()
    for B in (1, dev["minb4"], dev["sliced"]):
        x = torch.from_numpy(np.ascontiguousarray(np.repeat(c.x, B, axis=1))).cuda()
        sl = torch.full((B,), c.T, dtype=torch.int32).cuda()
        _assert_oracle(_decode_deep(op, c, x, sl, tab), _want_deep(c, B), "%s B=%d" % (c.name, B))
    xh = torch.from_numpy(c.x).pin_memory()
    _assert_oracle(_decode_deep(op, c, xh, torch.from_numpy(c.sl)), _want_deep(c), "%s host" % c.name)


def _padded(c, C2):
    """c with classes C .. C2 - 1 added at -inf in the logits and the table: the same decode, a wider row."""
    x = np.full((c.T, 1, C2), -np.inf, np.float32)
    x[:, :, :c.C] = c.x
    lm = np.full((C2 + 1, C2), -np.inf, np.float32)
    lm[:c.C + 1, :c.C] = c.lm
    return x, lm


def test_deep_fixed_points_generic_list_and_sweep(op, request):
    """The generic kernel's candidate list holds W x C entries up to 4608; beyond that it sweeps every
    (row, class) pair in each query: every case as it is, and padded with -inf classes past 4608."""
    if _impl(request) != "generic":
        pytest.skip("the forced generic kernel's run covers it")
    for c in DEEP:
        assert c.W * c.C <= 4608
        _assert_oracle(_decode_deep(op, c, c.x, c.sl), _want_deep(c), "%s list" % c.name)
        x, lm = _padded(c, 4608 // c.W + 1)
        _assert_oracle(_decode(op, x, c.sl, c.W, c.P, c.merge, c.blank, lm), _want_deep(c), "%s sweep" % c.name)


@pytest.mark.parametrize("dt", ["float32", "bfloat16"])
def test_deep_fixed_points_streamed_with_cuts_at_the_deepest_frame(op, dt):
    """Chunk boundaries right before and after the deepest frame. A stream with a table steps float32
    logits: a bfloat16 chunk is widened by step() before the kernel reads it (the narrow scorer variant
    reads float32 only), so this checks that path, with values (k/16, |k| <= 128) exact in bfloat16."""
    import torch
    for c in DEEP:
        t = int(np.argmax(c.iters))
        cuts = sorted({0, t, t + 1, c.T} | ({32, 64} if c.T >= 64 else set()))
        dec = op.CTCExtBeamSearchDecoderStream(batch_size=1, num_classes=c.C, beam_width=c.W, top_paths=c.P,
                                               max_time=c.T, merge_repeated=c.merge, blank_index=c.blank,
                                               expansion_scores=c.lm)
        x = torch.from_numpy(c.x).to(getattr(torch, dt)).cuda()
        for a, b in zip(cuts[:-1], cuts[1:]):
            dec.step(x[a:b], np.array([b - a], np.int32))
        _assert_oracle(dec.top_paths_raw(), _want_deep(c), "%s stream %s cuts %s" % (c.name, dt, cuts))


def test_timing_build_counts_equal_the_model_with_a_table(op, request):
    """The tier-128 timing build of the scorer variant lists every member whose parent holds an earlier
    slot: its at-risk (slot 20), wiped (22) and frames-with-at-risk (23) counts equal the model's, on every
    case of the 128-slot tier (W 33 .. 128)."""
    import torch
    from ctc_beam_search_op_b200 import _lib
    if _impl(request) != "fast":
        pytest.skip("the narrow kernel's timing build")
    lib = _lib.load()
    cs = [c for c in DEEP if 32 < c.W <= 128]
    assert len(cs) >= 4
    for c in cs:
        buf = torch.zeros((1, 24), dtype=torch.int64, device="cuda")
        lib.ctcx_debug_set_cycles_buffer(buf.data_ptr())
        try:
            raw = _decode_deep(op, c, c.x, c.sl)
            torch.cuda.synchronize()
        finally:
            lib.ctcx_debug_set_cycles_buffer(None)
        _assert_oracle(raw, _want_deep(c), "%s timing build" % c.name)
        cyc = buf[0].cpu().numpy()
        st = c.stats
        assert (cyc[20], cyc[22], cyc[23]) == (st["at_risk"], st["wiped"], st["frames_at_risk"]), (c.name, cyc[20:24], st)


# ------------------------------------------------------------------------------------------------
# Streaming
def test_streaming_exact_after_every_chunk_with_a_dag_table(op):
    """TopPaths after each chunk = exact constrained CTC of the frames consumed so far; utterances take no
    frame in some chunks and frames again later."""
    T, B, C, blank, P = 64, 4, 12, 0, 3
    table, n = X.dag_table(C, blank, 77, 30)
    W = 32
    rng = np.random.default_rng(78)
    dec = op.CTCExtBeamSearchDecoderStream(batch_size=B, num_classes=C, beam_width=W, top_paths=P, max_time=T,
                                           blank_index=blank, expansion_scores=table)
    frames = [[] for _ in range(B)]
    while min(len(f) for f in frames) < T - 8:
        ct = int(rng.integers(1, 9))
        ln = np.where(rng.random(B) < 0.3, 0, rng.integers(1, ct + 1, B))
        ln = np.minimum(ln, [T - len(f) for f in frames]).astype(np.int32)
        ch = (rng.standard_normal((ct, B, C)) * 1.5).astype(np.float32)
        dec.step(ch, ln)
        for b in range(B):
            frames[b].extend(ch[:ln[b], b])
        done = np.array([len(f) for f in frames], np.int32)
        x = np.zeros((max(done.max(), 1), B, C), np.float32)
        for b in range(B):
            if done[b]:
                x[:done[b], b] = np.stack(frames[b])
        if min(len(X.enumerate_labelings(X.log_softmax(x[:done[b], b]), blank, table=table)) for b in range(B)) < P:
            continue  # fewer leaves than paths
        raw = dec.top_paths_raw()
        _assert_oracle(raw, L.oracle_decode(x, done, W, P, False, blank, -1, lm=table), "stream")
        _check_paths(raw, x, done, P, False, blank, table, range(B), exact=True)
        assert raw.flags == 0


def test_stream_slots_with_a_constraint_table(op):
    """reset(slots) / top_paths_raw(slots) with a DAG table: the reset slots decode their new frames alone."""
    T, B, C, blank, P, W = 40, 4, 29, 28, 2, 128
    table, n = X.dag_table(C, blank, 91, 100)
    rng = np.random.default_rng(92)
    a = (rng.standard_normal((T, B, C)) * 1.5).astype(np.float32)
    b = (rng.standard_normal((T, B, C)) * 1.5).astype(np.float32)
    dec = op.CTCExtBeamSearchDecoderStream(batch_size=B, num_classes=C, beam_width=W, top_paths=P, max_time=2 * T,
                                           merge_repeated=True, blank_index=blank, expansion_scores=table)
    dec.step(a)
    dec.reset([1, 3])
    dec.step(b)
    # slots 1 and 3 consumed b only; slots 0 and 2 consumed a then b
    ab = np.concatenate([a, b], axis=0)
    raw = dec.top_paths_raw([1, 3])
    _assert_oracle(raw, L.oracle_decode(np.ascontiguousarray(b[:, [1, 3]]), np.full(2, T, np.int32), W, P, True,
                                        blank, -1, lm=table), "slots 1, 3")
    _check_paths(raw, b[:, [1, 3]], np.full(2, T, np.int32), P, True, blank, table, range(2), exact=True)
    raw = dec.top_paths_raw([0, 2])
    _assert_oracle(raw, L.oracle_decode(np.ascontiguousarray(ab[:, [0, 2]]), np.full(2, 2 * T, np.int32), W, P, True,
                                        blank, -1, lm=table), "slots 0, 2")
