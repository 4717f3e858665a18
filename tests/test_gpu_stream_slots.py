"""Per-slot lifecycle of the streaming decoder: `reset(slots)` and `top_paths(slots)` let each of the B
utterance positions of a stream start and finish on its own. Every utterance that passes through a slot
must decode exactly as in one one-shot decode of all of them (labels, alignments and the bits of
log_probability), whatever its neighbours do."""
import ctypes

import numpy as np
import pytest

import ctcx_testlib as L
from test_gpu_stream_dtypes import _bigram, _inputs, _npy, _sms, assert_same

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module", params=["fast", "generic"])
def op(request):
    """Both beam-kernel families: the default dispatch and the generic kernel forced by the test hook."""
    import torch
    if not torch.cuda.is_available():
        pytest.skip("no CUDA device")
    import ctc_beam_search_op_b200 as m
    m.set_beam_impl(request.param)
    yield m
    m.set_beam_impl(None)


def host(raw):
    """A raw result with every tensor on the host (numpy), the six sparse groups and log_probability."""
    return [[_npy(t) for t in g] for g in raw[:6]] + [_npy(raw[6])]


def rows(raw, i, P):
    """Row i of a raw result (see host()): per path (decoded labels, alignment), and the log_probability
    bits. The sparse rows must be row-major."""
    out = []
    for p in range(P):
        for g in (0, 3):
            idx, val = raw[g][p], raw[g + 1][p]
            assert idx.shape[0] == 0 or (np.diff(idx[:, 0]) >= 0).all()
            a, b = np.searchsorted(idx[:, 0], i, "left"), np.searchsorted(idx[:, 0], i, "right")
            assert (idx[a:b, 1] == np.arange(b - a)).all()
            out.append(val[a:b].tolist())
    lp = raw[6][i]
    out.append(lp.view(np.uint64 if lp.dtype == np.float64 else np.uint32).tolist())
    return out


def check_selected(res, want, utts, P):
    """res: a per-slot read whose row i holds utterance utts[i] of the one-shot result `want`."""
    res, want = host(res), host(want)
    n = len(utts)
    assert res[6].shape == (n, P)
    for p in range(P):
        for g in (0, 3):
            lens = np.bincount(res[g][p][:, 0], minlength=n)
            assert len(lens) == n
            assert res[g + 2][p].tolist() == [n, int(lens.max())]
    for i, u in enumerate(utts):
        assert rows(res, i, P) == rows(want, u, P), "utterance %d (row %d)" % (u, i)


def continuous_batching(op, dt, T, B, C, W, P, blank, table=None, seed=5, pool=3):
    """pool * B ragged utterances through B slots in random per-slot chunks (0- and 1-frame chunks
    included); finished slots are read in random groups, blocking or wait=False (read while the next
    chunks are stepped), then reset with a random kind of selection and refilled."""
    import torch
    N = pool * B
    xd, xo = _inputs(dt, T, N, C, blank, seed)
    sl = L.ragged_lengths(T, N, seed)
    one = op.ctc_ext_beam_search_decoder_raw(xd, torch.from_numpy(sl).cuda(), beam_width=W, top_paths=P,
                                             blank_index=blank, expansion_scores=table)
    bad = L.raw_mismatches(one, L.oracle_decode(xo, sl, W, P, False, blank, -1, lm=table))
    assert not bad, "one-shot decode differs from the oracle at %s" % bad[:8]
    rng = np.random.default_rng(seed + 1)
    dec = op.CTCExtBeamSearchDecoderStream(batch_size=B, num_classes=C, beam_width=W, top_paths=P, max_time=T,
                                           blank_index=blank, dtype=torch.float64 if dt == "float64" else torch.float32,
                                           expansion_scores=table)
    queue = list(range(N))
    utt = np.array([queue.pop(0) for _ in range(B)])
    pos = np.zeros(B, np.int64)
    reads, done = [], 0
    while done < N:
        ct = min(int(rng.choice([1, 1, 2, 5, 9, 17])), T)
        active = utt >= 0
        lens = np.where(active, np.minimum(rng.integers(0, ct + 1, B), sl[np.maximum(utt, 0)] - pos), 0)
        t = torch.from_numpy(np.minimum(pos[None, :] + np.arange(ct)[:, None], T - 1)).cuda()
        u = torch.from_numpy(np.maximum(utt, 0)[None, :].repeat(ct, 0)).cuda()
        dec.step(xd[t, u], lens.astype(np.int32))
        pos += lens
        finished = np.flatnonzero(active & (pos == sl[np.maximum(utt, 0)]))
        if len(finished) == 0 or rng.random() < 0.3:
            continue
        group = np.sort(rng.choice(finished, int(rng.integers(1, len(finished) + 1)), replace=False))
        kind = int(rng.integers(0, 3))
        sel = ([int(b) for b in group] if kind == 0 else np.isin(np.arange(B), group) if kind == 1
               else torch.from_numpy(np.isin(np.arange(B), group).astype(np.int32)).cuda())
        wait = bool(rng.random() < 0.5)
        res = dec.top_paths_raw(sel, wait=wait)
        reads.append((res, utt[group].copy(), group))
        dec.reset(sel)
        done += len(group)
        for b in group:
            utt[b] = queue.pop(0) if queue else -1
            pos[b] = 0
    seen = []
    for res, utts, group in reads:
        r = res if not hasattr(res, "result") else res.result()
        assert r.slots.tolist() == group.tolist()
        check_selected(r, one, utts, P)
        seen += utts.tolist()
    assert sorted(seen) == list(range(N))


POOL_CASES = [("float32", 30, 6, 29, 20, 2, 28, False), ("bfloat16", 30, 6, 29, 20, 2, 28, False),
              ("float64", 30, 5, 29, 20, 2, 28, False), ("float32", 30, 6, 29, 20, 1, 28, True),
              ("float32", 24, 5, 40, 24, 2, 7, False), ("bfloat16", 16, 3, 1024, 16, 1, 1023, False),
              ("float32", 16, 3, 12, 300, 2, 0, False)]


@pytest.mark.parametrize("case", POOL_CASES,
                         ids=lambda c: "%s-C%d-W%d%s" % (c[0], c[3], c[4], "-table" if c[7] else ""))
def test_continuous_batching_equals_the_one_shot_decode(op, case):
    dt, T, B, C, W, P, blank, table = case
    continuous_batching(op, dt, T, B, C, W, P, blank, table=_bigram(C, 3) if table else None)


def test_continuous_batching_beyond_the_resident_ctas(op):
    continuous_batching(op, "float32", 12, 2 * _sms() + 9, 29, 16, 1, 28, seed=8, pool=2)


def _feed(dec, xd, chunks):
    for a, b, lens in chunks:
        dec.step(xd[a:b], lens)


# (T, B, C, W, P): a batch whose trace-back takes the warp-per-walk kernel, and one with B * P >= 4096
# walks, which takes the thread-per-walk kernel
@pytest.mark.parametrize("shape", [(40, 7, 29, 20, 2), (16, 2048, 29, 8, 2)], ids=["B7", "B2048"])
def test_selected_rows_match_the_full_read_and_leave_the_state_alone(op, shape, monkeypatch):
    import torch
    from ctc_beam_search_op_b200 import decoder
    T, B, C, W, P = shape
    blank = C - 1
    xd, _ = _inputs("float32", T, B, C, blank, 4)
    rng = np.random.default_rng(4)
    chunks = [(t, t + 8, rng.integers(1, 9, B).astype(np.int32)) for t in range(0, T, 8)]
    mk = lambda: op.CTCExtBeamSearchDecoderStream(batch_size=B, num_classes=C, beam_width=W,  # noqa: E731
                                                  top_paths=P, max_time=T, blank_index=blank)
    dec, ref = mk(), mk()
    subset = sorted(rng.choice(B, min(B, 300), replace=False).tolist())
    for k, c in enumerate(chunks):
        _feed(dec, xd, [c])
        _feed(ref, xd, [c])
        if k < 1:
            continue
        full = dec.top_paths_raw()
        for sel in ([3], [0, 2, 6], subset):
            for wait in (True, False):
                r = dec.top_paths_raw(sel, wait=wait)
                r = r if wait else r.result()
                check_selected(r, full, sel, P)
        out = dec.top_paths(np.isin(np.arange(B), [1, 5]))
        assert out.slots.tolist() == [1, 5] and out[2].shape == (2, P)
    assert_same(dec.top_paths_raw(), ref.top_paths_raw(), P)
    # a read too large for the deferred route (DEFER_MAX_BYTES_DEVICE) is made at once and handed back
    monkeypatch.setattr(decoder, "DEFER_MAX_BYTES_DEVICE", 0)
    r = dec.top_paths_raw([0, 2], wait=False)
    _feed(dec, xd, [(0, 8, np.full(B, 0, np.int32))])
    check_selected(r.result(), ref.top_paths_raw(), [0, 2], P)
    empty = dec.top_paths_raw([])
    assert empty.slots.tolist() == [] and tuple(empty[6].shape) == (0, P)
    assert _npy(empty[2][0]).tolist() == [0, 0]
    torch.cuda.synchronize()


@pytest.mark.parametrize("dt", ["float32", "float64"])
def test_reset_leaves_every_other_slot_untouched(op, dt):
    """Resetting (and refeeding) some slots mid-stream leaves the others bit-identical to the same
    stream without those resets; a reset slot starts from the root with its max_time budget renewed."""
    import torch
    T, B, C, W, P, blank = 24, 6, 29, 16, 2, 28
    xd, xo = _inputs(dt, T, B, C, blank, 6)
    sd = torch.float64 if dt == "float64" else torch.float32
    mk = lambda: op.CTCExtBeamSearchDecoderStream(batch_size=B, num_classes=C, beam_width=W,  # noqa: E731
                                                  top_paths=P, max_time=T, blank_index=blank, dtype=sd)
    dec, ref = mk(), mk()
    reset = [1, 4]
    for t in range(0, T, 6):
        if t == 12:
            dec.reset(reset)
        dec.step(xd[t:t + 6])
        ref.step(xd[t:t + 6])
    keep = [b for b in range(B) if b not in reset]
    check_selected(dec.top_paths_raw(keep), ref.top_paths_raw(), keep, P)
    # the reset slots consumed the last 12 frames only: the oracle on those
    want = L.oracle_decode(np.ascontiguousarray(xo[12:, reset]), np.full(len(reset), T - 12, np.int32), W, P,
                           False, blank, -1)
    assert not L.raw_mismatches(dec.top_paths_raw(reset), want)
    # a whole budget again: T more frames fit into a reset slot
    dec.reset(reset)
    for t in range(0, T, 6):
        dec.step(xd[t:t + 6], np.isin(np.arange(B), reset).astype(np.int32) * 6)
    check_selected(dec.top_paths_raw(reset), ref.top_paths_raw(), reset, P)


@pytest.mark.parametrize("dt", ["float32", "float64"])
def test_reset_and_step_replayed_from_a_cuda_graph(op, dt):
    """reset(mask_cuda) and step_device captured in one CUDA graph and replayed with a changing mask, chunk
    and lengths equal the same calls made eagerly."""
    import torch
    T, B, C, W, P, blank, Tc = 40, 6, 29, 20, 2, 28, 4
    xd, _ = _inputs(dt, T, B, C, blank, 12)
    rng = np.random.default_rng(12)
    plan = [(rng.random(B) < 0.2).astype(np.int32) for _ in range(T // Tc)]
    lens = [rng.integers(0, Tc + 1, B).astype(np.int32) for _ in range(T // Tc)]
    sd = torch.float64 if dt == "float64" else torch.float32
    mk = lambda: op.CTCExtBeamSearchDecoderStream(batch_size=B, num_classes=C, beam_width=W,  # noqa: E731
                                                  top_paths=P, max_time=T, blank_index=blank, dtype=sd)
    ref = mk()
    for k in range(T // Tc):
        ref.reset(plan[k])
        ref.step(xd[k * Tc:(k + 1) * Tc], lens[k])
    dec = mk()
    x_s = torch.zeros((Tc, B, C), dtype=xd.dtype, device="cuda")
    l_s = torch.zeros((B,), dtype=torch.int32, device="cuda")
    m_s = torch.zeros((B,), dtype=torch.int32, device="cuda")
    side = torch.cuda.Stream()
    side.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(side):  # warm-up outside the capture
        dec.reset(m_s)
        dec.step_device(x_s, l_s)
    torch.cuda.current_stream().wait_stream(side)
    g = torch.cuda.CUDAGraph()
    with torch.cuda.graph(g):
        dec.reset(m_s)
        dec.step_device(x_s, l_s)
    dec.reset()
    for k in range(T // Tc):
        m_s.copy_(torch.from_numpy(plan[k]))
        l_s.copy_(torch.from_numpy(lens[k]))
        x_s.copy_(xd[k * Tc:(k + 1) * Tc])
        g.replay()
    assert_same(dec.top_paths_raw(), ref.top_paths_raw(), P)


def test_errors_are_per_slot(op):
    import torch
    T, B, C, W, blank = 8, 3, 6, 4, 5
    x = np.random.default_rng(2).standard_normal((12, B, C)).astype(np.float32)
    # an over-fed slot is reported, with its own index, only when it is selected; its reset clears it
    dec = op.CTCExtBeamSearchDecoderStream(B, C, W, 1, max_time=T, blank_index=blank)
    dec.step(x[:6])
    dec.step(x[6:12], np.array([0, 6, 0], np.int32))
    assert dec.top_paths([0, 2])[2].shape == (2, 1)
    for sel in ([1], [0, 1], None):
        with pytest.raises(op.FailedPreconditionError, match=r"sequence_length\(1\) <= 8") as e:
            dec.top_paths(sel)
        assert e.value.batch_index == 1
    with pytest.raises(op.FailedPreconditionError):
        dec.top_paths([1, 2], wait=False).result()
    dec.reset([1])
    root = dec.top_paths_raw([1])  # the root: empty sequences, log-probability 0
    assert rows(host(root), 0, 1) == [[], [], [0]] and _npy(root[5][0]).tolist() == [1, 0]
    dec.step(x[:8], np.array([0, 8, 0], np.int32))  # a whole budget again
    got = dec.top_paths_raw([1])
    assert not L.raw_mismatches(got, L.oracle_decode(np.ascontiguousarray(x[:8, 1:2]), np.array([8], np.int32), W, 1,
                                                     False, blank, -1))
    assert rows(host(dec.top_paths_raw()), 1, 1) == rows(host(got), 0, 1)
    # too few leaves: only for the selected slots (a freshly reset slot holds the root alone)
    dec = op.CTCExtBeamSearchDecoderStream(B, C, W, 2, max_time=T, blank_index=blank)
    dec.step(x[:4])
    dec.reset([0])
    assert dec.top_paths([1, 2])[2].shape == (2, 2)
    for sel in ([0], None):
        with pytest.raises(op.InvalidArgumentError, match="Less leaves"):
            dec.top_paths(sel)
    # mixed score types, per slot, through the C-ABI; the stream-wide table mark survives slot resets
    from ctc_beam_search_op_b200 import _lib
    lib = _lib.load()
    C, W, P, blank = 29, 8, 1, 28
    x32 = torch.from_numpy(L.make_logits("gauss", 16, B, C, blank, 1)).cuda()
    stream = torch.cuda.current_stream().cuda_stream
    sizes = _lib.CtcxSizes(*[(ctypes.c_int64 * P)() for _ in range(4)])
    n32 = lib.ctcx_stream_workspace_bytes_v(_lib.F32, 16, B, C, W, P)
    n64 = lib.ctcx_stream_workspace_bytes_v(_lib.F64, 16, B, C, W, P)
    ws = torch.empty(n64, dtype=torch.uint8, device="cuda")
    lens = torch.full((B,), 4, dtype=torch.int32, device="cuda")

    def step(x, nb, lm=None):
        return lib.ctcx_stream_step_v(ws.data_ptr(), nb, 16, B, C, W, P, x.data_ptr(),
                                      _lib.F64 if x.dtype == torch.float64 else _lib.F32, 0, 4, lens.data_ptr(),
                                      blank, None if lm is None else lm.data_ptr(), stream)

    def mask(sel):
        return torch.tensor([1 if b in sel else 0 for b in range(B)], dtype=torch.int32, device="cuda")

    def top(sel):
        m = mask(sel)
        return lib.ctcx_stream_top_paths_slots(ws.data_ptr(), 16, B, C, W, P, 0, -1, m.data_ptr(), stream,
                                               ctypes.byref(sizes), None)

    def reset_slots(sel):
        m = mask(sel)
        assert lib.ctcx_stream_reset_slots(ws.data_ptr(), n64, _lib.F32, 16, B, C, W, P, m.data_ptr(), stream) == 0
        torch.cuda.synchronize()

    assert lib.ctcx_stream_reset_v(ws.data_ptr(), n64, _lib.F32, 16, B, C, W, P, stream) == 0
    assert step(x32[:4], n32) == 0
    assert step(x32[4:8].double(), n64) == 0     # a float64 step on a float stream: every slot is mixed now
    assert top([0]) == 8 and top([2]) == 8
    reset_slots([0])
    assert top([0]) == 0
    assert top([0, 1]) == 8
    assert top([1]) == 8
    # a positive table entry marks the stream, not a slot: a slot reset keeps it, the full reset clears it
    assert lib.ctcx_stream_reset_v(ws.data_ptr(), n64, _lib.F32, 16, B, C, W, P, stream) == 0
    bad = torch.zeros((C + 1, C), dtype=torch.float32, device="cuda")
    bad[3, 4] = 0.5
    assert step(x32[:4], n32, bad) == 0
    assert top([1]) == 8
    reset_slots([0, 1, 2])
    assert top([1]) == 8
    assert lib.ctcx_stream_reset_v(ws.data_ptr(), n64, _lib.F32, 16, B, C, W, P, stream) == 0
    assert top([1]) == 0
    torch.cuda.synchronize()


def test_python_rejects_bad_selections(op):
    import torch
    dec = op.CTCExtBeamSearchDecoderStream(4, 6, 4, 1, max_time=8, blank_index=5)
    for bad in ([4], [-1], np.zeros(3, bool), torch.zeros(5, dtype=torch.int32).cuda(),
                torch.zeros(4, dtype=torch.int64).cuda(), torch.zeros(4, dtype=torch.float32)):
        with pytest.raises(op.InvalidArgumentError):
            dec.reset(bad)
        with pytest.raises(op.InvalidArgumentError):
            dec.top_paths(bad)


def test_cabi_deferred_read_packed_before_later_steps(op):
    """The C-ABI's deferred read, packed right after the trace: later steps and a slot reset enqueued before
    ctcx_finish leave the packed result and the sizes alone (the pack took log_probability from the final
    beam before they rewrote it)."""
    import torch
    from ctc_beam_search_op_b200 import _lib, decoder
    lib = _lib.load()
    T, B, C, W, P, blank = 32, 5, 29, 16, 2, 28
    xd, _ = _inputs("float32", T, B, C, blank, 21)
    dec = op.CTCExtBeamSearchDecoderStream(batch_size=B, num_classes=C, beam_width=W, top_paths=P, max_time=T,
                                           blank_index=blank)
    dec.step(xd[:12])
    want = host(dec.top_paths_raw())
    sel = [0, 3]
    m = torch.tensor([1 if b in sel else 0 for b in range(B)], dtype=torch.int32, device="cuda")
    st = torch.cuda.current_stream().cuda_stream
    ws = dec._ws.data_ptr()
    n_bound = decoder._bound_elems(T, B, P, torch.full((len(sel),), T, dtype=torch.int32), False)
    buf = torch.empty((n_bound,), dtype=torch.int64, device="cuda")
    assert lib.ctcx_stream_top_paths_slots(ws, T, B, C, W, P, 0, -1, m.data_ptr(), st, None, None) == 0
    assert lib.ctcx_pack_compact(ws, T, B, P, 4, buf.data_ptr(), n_bound, st) == 0
    dec.step(xd[12:20])
    dec.reset(sel)
    dec.step(xd[20:24])
    arr = ctypes.c_int64 * P
    n_dec, max_dec, n_ali, max_ali = arr(), arr(), arr(), arr()
    sizes = _lib.CtcxSizes(n_dec, max_dec, n_ali, max_ali)
    assert lib.ctcx_finish(ws, T, B, P, st, ctypes.byref(sizes), None) == 0
    groups, logp = decoder._carve(buf[:decoder._pack_elems(B, P, (n_dec, n_ali), False)], B, P, (n_dec, n_ali),
                                  False)
    got = host(decoder.CTCExtBeamSearchDecoder(*groups, logp))
    for b in range(B):
        if b in sel:
            assert rows(got, b, P) == rows(want, b, P), "slot %d" % b
        else:
            assert rows(got, b, P)[:2 * P] == [[]] * (2 * P), "slot %d" % b


def test_stream_on_an_unindexed_device_takes_cuda_masks(op):
    import torch
    dec = op.CTCExtBeamSearchDecoderStream(4, 6, 4, 1, max_time=8, blank_index=5, device="cuda")
    dec.step(np.random.default_rng(3).standard_normal((4, 4, 6)).astype(np.float32))
    m = torch.tensor([0, 1, 0, 1], dtype=torch.int32, device="cuda")
    assert dec.top_paths(m).slots.tolist() == [1, 3]
    dec.reset(m)
    assert dec.top_paths_raw(m)[4][0].numel() == 0
