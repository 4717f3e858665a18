"""The streaming decoder with every score type and input the one-shot decode takes: float16 / bfloat16
chunks read in place, float64 streams (the double kernels' state blocks), the scorer table, batch
shards stepped in place. Any chunking must equal the one-shot decode of the same score type and table,
and TopPaths mid-stream the oracle on the prefix, bit for bit: labels, alignments and the uint32 /
uint64 bits of log_probability."""
import ctypes

import numpy as np
import pytest

import ctcx_testlib as L

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


def _npy(a):
    return a.detach().cpu().numpy() if hasattr(a, "detach") else np.asarray(a)


def assert_same(raw, one, P):
    for g in range(6):
        for p in range(P):
            np.testing.assert_array_equal(_npy(raw[g][p]), _npy(one[g][p]))
    a, b = _npy(raw[6]), _npy(one[6])
    assert a.dtype == b.dtype
    view = np.uint64 if a.dtype == np.float64 else np.uint32
    np.testing.assert_array_equal(a.view(view), b.view(view))


def _inputs(dt, T, B, C, blank, seed):
    """Device logits of torch dtype `dt`, and the values the kernels see, for the oracle (float32 for the
    half types, float64 for float64)."""
    import torch
    if dt == "float64":
        x = np.random.default_rng(seed).standard_normal((T, B, C))
        return torch.from_numpy(x).cuda(), x
    xd = torch.from_numpy(L.make_logits("gauss", T, B, C, blank, seed)).to(getattr(torch, dt)).cuda()
    return xd, xd.float().cpu().numpy()


def _bigram(C, seed):
    return -np.abs(np.random.default_rng(seed).standard_normal((C + 1, C))).astype(np.float32)


def stream_and_check(op, dt, T, B, C, W, P, blank, table=None, seed=3, prefix_checks=True):
    """Feeds every utterance in its own random chunking (1-frame chunks and chunks of 0 frames for some
    utterances included), checks TopPaths at random points against the oracle on the prefix, the end
    against the one-shot decode; twice, the second time after reset()."""
    import torch
    xd, xo = _inputs(dt, T, B, C, blank, seed)
    sl = L.ragged_lengths(T, B, seed)
    rng = np.random.default_rng(seed + 7)
    dec = op.CTCExtBeamSearchDecoderStream(batch_size=B, num_classes=C, beam_width=W, top_paths=P, max_time=T,
                                           blank_index=blank, dtype=torch.float64 if dt == "float64" else torch.float32,
                                           expansion_scores=table)
    one = op.ctc_ext_beam_search_decoder_raw(xd, torch.from_numpy(sl).cuda(), beam_width=W, top_paths=P,
                                             blank_index=blank, expansion_scores=table)
    bidx = torch.arange(B, device="cuda")
    for _ in range(2):
        pos = np.zeros(B, np.int64)
        while (pos < sl).any():
            ct = min(int(rng.choice([1, 1, 2, 5, 9, 17])), T)  # (a chunk is at most the stream's max_time)
            lens = np.minimum(rng.integers(0, ct + 1, B), sl - pos).astype(np.int32)
            # chunk row i of utterance b = frame pos[b] + i of that utterance (rows past its end: anything)
            t = torch.from_numpy(np.minimum(pos[None, :] + np.arange(ct)[:, None], T - 1)).cuda()
            chunk = xd[t, bidx[None, :].expand(ct, B)]
            dec.step(chunk, lens)
            pos += lens
            if prefix_checks and rng.random() < 0.25 and (P == 1 or pos.min() >= 2):
                want = L.oracle_decode(xo, pos.astype(np.int32), W, P, False, blank, -1, lm=table)
                bad = L.raw_mismatches(dec.top_paths_raw(), want)
                assert not bad, "prefix %s: utterances %s differ from the oracle" % (pos.tolist(), bad[:8])
        raw = dec.top_paths_raw()
        assert_same(raw, one, P)
        dec.reset()
    return raw


# (dtype, T, B, C, W, P, blank): narrow (C <= 32), wide (32 < C <= 2048, W <= 256), generic (W = 300)
HALF_CASES = [(dt,) + s for dt in ("float16", "bfloat16")
              for s in ((40, 5, 29, 20, 2, 28), (30, 4, 40, 24, 2, 7), (24, 3, 1024, 16, 1, 1023),
                        (20, 3, 12, 300, 2, 0))]
F64_CASES = [("float64",) + s for s in ((40, 5, 29, 20, 2, 28), (40, 4, 29, 100, 1, 28), (30, 3, 29, 200, 2, 0),
                                         (30, 4, 40, 24, 2, 7), (20, 3, 40, 300, 1, 7), (16, 2, 40, 512, 2, 0))]


@pytest.mark.parametrize("case", HALF_CASES + F64_CASES, ids=lambda c: "%s-C%d-W%d" % (c[0], c[3], c[4]))
def test_any_chunking_equals_the_one_shot_decode(op, case):
    dt, T, B, C, W, P, blank = case
    stream_and_check(op, dt, T, B, C, W, P, blank)


@pytest.mark.parametrize("shape", [(40, 5, 29, 20, 2, 28), (40, 4, 29, 100, 1, 28), (30, 4, 40, 24, 2, 7),
                                   (20, 3, 12, 300, 1, 0)], ids=lambda s: "C%d-W%d" % (s[2], s[3]))
@pytest.mark.parametrize("dt", ["float32", "bfloat16"])
def test_scorer_table_streams(op, shape, dt):
    """A random bigram table: narrow (its LM variant), wide and generic shapes, which all take the table
    on the generic kernel or the narrow kernel's LM variant; bfloat16 chunks are widened where the one-shot
    decode widens them."""
    T, B, C, W, P, blank = shape
    stream_and_check(op, dt, T, B, C, W, P, blank, table=_bigram(C, 11))


@pytest.mark.parametrize("dt", ["bfloat16", "float64"])
def test_batch_shards_are_stepped_in_place(op, dt):
    """x[:, b0:b1, :] of a wider device tensor, chunk by chunk, equals the one-shot decode of the shard."""
    import torch
    for (T, Bw, C, W, P, blank, b0, b1) in [(30, 9, 29, 16, 2, 28, 2, 7), (24, 7, 40, 12, 1, 7, 3, 6)]:
        xd, _ = _inputs(dt, T, Bw, C, blank, 5)
        B = b1 - b0
        dec = op.CTCExtBeamSearchDecoderStream(batch_size=B, num_classes=C, beam_width=W, top_paths=P, max_time=T,
                                               blank_index=blank, dtype=np.float64 if dt == "float64" else np.float32)
        for t in range(0, T, 7):
            view = xd[t:t + 7, b0:b1, :]
            assert not view.is_contiguous()
            dec.step(view)
        one = op.ctc_ext_beam_search_decoder_raw(xd[:, b0:b1, :], [T] * B, beam_width=W, top_paths=P,
                                                 blank_index=blank)
        assert_same(dec.top_paths_raw(), one, P)


def _sms():
    import torch
    return int(torch.cuda.get_device_properties(torch.cuda.current_device()).multi_processor_count)


@pytest.mark.parametrize("variant", ["bfloat16", "float16", "table", "float64"])
def test_large_batches(op, variant):
    """B beyond 2 x SMs: the four-CTAs-per-SM variants of the half-precision and scorer kernels, with
    chunks in which every utterance idles."""
    import torch
    T, C, W, P, blank = 24, 29, 16, 1, 28
    B = 2 * _sms() + 9
    dt = "float32" if variant == "table" else variant
    table = _bigram(C, 4) if variant == "table" else None
    xd, _ = _inputs(dt, T, B, C, blank, 9)
    sl = L.ragged_lengths(T, B, 9)
    dec = op.CTCExtBeamSearchDecoderStream(batch_size=B, num_classes=C, beam_width=W, top_paths=P, max_time=T,
                                           blank_index=blank, dtype=np.float64 if dt == "float64" else np.float32,
                                           expansion_scores=table)
    for t in range(0, T, 6):
        dec.step(xd[t:t + 6], np.zeros(B, np.int32))  # an idle chunk
        dec.step(xd[t:t + 6], np.clip(sl - t, 0, 6).astype(np.int32))
    one = op.ctc_ext_beam_search_decoder_raw(xd, torch.from_numpy(sl).cuda(), beam_width=W, top_paths=P,
                                             blank_index=blank, expansion_scores=table)
    assert_same(dec.top_paths_raw(), one, P)


WIPE = [c for c in L.wipe_cases() if c.W <= 256]


@pytest.mark.parametrize("variant", ["float16", "bfloat16", "float64", "zero-table"])
@pytest.mark.parametrize("c", WIPE, ids=[c.name for c in WIPE])
def test_revisit_wipe_cases_streamed_through_their_deepest_frames(op, c, variant):
    """tests/golden/wipe_cases.npz (logits on the k/16 grid: exact in half precision), one chunk ending
    right before the deepest frame of the revisit-wipe fixed point and one right after it: equal to the
    oracle (an all-zero table is an exact no-op on the scores)."""
    import torch
    f64 = variant == "float64"
    if f64 and c.C > 65:
        pytest.skip("the double kernel's shared memory does not take this vocabulary at this beam width")
    t = int(np.argmax(c.iters))
    cuts = sorted({0, t, t + 1, c.T} | ({32, 64} if c.T >= 64 else set()))
    xt = torch.from_numpy(np.ascontiguousarray(c.x)).to(
        torch.float64 if f64 else torch.float32 if variant == "zero-table" else getattr(torch, variant)).cuda()
    table = np.zeros((c.C + 1, c.C), np.float32) if variant == "zero-table" else None
    dec = op.CTCExtBeamSearchDecoderStream(batch_size=1, num_classes=c.C, beam_width=c.W, top_paths=c.P,
                                           max_time=c.T, merge_repeated=c.merge, blank_index=c.blank,
                                           dtype=torch.float64 if f64 else torch.float32, expansion_scores=table)
    for a, b in zip(cuts[:-1], cuts[1:]):
        if b > a:
            dec.step(xt[a:b])
    want = L.oracle_decode(c.x.astype(np.float64) if f64 else c.x, c.sl, c.W, c.P, c.merge, c.blank, -1)
    bad = L.raw_mismatches(dec.top_paths_raw(), want)
    assert not bad, "%s %s cuts %s" % (c.name, variant, cuts)


@pytest.mark.parametrize("variant", ["bfloat16", "float64", "table"])
def test_step_device_replayed_from_a_cuda_graph(op, variant, request):
    """step_device() with half chunks, a float64 stream and a table only enqueues work: captured once into
    a CUDA graph and replayed per chunk it gives what step() gives. (The test hook's generic kernel on a
    fast-path shape has no room to widen half chunks, and step_device() never allocates: there it takes
    a shape of the generic kernel's own.)"""
    import torch
    T, B, C, W, P, blank, Tc = 64, 6, 29, 20, 2, 28, 8
    if variant == "bfloat16" and request.node.callspec.params["op"] == "generic":
        C, W, blank = 12, 300, 0
    dt = "float32" if variant == "table" else variant
    table = _bigram(C, 8) if variant == "table" else None
    xd, _ = _inputs(dt, T, B, C, blank, 19)
    mk = lambda: op.CTCExtBeamSearchDecoderStream(  # noqa: E731
        batch_size=B, num_classes=C, beam_width=W, top_paths=P, max_time=T, blank_index=blank,
        dtype=np.float64 if dt == "float64" else np.float32, expansion_scores=table)
    ref = mk()
    for t in range(0, T, Tc):
        ref.step(xd[t:t + Tc])
    dec = mk()
    x_static = torch.zeros((Tc, B, C), dtype=xd.dtype, device="cuda")
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
    for t in range(0, T, Tc):
        x_static.copy_(xd[t:t + Tc])
        g.replay()
    assert_same(dec.top_paths_raw(), ref.top_paths_raw(), P)


def test_python_errors(op):
    import torch
    dec = op.CTCExtBeamSearchDecoderStream(2, 6, 4, 1, max_time=8, blank_index=5, dtype=torch.float64)
    for dt in (np.float32, np.float16):
        with pytest.raises(TypeError):
            dec.step(np.zeros((2, 2, 6), dt))
    with pytest.raises(TypeError):
        dec.step(torch.zeros((2, 2, 6), dtype=torch.bfloat16).cuda())
    with pytest.raises(op.InvalidArgumentError):
        dec.step_device(torch.zeros((2, 2, 6), dtype=torch.float32).cuda(), torch.full((2,), 2, dtype=torch.int32).cuda())
    # overflow past max_time in a float64 stream: reported as in float32
    x = np.random.default_rng(2).standard_normal((12, 2, 6))
    dec.step(x[:6])
    dec.step(x[6:12])
    with pytest.raises(op.FailedPreconditionError, match=r"sequence_length\(0\) <= 8"):
        dec.top_paths()
    dec.reset()
    dec.step(x[:8])
    lp = dec.top_paths()[2]
    assert lp.dtype == torch.float64
    want = L.oracle_decode(x[:8], np.full(2, 8, np.int32), 4, 1, False, 5, -1)
    np.testing.assert_array_equal(lp.cpu().numpy().view(np.uint64), want.logp.view(np.uint64))


def test_cabi_errors_reported_at_top_paths(op):
    """A table entry > 0 passed to a step, and float32 and float64 steps mixed in one stream, make the
    next top_paths return CTCX_ERR_BAD_ARGUMENT (the steps themselves never synchronise); a reset clears
    both. A float stream's workspace is too small for a float64 step."""
    import torch
    from ctc_beam_search_op_b200 import _lib
    lib = _lib.load()
    T, B, C, W, P, blank = 16, 3, 29, 8, 1, 28
    x32 = torch.from_numpy(L.make_logits("gauss", T, B, C, blank, 1)).cuda()
    x64 = x32.double()
    lens = torch.full((B,), 4, dtype=torch.int32, device="cuda")
    stream = torch.cuda.current_stream().cuda_stream
    sizes = _lib.CtcxSizes((ctypes.c_int64 * P)(), (ctypes.c_int64 * P)(), (ctypes.c_int64 * P)(), (ctypes.c_int64 * P)())

    def step(ws, nb, x, lm=None):
        return lib.ctcx_stream_step_v(ws.data_ptr(), nb, T, B, C, W, P, x.data_ptr(), _lib.F64 if x.dtype == torch.float64
                                      else _lib.F32, 0, 4, lens.data_ptr(), blank,
                                      None if lm is None else lm.data_ptr(), stream)

    def top(ws):
        return lib.ctcx_stream_top_paths(ws.data_ptr(), T, B, C, W, P, 0, -1, stream, ctypes.byref(sizes), None)

    def reset(ws, nb, sd):
        assert lib.ctcx_stream_reset_v(ws.data_ptr(), nb, sd, T, B, C, W, P, stream) == 0

    n32 = lib.ctcx_stream_workspace_bytes_v(_lib.F32, T, B, C, W, P)
    n64 = lib.ctcx_stream_workspace_bytes_v(_lib.F64, T, B, C, W, P)
    ws = torch.empty(n64, dtype=torch.uint8, device="cuda")
    # a positive table entry
    reset(ws, n64, _lib.F32)
    bad = torch.zeros((C + 1, C), dtype=torch.float32, device="cuda")
    bad[3, 4] = 0.5
    assert step(ws, n32, x32[:4]) == 0
    assert step(ws, n32, x32[4:8], bad) == 0
    assert step(ws, n32, x32[8:12], torch.zeros_like(bad)) == 0
    assert top(ws) == 8
    reset(ws, n64, _lib.F32)
    assert step(ws, n32, x32[:4], torch.zeros_like(bad)) == 0
    assert top(ws) == 0
    # mixed score types, both ways, in a workspace with room for both
    for first, then, sd in ((x32, x64, _lib.F32), (x64, x32, _lib.F64)):
        reset(ws, n64, sd)
        assert step(ws, n64, first[:4]) == 0
        assert top(ws) == 0
        assert step(ws, n64, then[4:8]) == 0
        assert top(ws) == 8
        reset(ws, n64, sd)
        assert step(ws, n64, first[:4]) == 0
        assert top(ws) == 0
    # a float64 stream stepped only in float32 is mixed too
    reset(ws, n64, _lib.F64)
    assert step(ws, n64, x32[:4]) == 0
    assert top(ws) == 8
    # a float stream's workspace is short of a float64 step
    assert step(ws, n32, x64[:4]) == 10
    torch.cuda.synchronize()
