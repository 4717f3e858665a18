"""CPU suite, part 2: host logic and the C-ABI surface. No compute calls (no GPU here): the library
must load, export every symbol include/ctcx.h declares, map return codes to the reference's
messages, and the Python host must validate exactly like the reference op (kernels.cc:97-160).
"""
import ctypes
import os
import re

import numpy as np
import pytest

import ctcx_testlib as L

ROOT = L.ROOT


@pytest.fixture(scope="module")
def lib():
    from ctc_beam_search_op_b200 import _lib
    return _lib.load()


def test_cabi_exports_every_declared_symbol(lib):
    hdr = open(os.path.join(ROOT, "include", "ctcx.h")).read()
    declared = set(re.findall(r"\b(ctcx_[a-z0-9_]+)\s*\(", hdr))
    assert {"ctcx_decode_f32", "ctcx_pack_f32", "ctcx_decode_host_f32", "ctcx_workspace_bytes"} <= declared
    for sym in sorted(declared):
        assert hasattr(lib, sym), "libctcx.so does not export %s" % sym
    from ctc_beam_search_op_b200 import _lib
    assert declared == set(_lib.EXPORTS)


def test_error_messages_are_the_references(lib):
    want = {1: "inputs is not a 3-Tensor", 2: "max_time is 0", 3: "sequence_length is not a vector",
            6: "requested more paths than the beam width.",
            7: "Less leaves in the beam search than requested."}
    for code, msg in want.items():
        assert lib.ctcx_strerror(code).decode() == msg
    assert lib.ctcx_strerror(4).decode().startswith("len(sequence_length) != batch_size.")


def test_workspace_and_limits(lib):
    from ctc_beam_search_op_b200 import _lib
    lim = _lib.CtcxLimits()
    assert lib.ctcx_get_limits(ctypes.byref(lim)) == 100  # built for sm_100
    assert lim.max_beam_width >= 256 and lim.max_classes >= 1024
    small = lib.ctcx_workspace_bytes(50, 8, 29, 10, 3)
    big = lib.ctcx_workspace_bytes(500, 256, 29, 100, 1)
    assert 0 < small < big
    assert big >= 500 * 256 * 100 * 4  # back-pointer records (4 B per slot and frame here) dominate
    assert lib.ctcx_workspace_bytes(0, 8, 29, 10, 3) == 0


def test_cabi_validation_without_device(lib):
    """Argument errors are reported before any CUDA call."""
    from ctc_beam_search_op_b200 import _lib
    sizes = _lib.CtcxSizes()
    args = lambda T, B, C, W, P, blank: (None, T, B, C, None, W, P, 0, blank, -1, None, 0, None,  # noqa: E731
                                         ctypes.byref(sizes), None)
    assert lib.ctcx_decode_f32(*args(0, 1, 3, 2, 1, 0)) == 2     # max_time is 0
    assert lib.ctcx_decode_f32(*args(5, 1, 3, 0, 1, 0)) == 8     # beam_width < 1
    assert lib.ctcx_decode_f32(*args(5, 1, 3, 2, 1, 3)) == 8     # blank_index out of range
    assert lib.ctcx_decode_f32(*args(5, 1, 3, 5000, 1, 0)) == 9  # beyond this build's limits
    assert lib.ctcx_decode_f32(*args(5, 1, 3, 2, 1, 0)) == 10    # no workspace

    # Every other entry that validates before touching a device pointer. All device pointers are
    # null: a call that got past its checks would return 10 (no workspace), never dereference one.
    sz, fl = ctypes.byref(sizes), None
    view = lambda dt, ts, T, B, C, W, P, blank: lib.ctcx_decode_view(  # noqa: E731
        None, dt, ts, T, B, C, None, W, P, 0, blank, -1, None, 0, None, sz, fl)
    assert view(7, 0, 5, 1, 3, 2, 1, 0) == 8          # no such dtype (before max_time)
    assert view(7, 0, 0, 1, 3, 2, 1, 0) == 8
    assert view(0, -1, 5, 1, 3, 2, 1, 0) == 8         # negative time stride
    assert view(2, 0, 0, 1, 3, 2, 1, 0) == 2
    assert view(3, 0, 0, 1, 3, 2, 1, 0) == 2
    assert view(1, 0, 5, -1, 3, 2, 1, 0) == 8         # negative batch
    assert view(0, 0, 5, 1, 0, 2, 1, 0) == 8          # no classes
    assert view(3, 0, 5, 1, 3, 2, 0, 0) == 8          # top_paths < 1
    assert view(2, 0, 5, 1, 3, 2, 1, -1) == 8         # negative blank
    assert view(0, 0, 5, 1, 70000, 2, 1, 0) == 9      # more classes than this build takes
    assert view(3, 0, 5, 1, 3, 1025, 1, 0) == 9
    assert view(0, 5, 5, 2, 3, 2, 1, 0) == 8          # stride shorter than a frame (B * C = 6)
    assert view(0, 6, 5, 2, 3, 2, 1, 0) == 10
    assert view(3, 0, 5, 0, 3, 2, 1, 0) == 10         # an empty batch still needs its workspace
    assert view(1, 0, 5, 1, 3, 1, 2, 0) == 10         # top_paths > beam_width: reported on the device
    half = lambda dt, T, W, blank: lib.ctcx_decode_half(  # noqa: E731
        None, dt, None, T, 1, 3, None, W, 1, 0, blank, -1, None, 0, None, sz, fl)
    assert half(2, 0, 2, 0) == 2                      # unknown half type: max_time is checked first
    assert half(2, 5, 2, 0) == 8
    assert half(-1, 5, 2, 0) == 8
    assert half(0, 0, 2, 0) == 2
    assert half(1, 5, 0, 0) == 8
    assert half(0, 5, 2, 3) == 8
    assert half(1, 5, 2000, 0) == 9
    assert half(0, 5, 2, 0) == 10
    f64 = lambda T, C, W, P, blank: lib.ctcx_decode_f64(  # noqa: E731
        None, T, 1, C, None, W, P, 0, blank, -1, None, 0, None, sz, fl)
    assert f64(0, 3, 2, 1, 0) == 2
    assert f64(-1, 3, 2, 1, 0) == 8
    assert f64(5, 3, 2, 1, 3) == 8
    assert f64(5, 65536, 2, 1, 0) == 9
    assert f64(5, 3, 2, 1, 0) == 10
    scorer = lambda T, C, W, blank: lib.ctcx_decode_scorer_f32(  # noqa: E731  (no table: the plain decode)
        None, T, 1, C, None, W, 1, 0, blank, -1, None, None, 0, None, sz, fl)
    assert scorer(0, 3, 2, 0) == 2
    assert scorer(5, 3, 0, 0) == 8
    assert scorer(5, 3, 2, 5) == 8
    assert scorer(5, 3, 4096, 0) == 9
    assert scorer(5, 3, 2, 0) == 10
    hostin = lambda dt, ts, T, B, C, W, P, blank: lib.ctcx_decode_hostin(  # noqa: E731
        None, dt, ts, T, B, C, None, W, P, 0, blank, -1, None, 0, None, 0, None, None, sz, fl)
    assert hostin(9, 0, 0, 1, 3, 2, 1, 0) == 2        # max_time before the dtype here
    assert hostin(9, 0, 5, 1, 3, 2, 1, 0) == 8
    assert hostin(3, 0, 5, 1, 3, 0, 1, 0) == 8
    assert hostin(0, 0, 5, 1, 3, 2, 1, 3) == 8
    assert hostin(1, 0, 5, 1, 3, 1025, 1, 0) == 9
    assert hostin(0, 2, 5, 1, 3, 2, 1, 0) == 8        # host stride shorter than a frame
    assert hostin(0, 0, 5, 1, 3, 2, 1, 0) == 10       # workspace before staging, host pointers and streams
    assert hostin(2, 9, 5, 3, 3, 2, 5, 0) == 10
    reset = lambda T, B, C, W, P: lib.ctcx_stream_reset(None, 0, T, B, C, W, P, None)  # noqa: E731
    assert reset(0, 1, 3, 2, 1) == 8
    assert reset(5, -1, 3, 2, 1) == 8
    assert reset(5, 1, 0, 2, 1) == 8
    assert reset(5, 1, 3, 2, 0) == 8
    assert reset(5, 1, 3, 1025, 1) == 9
    assert reset(5, 1, 65536, 2, 1) == 9
    assert reset(5, 1, 3, 2, 3) == 6                  # top_paths > beam_width, before the workspace
    assert reset(5, 1, 3, 2, 1) == 10
    assert reset(5, 0, 3, 2, 1) == 10
    # the stream step and top_paths check the workspace before their arguments
    assert lib.ctcx_stream_step_f32(None, 0, 1, 3, 2, 1, None, 0, None, 9, None) == 10
    assert lib.ctcx_stream_step_f32(None, 5, 1, 3, 5000, 1, None, 1, None, 0, None) == 10
    assert lib.ctcx_stream_top_paths(None, 0, 1, 3, 2, 1, 0, -1, None, sz, fl) == 10
    assert lib.ctcx_stream_top_paths(None, 5, 1, 3, 5000, 1, 0, -1, None, None, fl) == 10
    nul6 = [None] * 6
    for pack in (lib.ctcx_pack_f32, lib.ctcx_pack_f64):
        for T, B, P in ((5, 1, 1), (0, 1, 1), (5, -1, 1), (5, 1, 0), (5, 0, 1)):
            assert pack(None, T, B, P, *nul6, None, None) == 10
    for T, B, P, rb in ((5, 1, 1, 4), (5, 1, 1, 8), (5, 1, 1, 2), (0, 1, 1, 4), (5, 0, 1, 4), (5, 1, 0, 8)):
        assert lib.ctcx_pack_compact(None, T, B, P, rb, None, 0, None) == 10
    for T, B, P in ((5, 1, 1), (0, 1, 1), (5, -1, 1), (5, 1, 0), (5, 0, 1)):
        assert lib.ctcx_finish(None, T, B, P, None, sz, fl) == 10
        assert lib.ctcx_result_copy_async(None, T, B, P, None, 0, None) == 10
    buf = ctypes.create_string_buffer(1024)
    assert lib.ctcx_finish(None, 5, 1, 1, None, None, fl) == 10
    assert lib.ctcx_result_copy_async(None, 5, 1, 1, buf, 1024, None) == 10
    prep = lambda route, dt, T, B, C, ts, blank, W: lib.ctcx_debug_prepass(  # noqa: E731
        route, None, dt, T, B, C, ts, blank, W, None, None, None, None, None)
    for route in (0, 1, 2):
        assert prep(route, 0, 2, 2, 40, 0, 0, 4) == 8    # no logits
        assert prep(route, 0, 0, 2, 40, 0, 0, 4) == 8
        assert prep(route, 3, 2, 2, 40, 0, 40, 4) == 8
        assert prep(route, 5, 2, 2, 40, 0, 0, 4) == 8
        assert prep(route, 1, 2, 2, 40, 79, 0, 4) == 8
        assert prep(route, 2, 2, 2, 70000, 0, 0, 4) == 8


# ctcx_workspace_bytes at shapes on both sides of every route and tier edge: the layout is part of the
# ABI (a caller sizes its buffer from it), so these values do not change without a reason.
WORKSPACE_BYTES = [
    # narrow: beam tiers 32 / 128 / 256, the 4608-entry candidate list (32 x 144), C = 1, 2
    ((50, 8, 29, 10, 3), 36352), ((50, 8, 32, 32, 1), 72448), ((50, 8, 32, 33, 2), 77568),
    ((50, 8, 29, 128, 4), 265984), ((50, 8, 29, 129, 1), 258816), ((50, 8, 16, 256, 1), 502528),
    ((50, 8, 16, 257, 1), 941312), ((50, 8, 32, 144, 1), 287488), ((50, 8, 32, 145, 1), 340736),
    ((20, 3, 2, 1024, 7), 623616), ((10, 2, 1, 1, 1), 5120), ((1, 1, 3, 1, 1), 5120),
    # wide: C = 33 and 2048 / 2049, beam tiers
    ((40, 4, 33, 1, 1), 15360), ((40, 4, 33, 32, 2), 64256), ((40, 4, 33, 33, 1), 64000),
    ((40, 4, 1000, 128, 1), 831232), ((40, 4, 1000, 129, 3), 835072), ((40, 4, 2048, 8, 1), 41472),
    ((40, 4, 2048, 256, 2), 1687296), ((40, 4, 2048, 257, 1), 1687552), ((40, 4, 2049, 8, 1), 1329920),
    # generic: beams up to 1024, C up to 65535, empty batches, a beam beyond the limits
    ((7, 3, 300, 512, 5), 178176), ((7, 3, 300, 513, 1), 177920), ((7, 3, 300, 1024, 1024), 687616),
    ((6, 2, 65535, 8, 2), 3151872), ((6, 2, 65535, 1024, 1), 3330816), ((6, 2, 5000, 100, 3), 262656),
    ((10, 0, 29, 10, 1), 1024), ((10, 0, 5000, 300, 2), 1024), ((5, 1, 3, 5000, 1), 405248),
]


def test_workspace_bytes_table(lib):
    for shape, want in WORKSPACE_BYTES:
        assert lib.ctcx_workspace_bytes(*shape) == want, shape
        assert lib.ctcx_stream_workspace_bytes(*shape) == want, shape
    for bad in ((5, -1, 3, 2, 1), (5, 1, 0, 2, 1), (5, 1, 3, 0, 1), (5, 1, 3, 2, 0)):
        assert lib.ctcx_workspace_bytes(*bad) == 0
    assert [lib.ctcx_result_bytes(p) for p in (0, 1, 3)] == [0, 96, 160]


def _result_block(P, sizes, stats):
    """A result block as ctcx_result_copy_async delivers it: sizes [4, P] int64, then 16 status words."""
    blk = np.zeros(4 * P * 2 + 8, np.int64)
    blk[:4 * P] = np.asarray(sizes, np.int64).reshape(-1)
    st = blk[4 * P:].view(np.int32)
    st[:len(stats)] = stats
    return blk


def test_result_parse(lib):
    """ctcx_result_parse reads the status words in a fixed order, then copies the sizes out."""
    from ctc_beam_search_op_b200 import _lib
    T, B, P = 9, 5, 3
    sz = [[7, 0, 12], [4, 0, 6], [40, 40, 33], [9, 9, 8]]
    ok = [0x3, B, B, B, B, B]

    def parse(stats, P=P, flags=True, fields=(0, 1, 2, 3)):
        blk = _result_block(P, sz if P == 3 else [[0] * P] * 4, stats)
        got = [np.full(P, -7, np.int64) for _ in range(4)]
        ptr = lambda a: a.ctypes.data_as(_lib._i64p)  # noqa: E731
        s = _lib.CtcxSizes(*[ptr(got[k]) if k in fields else None for k in range(4)])
        f = ctypes.c_int32(-7)
        rc = lib.ctcx_result_parse(blk.ctypes.data, T, B, P, ctypes.byref(s), ctypes.byref(f) if flags else None)
        return rc, [g.tolist() for g in got], f.value

    rc, got, f = parse(ok)
    assert rc == 0 and got == sz and f == 3
    rc, got, _ = parse(ok, flags=False, fields=(1, 3))
    assert rc == 0 and got == [[-7] * 3, sz[1], [-7] * 3, sz[3]]
    assert parse([0, 1, B, B, B, B], P=1)[0] == 7  # P = 1 layout: status words right after 4 sizes
    # one failing status word at a time, and which of two wins
    assert parse(ok + [1])[0] == 10                               # compact pack: the buffer was too small
    assert parse([0, 0, 0, 0, 0, 0, 1])[0] == 10                  # ... before everything else
    rc = parse([0, B, B, B, B, 3])[0]                             # the input copy never delivered b = 3
    assert rc == 11 and "utterance 3" in lib.ctcx_last_cuda_error().decode()
    assert parse([0, 0, 0, 0, 0, 2])[0] == 11
    rc = parse([0, B, 2, B, B, B])[0]                             # sequence_length(2) > T
    assert rc == 5 and lib.ctcx_error_batch_index() == 2
    assert lib.ctcx_strerror(5).decode() == "sequence_length(2) <= 9"
    rc = parse([0, 0, 4, 0, 0, B])[0]
    assert rc == 5 and lib.ctcx_error_batch_index() == 4
    assert parse([0, B, B, 1, B, B])[0] == 8                      # negative sequence_length
    assert parse([0, 0, B, 1, 0, B])[0] == 8
    rc = parse([0, B, B, B, 3, B])[0]                             # stream fed past its frames
    assert rc == 5 and lib.ctcx_error_batch_index() == 3
    rc = parse([0, 0, B, B, 1, B])[0]
    assert rc == 5 and lib.ctcx_error_batch_index() == 1
    rc, got, f = parse([1, 0, B, B, B, B])                        # too few leaves
    assert rc == 7 and got == [[-7] * 3] * 4 and f == -7
    # argument errors
    blk = _result_block(P, sz, ok)
    s = _lib.CtcxSizes()
    assert lib.ctcx_result_parse(None, T, B, P, ctypes.byref(s), None) == 8
    assert lib.ctcx_result_parse(blk.ctypes.data, T, B, P, None, None) == 8
    assert lib.ctcx_result_parse(blk.ctypes.data, 0, B, P, ctypes.byref(s), None) == 8
    assert lib.ctcx_result_parse(blk.ctypes.data, T, -1, P, ctypes.byref(s), None) == 8
    assert lib.ctcx_result_parse(blk.ctypes.data, T, B, 0, ctypes.byref(s), None) == 8
    assert lib.ctcx_result_parse(blk.ctypes.data, T, 0, P, ctypes.byref(s), None) == 0  # empty batch


def test_python_host_validation_order():
    import ctc_beam_search_op_b200 as op
    x = np.zeros((4, 2, 3), np.float32)
    with pytest.raises(ValueError, match="beam_width"):
        op.ctc_ext_beam_search_decoder(x, [4, 4], beam_width=0, top_paths=1)
    with pytest.raises(ValueError, match="top_paths"):
        op.ctc_ext_beam_search_decoder(x, [4, 4], beam_width=1, top_paths=0)
    with pytest.raises(op.InvalidArgumentError, match="inputs is not a 3-Tensor"):
        op.ctc_ext_beam_search_decoder(x[0], [4, 4], beam_width=2, top_paths=1)
    with pytest.raises(op.InvalidArgumentError, match="max_time is 0"):
        op.ctc_ext_beam_search_decoder(x[:0], [4, 4], beam_width=2, top_paths=1)
    with pytest.raises(op.InvalidArgumentError, match="sequence_length is not a vector"):
        op.ctc_ext_beam_search_decoder(x, [[4, 4]], beam_width=2, top_paths=1)
    with pytest.raises(op.FailedPreconditionError, match=r"len\(sequence_length\) != batch_size"):
        op.ctc_ext_beam_search_decoder(x, [4], beam_width=2, top_paths=1)
    with pytest.raises(TypeError):
        op.ctc_ext_beam_search_decoder(x.astype(np.int32), [4, 4], beam_width=2, top_paths=1)


def test_no_cpu_fallback():
    """Without a CUDA device the op must raise, not compute on the CPU."""
    import torch
    import ctc_beam_search_op_b200 as op
    if torch.cuda.is_available():
        pytest.skip("a CUDA device is present")
    with pytest.raises(RuntimeError, match="no CPU fallback"):
        op.ctc_ext_beam_search_decoder(np.zeros((4, 2, 3), np.float32), [4, 4], beam_width=2, top_paths=1)


def test_product_never_imports_the_oracle():
    """The oracle is test infrastructure: nothing in the product package may import, include, link
    or dlopen anything under oracle/ (a product path that routes through it would void parity)."""
    pkg = os.path.join(ROOT, "ctc-beam-search-op_b200")
    loaders = ("import", "#include", "CDLL", "dlopen", "load_library", "subprocess", "open(")
    for dirpath, _, files in os.walk(pkg):
        for f in files:
            if not f.endswith((".py", ".cu", ".cuh", ".h")):
                continue
            for ln in open(os.path.join(dirpath, f)).read().splitlines():
                if "oracle" in ln.lower():
                    assert not any(k in ln for k in loaders), "%s: %s" % (f, ln.strip())


def test_shard_bounds_and_merge():
    import ctc_beam_search_op_b200 as op
    assert op.shard_bounds(10, 4) == [(0, 3), (3, 6), (6, 8), (8, 10)]
    assert op.shard_bounds(2, 4) == [(0, 1), (1, 2), (2, 2), (2, 2)]
    x = L.make_logits("peaky", 20, 7, 6, 5, 3)
    sl = L.ragged_lengths(20, 7, 3)
    whole = L.pack_sparse(L.oracle_decode(x, sl, 4, 2, True, 5, -1))
    bounds = op.shard_bounds(7, 3)
    shards = [L.pack_sparse(L.oracle_decode(x[:, b0:b1], sl[b0:b1], 4, 2, True, 5, -1)) for b0, b1 in bounds]
    merged = op.merge_raw(shards, bounds, 7)
    for g in range(6):
        for p in range(2):
            np.testing.assert_array_equal(merged[g][p], whole[g][p])
    np.testing.assert_array_equal(merged[6], whole[6])


def test_torch_library_registration_traces_with_fake_tensors():
    """torch.ops.ctcx.ctc_ext_beam_search_decoder exists, has the reference op's argument order
    (ops.cc:10-16) and infers its output shapes without a device (ops.cc:41-61: data-dependent
    numbers of sparse entries, [batch, top_paths] log-probabilities)."""
    import torch
    from torch._subclasses.fake_tensor import FakeTensorMode
    from torch.fx.experimental.symbolic_shapes import ShapeEnv
    import ctc_beam_search_op_b200 as m  # noqa: F401
    op = torch.ops.ctcx.ctc_ext_beam_search_decoder
    schema = str(op.default._schema)
    for a in ("Tensor inputs", "Tensor sequence_length", "Int beam_width", "Int top_paths",
              "bool merge_repeated=False", "Int blank_index=0", "Int blank_label=-1"):
        assert a in schema, schema
    with FakeTensorMode(shape_env=ShapeEnv()):
        for dt in (torch.float32, torch.float64):
            x = torch.empty((50, 8, 29), device="cuda", dtype=dt)
            sl = torch.empty((8,), dtype=torch.int32, device="cuda")
            out = op(x, sl, 10, 3, True, 28, -1)
            assert len(out) == 19
            assert out[0].shape[1] == 2 and out[0].dtype == torch.int64 and out[6].shape == (2,)
            assert out[18].shape == (8, 3) and out[18].dtype == dt
    # the flat list maps back onto the raw namedtuple
    r = m.torch_op.unflatten(list(range(19)), 3)
    assert r.decoded_indices == [0, 1, 2] and r.alignment_shape == [15, 16, 17] and r.log_probability == 18


def test_error_classes_survive_pickling():
    """decode_distributed ships a rank's exception to the gathering rank: code and text must survive."""
    import pickle
    import ctc_beam_search_op_b200 as m
    for cls, code in ((m.InvalidArgumentError, 6), (m.FailedPreconditionError, 5), (m.UnsupportedError, 9)):
        e = pickle.loads(pickle.dumps(cls(code, "sequence_length(3) <= 8")))
        assert type(e) is cls and e.code == code and str(e) == "sequence_length(3) <= 8"


def test_packed_output_buffer_layout():
    """All 6*P sparse tensors + log_probability are views of ONE int64 buffer (one D2H copy for host
    callers): the carve-up must be gap-free, non-overlapping and typed as ops.cc:17-23 says."""
    import torch
    from ctc_beam_search_op_b200 import decoder as D
    for f64 in (False, True):
        B, P = 5, 3
        counts = ([7, 0, 12], [40, 40, 33])
        n = D._pack_elems(B, P, counts, f64)
        buf = torch.arange(n, dtype=torch.int64)
        groups, lp = D._carve(buf, B, P, counts, f64)
        seen = torch.zeros(n, dtype=torch.int32)
        for g in range(6):
            for p in range(P):
                t = groups[g][p]
                nd = counts[0][p] if g < 3 else counts[1][p]
                want = {0: (nd, 2), 1: (nd,), 2: (2,)}[g % 3]
                assert tuple(t.shape) == want and t.dtype == torch.int64 and t.is_contiguous()
                if t.numel():
                    seen[t.reshape(-1)] += 1  # values are the buffer offsets themselves
        assert lp.shape == (B, P) and lp.dtype == (torch.float64 if f64 else torch.float32)
        lp_words = B * P if f64 else (B * P + 1) // 2
        assert int(seen.sum()) == n - lp_words and int(seen.max()) == 1
        assert lp.data_ptr() == buf.data_ptr() + 8 * (n - lp_words)
