"""CPU checks of the streaming decoder's score types, scorer table and strided chunks: the argument
validation of ctcx_stream_workspace_bytes_v / ctcx_stream_reset_v / ctcx_stream_step_v (before any CUDA
call), their workspace sizes, and the Python stream's checks at construction."""
import ctypes

import numpy as np
import pytest

from test_host import WORKSPACE_BYTES

F32, F16, BF16, F64 = 0, 1, 2, 3


@pytest.fixture(scope="module")
def lib():
    from ctc_beam_search_op_b200 import _lib
    return _lib.load()


def test_stream_workspace_bytes_per_score_type(lib):
    """A float32 stream takes exactly the bytes of the un-suffixed entry; a float64 one adds its double
    state blocks (24 + 60 W bytes per utterance, rounded to 16, the region to 256) after them."""
    for shape, want in WORKSPACE_BYTES:
        assert lib.ctcx_stream_workspace_bytes_v(F32, *shape) == want, shape
        T, B, C, W, P = shape
        blocks = -(-B * (-(-(24 + 60 * W) // 16) * 16) // 256) * 256
        assert lib.ctcx_stream_workspace_bytes_v(F64, *shape) == want + blocks, shape
    for sd in (F16, BF16, 4, -1):
        assert lib.ctcx_stream_workspace_bytes_v(sd, 50, 8, 29, 10, 3) == 0
    for bad in ((0, 1, 3, 2, 1), (5, -1, 3, 2, 1), (5, 1, 0, 2, 1), (5, 1, 3, 0, 1), (5, 1, 3, 2, 0)):
        assert lib.ctcx_stream_workspace_bytes_v(F64, *bad) == 0


def _aligned(buf):
    """A 256-byte aligned address inside a host buffer: passes the alignment check, never dereferenced."""
    return (ctypes.addressof(buf) + 255) // 256 * 256


def test_stream_v_validation_without_device(lib):
    """Argument errors of the new entries, before any CUDA call (same style and order as
    test_host.test_cabi_validation_without_device)."""
    reset = lambda sd, T, B, C, W, P: lib.ctcx_stream_reset_v(None, 0, sd, T, B, C, W, P, None)  # noqa: E731
    assert reset(F16, 5, 1, 3, 2, 1) == 8           # a chunk type, not a score type
    assert reset(7, 5, 1, 3, 2, 1) == 8
    assert reset(F64, 0, 1, 3, 2, 1) == 8
    assert reset(F64, 5, -1, 3, 2, 1) == 8
    assert reset(F64, 5, 1, 3, 2, 0) == 8
    assert reset(F64, 5, 1, 3, 1025, 1) == 9
    assert reset(F64, 5, 1, 65536, 2, 1) == 9
    assert reset(F64, 5, 1, 3, 2, 3) == 6           # top_paths > beam_width, before the workspace
    assert reset(F64, 5, 1, 3, 2, 1) == 10
    assert reset(F32, 5, 0, 3, 2, 1) == 10

    buf = ctypes.create_string_buffer(4096)
    ws, fake = _aligned(buf), _aligned(buf) + 256   # (fake: a non-null device pointer, never read)
    T, B, C, W, P = 5, 2, 3, 2, 1
    f32_bytes = lib.ctcx_stream_workspace_bytes_v(F32, T, B, C, W, P)
    f64_bytes = lib.ctcx_stream_workspace_bytes_v(F64, T, B, C, W, P)
    assert 0 < f32_bytes < f64_bytes

    def step(w, nb, dt, ts, T=T, B=B, C=C, W=W, P=P, Tc=2, lens=fake, blank=0, lm=None):
        return lib.ctcx_stream_step_v(w, nb, T, B, C, W, P, fake, dt, ts, Tc, lens, blank, lm, None)

    # the workspace pointer first (as ctcx_stream_step_f32), then the chunk's type and stride, the shape,
    # and last the workspace size for the chunk's score type
    assert step(None, f64_bytes, 9, 0) == 10
    assert step(ws + 8, f64_bytes, F32, 0) == 10   # misaligned
    assert step(ws, 0, 9, 0) == 8                  # no such dtype
    assert step(ws, 0, -1, 0) == 8
    assert step(ws, 0, F32, -1) == 8               # negative time stride
    assert step(ws, 0, F16, 0, T=0) == 8
    assert step(ws, 0, BF16, 0, W=1025) == 8
    assert step(ws, 0, F64, 0, P=3) == 8           # top_paths > beam_width
    assert step(ws, 0, F32, 0, Tc=6) == 8          # a chunk longer than the stream
    assert step(ws, 0, F32, 0, lens=None) == 8
    assert step(ws, 0, F64, 0, blank=3) == 8
    assert step(ws, 0, F32, 5) == 8                # stride shorter than a frame (B * C = 6)
    assert step(ws, 0, F64, 0, lm=fake) == 8       # scorer tables hold float32 scores
    assert step(ws, 0, F32, 6) == 10               # too small for anything
    assert step(ws, f32_bytes - 1, BF16, 0) == 10
    assert step(ws, f32_bytes, F64, 0) == 10       # a float stream's workspace handed to a float64 step
    assert step(ws, f64_bytes - 1, F64, 0) == 10
    # sized right, empty batch: nothing to enqueue
    assert step(ws, lib.ctcx_stream_workspace_bytes_v(F64, T, 0, C, W, P), F64, 0, B=0) == 0
    assert step(ws, lib.ctcx_stream_workspace_bytes_v(F32, T, 0, C, W, P), F16, 7, B=0) == 0


def test_python_stream_checks_its_table_and_score_type_at_construction():
    """dtype and expansion_scores are validated before anything touches a device (so without one too):
    the one-shot decode's errors for a table with float64 scores, a table of the wrong shape and a
    table with a positive entry."""
    import torch

    import ctc_beam_search_op_b200 as op
    kw = dict(batch_size=2, num_classes=4, beam_width=3, top_paths=1, max_time=8)
    with pytest.raises(TypeError):
        op.CTCExtBeamSearchDecoderStream(dtype=torch.float16, **kw)
    with pytest.raises(TypeError):
        op.CTCExtBeamSearchDecoderStream(dtype=np.int32, **kw)
    with pytest.raises(TypeError):
        op.CTCExtBeamSearchDecoderStream(dtype=np.float64, expansion_scores=np.zeros((5, 4), np.float32), **kw)
    with pytest.raises(TypeError):
        op.CTCExtBeamSearchDecoderStream(dtype=torch.float64, expansion_scores=np.zeros((5, 4), np.float32), **kw)
    with pytest.raises(op.InvalidArgumentError, match="shape"):
        op.CTCExtBeamSearchDecoderStream(expansion_scores=np.zeros((4, 4), np.float32), **kw)
    bad = np.zeros((5, 4), np.float32)
    bad[2, 1] = 0.5
    with pytest.raises(op.InvalidArgumentError):
        op.CTCExtBeamSearchDecoderStream(expansion_scores=bad, **kw)
    bad[2, 1] = np.nan
    with pytest.raises(op.InvalidArgumentError):
        op.CTCExtBeamSearchDecoderStream(expansion_scores=torch.from_numpy(bad), **kw)
