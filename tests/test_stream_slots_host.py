"""CPU checks of the streaming decoder's per-slot entries: the argument validation of
ctcx_stream_reset_slots / ctcx_stream_top_paths_slots (before any CUDA call), and the Python stream's
checks of a slot selection."""
import ctypes

import numpy as np
import pytest

F32, F16, BF16, F64 = 0, 1, 2, 3


@pytest.fixture(scope="module")
def lib():
    from ctc_beam_search_op_b200 import _lib
    return _lib.load()


def _aligned(buf):
    """A 256-byte aligned address inside a host buffer: passes the alignment check, never dereferenced."""
    return (ctypes.addressof(buf) + 255) // 256 * 256


def test_reset_slots_validation_without_device(lib):
    """The checks of ctcx_stream_reset_v in the same order, then the mask."""
    buf = ctypes.create_string_buffer(4096)
    ws, fake = _aligned(buf), _aligned(buf) + 256   # (fake: a non-null device pointer, never read)
    T, B, C, W, P = 5, 2, 3, 2, 1
    n32 = lib.ctcx_stream_workspace_bytes_v(F32, T, B, C, W, P)
    n64 = lib.ctcx_stream_workspace_bytes_v(F64, T, B, C, W, P)

    def reset(w, nb, sd=F32, T=T, B=B, C=C, W=W, P=P, mask=fake):
        return lib.ctcx_stream_reset_slots(w, nb, sd, T, B, C, W, P, mask, None)

    assert reset(ws, n32, sd=F16) == 8               # a chunk type, not a score type
    assert reset(ws, n32, sd=7) == 8
    assert reset(ws, n32, T=0) == 8
    assert reset(ws, n32, B=-1) == 8
    assert reset(ws, n32, C=0) == 8
    assert reset(ws, n32, W=0) == 8
    assert reset(ws, n32, P=0) == 8
    assert reset(ws, n32, W=1025) == 9
    assert reset(ws, n32, C=65536) == 9
    assert reset(ws, n32, P=3) == 6                  # top_paths > beam_width, before the workspace
    assert reset(None, n32) == 10
    assert reset(ws + 8, n32) == 10                  # misaligned
    assert reset(ws, n32 - 1) == 10                  # short
    assert reset(ws, n32, sd=F64) == 10              # a float stream's workspace for a float64 reset
    assert reset(ws, n64 - 1, sd=F64) == 10
    assert reset(ws, n32, mask=None) == 8            # no mask, after the workspace checks
    assert reset(ws, n64, sd=F64, mask=None) == 8
    # sized right, empty batch: nothing to enqueue
    assert reset(ws, lib.ctcx_stream_workspace_bytes_v(F32, T, 0, C, W, P), B=0) == 0


def test_top_paths_slots_validation_without_device(lib):
    """The checks of ctcx_stream_top_paths (sizes may be NULL: the deferred form), top_paths > beam_width,
    then the mask."""
    buf = ctypes.create_string_buffer(4096)
    ws, fake = _aligned(buf), _aligned(buf) + 256
    T, B, C, W, P = 5, 2, 3, 2, 1
    arr = ctypes.c_int64 * 3
    from ctc_beam_search_op_b200 import _lib
    sizes = _lib.CtcxSizes(arr(), arr(), arr(), arr())

    def top(w, T=T, B=B, C=C, W=W, P=P, mask=fake, sz=None):
        return lib.ctcx_stream_top_paths_slots(w, T, B, C, W, P, 0, -1, mask, None, sz, None)

    for sz in (None, ctypes.byref(sizes)):
        assert top(None, sz=sz) == 10
        assert top(ws + 8, sz=sz) == 10
        assert top(ws, T=0, sz=sz) == 8
        assert top(ws, B=-1, sz=sz) == 8
        assert top(ws, C=0, sz=sz) == 8
        assert top(ws, W=0, sz=sz) == 8
        assert top(ws, P=0, sz=sz) == 8
        assert top(ws, W=1025, sz=sz) == 8
        assert top(ws, C=65536, sz=sz) == 8
        assert top(ws, P=3, sz=sz) == 6              # top_paths > beam_width
        assert top(ws, mask=None, sz=sz) == 8
    # empty batch, synchronous form: nothing to trace, empty sizes
    assert top(ws, B=0, sz=ctypes.byref(sizes)) == 0
    assert list(sizes.n_decoded[:1]) == [0]


def test_python_rejects_bad_selections_before_any_launch():
    """A stream whose construction is skipped (no device here): the selection checks run before
    anything touches one."""
    import torch

    import ctc_beam_search_op_b200 as op
    dec = op.CTCExtBeamSearchDecoderStream.__new__(op.CTCExtBeamSearchDecoderStream)
    dec.B, dec.device = 4, torch.device("cuda", 0)
    for bad in ([4], [-1], [0, 7], [1.0], [True], np.zeros(3, bool), np.zeros(5, np.int32),
                np.zeros(4, np.float32), torch.zeros(4, dtype=torch.float32), np.zeros((1, 4), bool)):
        with pytest.raises(op.InvalidArgumentError) as e:
            dec._selection(bad)
        assert e.value.code == 8
