"""The narrow kernel's revisit-wipe event counters against the CPU model, on the golden revisit-wipe
cases (tests/golden/wipe_cases.npz): members PA lists as at risk (those that are not above every child
of every row) and contested members (round-1 count >= W, the only ones later rounds of the fixed point
touch)."""
import os
import sys

import pytest

import ctcx_testlib as L

sys.path.insert(0, os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "tools"))
import pc_model_report  # noqa: E402  (the CPU model's PC report, tools/pc_model_report.cc)

pytestmark = pytest.mark.gpu

NARROW = [c for c in L.wipe_cases() if c.C <= 32 and c.W <= 256]
SLOTS = 27


@pytest.mark.parametrize("c", NARROW, ids=[c.name for c in NARROW])
def test_narrow_listed_and_contested_equal_the_model(c):
    import torch
    if not torch.cuda.is_available():
        pytest.skip("no CUDA device")
    import ctc_beam_search_op_b200 as op
    from ctc_beam_search_op_b200 import _lib
    lib = _lib.load()
    buf = torch.zeros((1, SLOTS), dtype=torch.int64, device="cuda")
    lib.ctcx_debug_set_cycles_buffer_n(buf.data_ptr(), SLOTS)
    try:
        op.ctc_ext_beam_search_decoder_raw(torch.from_numpy(c.x).cuda(), torch.from_numpy(c.sl).cuda(),
                                           beam_width=c.W, top_paths=c.P, merge_repeated=c.merge,
                                           blank_index=c.blank, blank_label=-1)
        torch.cuda.synchronize()
    finally:
        lib.ctcx_debug_set_cycles_buffer(None)
    ev = buf[0].cpu().numpy()
    rep = pc_model_report.report(c.x, c.sl, c.W, c.blank)
    assert ev[20] == c.stats["at_risk"] == rep[1]
    assert (ev[24], ev[25]) == (rep[1] - rep[3], rep[2]), (ev[20:27].tolist(), rep.tolist())
