"""Decodes from several host threads at once. Each kernel instantiation raises its dynamic shared-memory
limit once per device, to the most any shape reaching it requests, so a launch never depends on what
another thread set the (process-wide) limit to. Here the threads of one group run the same kernel
instantiations with different dynamic shared memory:

* narrow kernel, 128-slot tier, beam 64 and 128 (C = 29); the trace-back's warp kernel with them
  (beam 64: 32 KB, beam 128: 64 KB of shared memory);
* wide kernel, 32-slot tier, beam 8 and 24 (C = 100), and its class-selection pre-pass;
* generic kernel, forced, 32-slot tier, beam 16 (C = 29) and 32 (C = 61), and the row normaliser.

Every result must equal, bit for bit, the same decode run alone on the main thread. A fixed, small
workload: it covers concurrent callers, it does not hunt for a race.
"""
import threading

import numpy as np
import pytest

import ctcx_testlib as L

pytestmark = pytest.mark.gpu

THREADS = 4
DECODES_PER_THREAD = 24
T, B, P = 40, 4, 3
# group -> [(beam_width, num_classes)], two shapes per kernel instantiation
GROUPS = {
    "narrow": [(64, 29), (128, 29)],
    "wide": [(8, 100), (24, 100)],
    "generic": [(16, 29), (32, 61)],
}


@pytest.fixture(scope="module")
def op():
    import torch
    if not torch.cuda.is_available():
        pytest.skip("no CUDA device")
    import ctc_beam_search_op_b200 as m
    m.set_beam_impl(None)
    yield m
    m.set_beam_impl(None)


def decode(op, x, sl, W, C):
    raw = op.ctc_ext_beam_search_decoder_raw(x, sl, beam_width=W, top_paths=P, merge_repeated=False,
                                             blank_index=C - 1, blank_label=-1)
    out = []
    for field in raw[:6]:
        out += [t.cpu().numpy() for t in field]
    out.append(raw[6].cpu().numpy().view(np.uint32))
    return out


@pytest.mark.parametrize("group", sorted(GROUPS))
def test_concurrent_decodes_match_a_lone_decode(op, group):
    import torch
    op.set_beam_impl("generic" if group == "generic" else None)
    shapes = GROUPS[group]
    inputs = []
    for i, (W, C) in enumerate(shapes):
        x = torch.from_numpy(L.make_logits("gauss", T, B, C, C - 1, seed=100 + i)).cuda()
        inputs.append((x, torch.full((B,), T, dtype=torch.int32, device="cuda"), W, C))
    alone = [decode(op, *a) for a in inputs]

    results = [[None] * DECODES_PER_THREAD for _ in range(THREADS)]
    errors = []
    start = threading.Barrier(THREADS)

    def worker(k):
        try:
            with torch.cuda.stream(torch.cuda.Stream()):
                start.wait()
                for j in range(DECODES_PER_THREAD):
                    results[k][j] = decode(op, *inputs[(k + j) % len(inputs)])
        except Exception as e:  # reported on the main thread
            errors.append("thread %d: %r" % (k, e))

    threads = [threading.Thread(target=worker, args=(k,)) for k in range(THREADS)]
    for th in threads:
        th.start()
    for th in threads:
        th.join()
    op.set_beam_impl(None)
    assert not errors, errors
    for k in range(THREADS):
        for j in range(DECODES_PER_THREAD):
            want, got = alone[(k + j) % len(inputs)], results[k][j]
            assert len(got) == len(want)
            for a, b in zip(got, want):
                np.testing.assert_array_equal(a, b, err_msg="%s: thread %d, decode %d" % (group, k, j))
