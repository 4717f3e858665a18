"""Per-slot reset and read of the streaming decoder in a continuous-batching serving loop. Usage:
  python tools/stream_slots_bench.py [n_utterances] [reps]
Workload: B=256 slots, C=29, W=100, P=1, float32 scores, Gaussian logits; n_utterances (default 1024)
of ragged length 250-500 frames drawn from a seed, fed in chunks of 10 and 50 frames.
  * continuous: a slot whose utterance ends is read with top_paths(slots, wait=False) and reset in the
    same step, then takes the next utterance; each read is collected LAG steps later (LAG = 1 and 16:
    collecting a read waits for the device to finish it, so LAG = 1 keeps at most one step in flight).
  * batch-synchronous: the same utterances in groups of B, every slot waiting for the group's longest
    utterance, then a full top_paths() and reset().
Both loops gather their chunks from the same device pool with the same indexing and step through
step_device() with lengths copied from page-locked memory, so that no step waits for the device;
utterance-frames/s =
the frames of all utterances over the loop's wall time (host clock, ended by a device synchronise).
Then device ms (CUDA events, median of `reps`) of: ctcx_stream_top_paths_slots with 1, 8 and 256
selected slots against ctcx_stream_top_paths (both synchronous, after every slot consumed 500 frames);
ctcx_stream_reset_slots against ctcx_stream_reset_v; one 10-frame step with 1, 64 and 256 active slots
(the others idle with 0 frames). The card's name and power limit are read in the same run."""
import ctypes
import os
import subprocess
import sys
import time

import numpy as np
import torch

sys.path.insert(0, os.path.join(os.path.dirname(os.path.abspath(__file__)), ".."))
import ctc_beam_search_op_b200 as op  # noqa: E402
from ctc_beam_search_op_b200 import _lib  # noqa: E402

T, B, C, W, P, BLANK = 500, 256, 29, 100, 1, 28
N = int(sys.argv[1]) if len(sys.argv) > 1 else 1024
REPS = int(sys.argv[2]) if len(sys.argv) > 2 else 20


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader", "-i",
                        str(torch.cuda.current_device())], capture_output=True, text=True)
    return q.stdout.strip() or "unknown card"


def device_ms(fn, reps=REPS):
    ms = []
    for i in range(reps + 1):  # call 0 warms up
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        fn()
        e1.record()
        e1.synchronize()
        if i > 0:
            ms.append(e0.elapsed_time(e1))
    return float(np.median(ms))


def new_stream():
    return op.CTCExtBeamSearchDecoderStream(batch_size=B, num_classes=C, beam_width=W, top_paths=P, max_time=T,
                                            merge_repeated=True, blank_index=BLANK)


def dev(a):
    """host array -> device, enqueued behind the work in flight (page-locked source)"""
    return torch.from_numpy(np.ascontiguousarray(a)).pin_memory().cuda(non_blocking=True)


def step(dec, pool, utt, pos, ct, lens):
    """one step of `ct` frames: row i of slot b = frame pos[b] + i of utterance utt[b], lens[b] of them"""
    t = dev(np.minimum(pos[None, :] + np.arange(ct)[:, None], T - 1))
    u = dev(np.broadcast_to(np.maximum(utt, 0)[None, :], (ct, B)))
    dec.step_device(pool[t, u], dev(lens.astype(np.int32)))


def continuous(dec, pool, sl, ct, lag):
    queue = list(range(B, N))
    utt = np.arange(B)
    pos = np.zeros(B, np.int64)
    dec.reset()
    pending, results, k = [], 0, 0
    while (utt >= 0).any():
        active = utt >= 0
        lens = np.where(active, np.minimum(ct, sl[np.maximum(utt, 0)] - pos), 0).astype(np.int32)
        step(dec, pool, utt, pos, ct, lens)
        while pending and pending[0][0] <= k - lag:  # the reads enqueued `lag` steps ago
            results += len(pending.pop(0)[1].result()[2])
        pos += lens
        done = np.flatnonzero(active & (pos == sl[np.maximum(utt, 0)]))
        if len(done):
            sel = np.isin(np.arange(B), done)
            pending.append((k, dec.top_paths(sel, wait=False)))
            dec.reset(sel)
            for b in done:
                utt[b] = queue.pop(0) if queue else -1
                pos[b] = 0
        k += 1
    for _, h in pending:
        results += len(h.result()[2])
    assert results == N


def synchronous(dec, pool, sl, ct):
    for g0 in range(0, N, B):
        utt = np.arange(g0, g0 + B)
        pos = np.zeros(B, np.int64)
        dec.reset()
        while (pos < sl[utt]).any():
            lens = np.minimum(ct, sl[utt] - pos).astype(np.int32)
            step(dec, pool, utt, pos, ct, lens)
            pos += lens
        assert len(dec.top_paths()[2]) == B


def wall(fn):
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    fn()
    torch.cuda.synchronize()
    return time.perf_counter() - t0


def main():
    assert N % B == 0
    print("card: %s" % card())
    sl = np.random.default_rng(1).integers(250, 501, N).astype(np.int64)
    pool = torch.from_numpy(np.random.default_rng(2).standard_normal((T, N, C)).astype(np.float32)).cuda()
    frames = int(sl.sum())
    print("B=%d C=%d W=%d P=%d float32; %d utterances of 250-500 frames (%d utterance-frames)" % (B, C, W, P, N, frames))
    dec = new_stream()
    print("\nserving loop, utterance-frames/s (wall time, one pass after a warm-up pass)")
    print("%-6s %14s %14s %14s %8s %8s" % ("chunk", "cont. lag 1", "cont. lag 16", "batch-sync", "ratio1", "ratio16"))
    for ct in (10, 50):
        continuous(dec, pool, sl, ct, 1)
        continuous(dec, pool, sl, ct, 16)
        synchronous(dec, pool, sl, ct)
        a1 = wall(lambda: continuous(dec, pool, sl, ct, 1))
        a16 = wall(lambda: continuous(dec, pool, sl, ct, 16))
        b = wall(lambda: synchronous(dec, pool, sl, ct))
        print("%-6d %14.0f %14.0f %14.0f %8.2f %8.2f" % (ct, frames / a1, frames / a16, frames / b, b / a1, b / a16))

    lib = _lib.load()
    ws, st = dec._ws.data_ptr(), torch.cuda.current_stream().cuda_stream
    arr = ctypes.c_int64 * P
    sizes = _lib.CtcxSizes(arr(), arr(), arr(), arr())
    flags = ctypes.c_int32(0)
    dec.reset()
    x = pool[:, :B].contiguous()
    for t in range(0, T, 50):
        dec.step_device(x[t:t + 50], torch.full((B,), 50, dtype=torch.int32, device="cuda"))

    def mask(k):
        return torch.from_numpy((np.arange(B) < k).astype(np.int32)).cuda()

    print("\ndevice ms, median of %d calls" % REPS)
    full = device_ms(lambda: lib.ctcx_stream_top_paths(ws, T, B, C, W, P, 1, -1, st, ctypes.byref(sizes),
                                                       ctypes.byref(flags)))
    print("ctcx_stream_top_paths (all %d slots, 500 frames each)   %8.3f" % (B, full))
    for k in (1, 8, 256):
        m = mask(k)
        ms = device_ms(lambda: lib.ctcx_stream_top_paths_slots(ws, T, B, C, W, P, 1, -1, m.data_ptr(), st,
                                                               ctypes.byref(sizes), ctypes.byref(flags)))
        print("ctcx_stream_top_paths_slots, %3d selected               %8.3f" % (k, ms))
    for k in (1, 256):
        m = mask(k)
        ms = device_ms(lambda: lib.ctcx_stream_reset_slots(ws, dec._nbytes, _lib.F32, T, B, C, W, P, m.data_ptr(), st))
        print("ctcx_stream_reset_slots, %3d selected                   %8.3f" % (k, ms))
    print("ctcx_stream_reset_v (full reset)                        %8.3f" % device_ms(dec.reset))
    xs = x[:10]
    for k in (1, 64, 256):
        lens = torch.from_numpy(np.where(np.arange(B) < k, 10, 0).astype(np.int32)).cuda()
        m = mask(B)

        def steps():
            dec.reset(m)  # (outside the timed window below: the budget of 500 frames starts again)
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            for _ in range(40):
                dec.step_device(xs, lens)
            e1.record()
            e1.synchronize()
            return e0.elapsed_time(e1) / 40
        ms = float(np.median([steps() for _ in range(REPS + 1)][1:]))
        print("10-frame step, %3d active slots (the rest idle)         %8.3f" % (k, ms))


if __name__ == "__main__":
    main()
