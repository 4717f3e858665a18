"""Streaming decoder per score type and input: device time of a whole utterance batch fed in chunks
(every step plus top_paths), beside the one-shot decode of the same dtype and table. Usage:
  python tools/stream_dtypes_bench.py [reps]
Workload: T=500, B=256, C=29, W=100, P=1, Gaussian logits (the bench's cfg2 shape); the batches rotate
through more bytes than the 126 MB L2 holds, so every pass reads its logits from HBM. Chunks of 10, 50
and 500 frames; variants float32, bfloat16, float64 and float32 with the bench's random bigram table.
Steps go through step_device() (no allocation per step), timed with CUDA events on the stream from the
first step to the end of top_paths; the median over `reps` passes is printed, with the card's name and
power limit read in the same run."""
import os
import subprocess
import sys

import numpy as np
import torch

sys.path.insert(0, os.path.join(os.path.dirname(os.path.abspath(__file__)), ".."))
import ctc_beam_search_op_b200 as op  # noqa: E402

T, B, C, W, P, BLANK = 500, 256, 29, 100, 1, 28
L2_BYTES = 126 << 20
REPS = int(sys.argv[1]) if len(sys.argv) > 1 else 5


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader", "-i",
                        str(torch.cuda.current_device())], capture_output=True, text=True)
    return q.stdout.strip() or "unknown card"


def timed(fn):
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    fn()
    e1.record()
    e1.synchronize()
    return e0.elapsed_time(e1)


def main():
    dev = torch.device("cuda")
    base = np.random.default_rng(1).standard_normal((T, B, C)).astype(np.float32)
    table = -np.abs(np.random.default_rng(5).standard_normal((C + 1, C))).astype(np.float32)  # bench.py --scorer
    seq = torch.full((B,), T, dtype=torch.int32, device=dev)
    print("card: %s" % card())
    print("T=%d B=%d C=%d W=%d P=%d; ms of device time, median of %d passes" % (T, B, C, W, P, REPS))
    print("%-10s %8s %8s %8s %9s" % ("variant", "chunk10", "chunk50", "chunk500", "one-shot"))
    for name, dt, lm in (("float32", torch.float32, None), ("bfloat16", torch.bfloat16, None),
                         ("float64", torch.float64, None), ("f32+table", torch.float32, table)):
        per = T * B * C * torch.tensor([], dtype=dt).element_size()
        n_rot = L2_BYTES // per + 2
        rng = np.random.default_rng(7)
        xs = [torch.from_numpy(base if r == 0 else np.ascontiguousarray(base[:, rng.permutation(B), :])).to(dt).to(dev)
              for r in range(n_rot)]
        score = torch.float64 if dt == torch.float64 else torch.float32
        dec = op.CTCExtBeamSearchDecoderStream(batch_size=B, num_classes=C, beam_width=W, top_paths=P, max_time=T,
                                               blank_index=BLANK, dtype=score, expansion_scores=lm)
        row = []
        for ct in (10, 50, 500):
            lens = torch.full((B,), ct, dtype=torch.int32, device=dev)
            ms = []
            for i in range(REPS + 1):  # pass 0 warms up
                x = xs[i % n_rot]
                dec.reset()

                def run():
                    for t in range(0, T, ct):
                        dec.step_device(x[t:t + ct], lens)
                    dec.top_paths_raw()
                m = timed(run)
                if i > 0:
                    ms.append(m)
            row.append(float(np.median(ms)))
        one = []
        for i in range(REPS + 1):
            x = xs[i % n_rot]
            m = timed(lambda: op.ctc_ext_beam_search_decoder_raw(x, seq, beam_width=W, top_paths=P, blank_index=BLANK,
                                                                 expansion_scores=lm))
            if i > 0:
                one.append(m)
        row.append(float(np.median(one)))
        print("%-10s %8.2f %8.2f %8.2f %9.2f" % ((name,) + tuple(row)))
        del xs, dec
        torch.cuda.empty_cache()


if __name__ == "__main__":
    main()
