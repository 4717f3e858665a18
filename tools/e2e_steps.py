import os, sys, time
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT); sys.path.insert(0, os.path.join(ROOT, "tests"))
import numpy as np, torch
import ctcx_testlib as L
import ctc_beam_search_op_b200 as op
T, B, C, W = 500, 256, 29, 100
kw = dict(beam_width=W, top_paths=1, merge_repeated=True, blank_index=28, blank_label=-1)
xs = [torch.from_numpy(L.make_logits("gauss", T, B, C, 28, s)).pin_memory() for s in range(10)]
sl = torch.full((B,), T, dtype=torch.int32).pin_memory()
xd = [x.cuda() for x in xs]; sd = sl.cuda()
for i in range(6): op.ctc_ext_beam_search_decoder_raw(xd[i], sd, **kw)
torch.cuda.synchronize()
ts = []
for i in range(25):
    t0 = time.perf_counter(); op.ctc_ext_beam_search_decoder_raw(xs[i % 10], sl, **kw); torch.cuda.synchronize(); ts.append((time.perf_counter() - t0) * 1e3)
print(" ".join("%.2f" % t for t in ts))
