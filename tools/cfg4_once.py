import os, sys
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT); sys.path.insert(0, os.path.join(ROOT, 'tests'))
import numpy as np, torch
import ctcx_testlib as L
import ctc_beam_search_op_b200 as op
T,B,C,W=400,128,1024,16
x = torch.from_numpy(L.make_logits("gauss", T, B, C, 1023, 3)).cuda()
sl = torch.full((B,), T, dtype=torch.int32).cuda()
for _ in range(2):
    op.ctc_ext_beam_search_decoder_raw(x, sl, beam_width=W, top_paths=1, blank_index=1023)
torch.cuda.synchronize(); print("ok")
