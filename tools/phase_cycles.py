"""Per-phase latency (clock64, thread 0 of each CTA) of the fast beam kernels:
python tools/phase_cycles.py [B] [kind] [cfg2|cfg4] [bf16|scorer]"""
import os
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))
import numpy as np
import torch

import ctcx_testlib as L
import ctc_beam_search_op_b200 as op
from ctc_beam_search_op_b200 import _lib

B = int(sys.argv[1]) if len(sys.argv) > 1 else 148
kind = sys.argv[2] if len(sys.argv) > 2 else "gauss"
cfg = sys.argv[3] if len(sys.argv) > 3 else "cfg2"
T, C, W, BLANK, MERGE = (500, 29, 100, 28, True) if cfg == "cfg2" else (400, 1024, 16, 1023, False)
lib = _lib.load()
x = torch.from_numpy(L.make_logits(kind, T, B, C, BLANK, 1)).cuda()
if len(sys.argv) > 4 and sys.argv[4] == "bf16":  # bfloat16-rounded values (many exact ties), float32 kernel
    x = x.bfloat16().float()
sl = torch.full((B,), T, dtype=torch.int32).cuda()
NS = 27  # the narrow kernel also fills its revisit-wipe event counters 24-26
buf = torch.zeros((B, NS), dtype=torch.int64, device="cuda")
kw = dict(beam_width=W, top_paths=1, merge_repeated=MERGE, blank_index=BLANK)
if len(sys.argv) > 4 and sys.argv[4] == "scorer":  # the bench's random label-bigram table
    kw["expansion_scores"] = torch.from_numpy(
        -np.abs(np.random.default_rng(5).standard_normal((C + 1, C))).astype(np.float32)).cuda()
op.ctc_ext_beam_search_decoder_raw(x, sl, **kw)
import ctypes
lib.ctcx_profile_enable(1)
ms = (ctypes.c_float * 5)()
op.ctc_ext_beam_search_decoder_raw(x, sl, **kw)
lib.ctcx_profile_get(ms)
prod_ms = ms[1]
lib.ctcx_debug_set_cycles_buffer_n(buf.data_ptr(), NS)
op.ctc_ext_beam_search_decoder_raw(x, sl, **kw)
torch.cuda.synchronize()
lib.ctcx_profile_get(ms)
lib.ctcx_debug_set_cycles_buffer(None)
print("beam kernel: production build %.3f ms, timing build %.3f ms" % (prod_ms, ms[1]))
c = buf.cpu().numpy().astype(np.float64) / T
names = ["PA(end)", "PB(end)", "PC", "PD", "PE", "PF", "PG(end)", "setup", "PA.lookup", "PA.lse1", "PA.lse2",
         "PA.store", "PA.minmax", "PG.rank", "PG.barrier", "PG.write", "PB.range", "PB.pass1", "PB.scan",
         "PB.pass2+bar"] + (["ev.n_risk", "ev.risk_below_cut", "ev.wiped", "ev.frames_with_risk", "ev.listed",
                                  "ev.contested", "ev.fp_rounds"] if cfg == "cfg2"
                                 else ["ev.slowcut", "ev.fullrange", "ev.capped", "ev.ncand"])
m = c.mean(axis=0)
tot = c[:, :20].sum(axis=1)
print("per-CTA total cycles/frame: min %.0f mean %.0f max %.0f (the kernel ends with the slowest CTA)" % (tot.min(), tot.mean(), tot.max()))
worst = int(tot.argmax())
print("slowest CTA %d: " % worst + "  ".join("%s %.0f" % (n, v) for n, v in zip(names[:20], c[worst][:20])))
print("B=%d %s: cycles per frame, thread 0 (mean over CTAs):" % (B, kind))
print("  " + "  ".join(("%s %.3f" if n.startswith("ev.") else "%s %.0f") % (n, v) for n, v in zip(names, m)) + "  | total %.0f" % m[:20].sum())
