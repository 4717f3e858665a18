"""What the narrow kernel's revisit-wipe fixed point (PC) has to do, from the CPU model, no GPU:
python tools/pc_model_report.py [B]

For bench.py's cfg2 (T=500, C=29, beam 100) Gaussian and peaky logits (seed 1) and the golden
revisit-wipe cases: per frame with at-risk members, how many there are, how many are contested (round-1
count >= W: the only ones later rounds touch), how many lie above lp_max + the old best total (never
listed by PA), the round-1 count distribution and the fixed-point rounds. tools/pc_model_report.cc is
compiled with g++ into a temporary directory on first use."""
import ctypes
import os
import subprocess
import sys
import tempfile

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, os.path.join(ROOT, "tests"))
import numpy as np

SRC = os.path.join(ROOT, "tools", "pc_model_report.cc")
_lib = None


def load():
    global _lib
    if _lib is None:
        so = os.path.join(tempfile.mkdtemp(prefix="ctcx_pc_report_"), "libctcx_pc_report.so")
        subprocess.check_call(["g++", "-O2", "-std=c++11", "-ffp-contract=off", "-fPIC", "-shared", "-o", so, SRC])
        _lib = ctypes.CDLL(so)
    return _lib


def report(x, sl, W, blank):
    """out[11]: frames with at-risk members, at-risk members, contested members, members above the bound,
    round-1 count / W in quarters (5 bins), fixed-point rounds over the frames with at-risk members, their max."""
    x = np.ascontiguousarray(x, np.float32)
    T, B, C = x.shape
    out = np.zeros(11, np.int64)
    sl = np.ascontiguousarray(sl, np.int32)
    rc = load().ctcx_pc_report_f32(ctypes.c_void_p(x.ctypes.data), T, B, C, ctypes.c_void_p(sl.ctypes.data), W,
                                   blank, ctypes.c_void_p(out.ctypes.data))
    assert rc == 0, rc
    return out


def show(name, o):
    f, r = max(o[0], 1), max(o[1], 1)
    q = o[4:9] / r
    print("%-16s frames with risk %6d | per such frame: at-risk %.2f, contested %.2f (%.1f %%), above the "
          "bound %.2f (%.1f %%) | round-1 count/W  <.25 %.2f  <.5 %.2f  <.75 %.2f  <1 %.2f  >=1 %.2f | "
          "rounds %.2f (max %d)" % (name, o[0], o[1] / f, o[2] / f, 100.0 * o[2] / r, o[3] / f, 100.0 * o[3] / r,
                                    *q, o[9] / f, o[10]))


def main():
    import ctcx_testlib as L
    B = int(sys.argv[1]) if len(sys.argv) > 1 else 32
    T, C, W, BLANK = 500, 29, 100, 28
    for kind in ("gauss", "peaky"):
        show("cfg2 %s" % kind, report(L.make_logits(kind, T, B, C, BLANK, 1), np.full(B, T, np.int32), W, BLANK))
    tot = np.zeros(11, np.int64)
    for c in L.wipe_cases():
        o = report(c.x, c.sl, c.W, c.blank)
        tot[:10] += o[:10]
        tot[10] = max(tot[10], o[10])
    show("wipe_cases.npz", tot)


if __name__ == "__main__":
    main()
