"""What each C-ABI entry enqueues: one small call of every entry and route under torch.profiler (CUDA
activities), printed per call as the ordered kernels (normalised names, grid, block, shared memory),
memcpys (kind, bytes) and memsets (bytes), stream by stream, with the call's return code. Two builds of
the library that should enqueue the same work print the same text:

    python tools/api_op_trace.py [--lib path/to/libctcx.so] > ops.txt

Each call runs once untraced first, so that module loading and first-launch set-up stay out of the trace.
"""
import argparse
import ctypes
import json
import os
import re
import sys
import tempfile
from collections import OrderedDict

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

import numpy as np  # noqa: E402
import torch  # noqa: E402

F32, F16, BF16, F64 = 0, 1, 2, 3
TORCH_DT = {F32: torch.float32, F16: torch.float16, F64: torch.float64, BF16: torch.bfloat16}
# (T, B, C, W, P, blank): one shape per beam kernel
SHAPES = OrderedDict(narrow=(40, 6, 29, 10, 2, 28), wide=(40, 4, 100, 8, 2, 99), generic=(12, 3, 3000, 8, 2, 2999))


def norm_kernel(name):
    name = name.replace("(anonymous namespace)", "anon")
    name = re.sub(r"\(.*\)$", "", name)  # the parameter list
    return re.sub(r"^void ", "", name)


def gpu_ops(prof):
    """[(stream, ts, text)] of the kernels, memcpys and memsets of one profiled call."""
    with tempfile.TemporaryDirectory() as d:
        path = os.path.join(d, "trace.json")
        prof.export_chrome_trace(path)
        with open(path) as fh:
            events = json.load(fh)["traceEvents"]
    ops = []
    for e in events:
        cat, a = e.get("cat", ""), e.get("args", {})
        if cat == "kernel":
            text = "kernel %s grid %s block %s smem %s" % (norm_kernel(e["name"]), a.get("grid"), a.get("block"),
                                                         a.get("shared memory"))
        elif cat == "gpu_memcpy":
            text = "%s %d B" % (e["name"], a.get("bytes", -1))
        elif cat == "gpu_memset":
            text = "%s %d B" % (e["name"], a.get("bytes", -1))
        else:
            continue
        ops.append((a.get("stream", -1), float(e["ts"]), text))
    return ops


def trace(label, fn, out):
    torch.cuda.synchronize()  # inputs made on other streams are in place
    fn()  # untraced first run
    torch.cuda.synchronize()
    acts = [torch.profiler.ProfilerActivity.CPU, torch.profiler.ProfilerActivity.CUDA]
    with torch.profiler.profile(activities=acts) as prof:
        rc = fn()
        torch.cuda.synchronize()
    ops = gpu_ops(prof)
    # streams named by the order of their first operation, operations in device order on each
    first = OrderedDict()
    for s, ts, _ in sorted(ops, key=lambda o: o[1]):
        first.setdefault(s, "s%d" % len(first))
    out.write("== %s: rc=%s\n" % (label, rc))
    for s, ts, text in sorted(ops, key=lambda o: (first[o[0]], o[1])):
        out.write("  %s %s\n" % (first[s], text))
    out.flush()


class Api:
    def __init__(self, lib_path):
        from ctc_beam_search_op_b200 import _lib
        self.m = _lib
        if lib_path:  # another build: the same bindings on a different library file
            saved = _lib._build.LIB_PATH, _lib._build.is_stale
            _lib._build.LIB_PATH, _lib._build.is_stale = os.path.abspath(lib_path), lambda: False
            try:
                self.lib = _lib.load()
            finally:
                _lib._build.LIB_PATH, _lib._build.is_stale = saved
        else:
            self.lib = _lib.load()
        self.stream = torch.cuda.Stream()
        self.copy_stream = torch.cuda.Stream()

    def sizes(self, P):
        arrs = [np.zeros(P, np.int64) for _ in range(4)]
        s = self.m.CtcxSizes(*[a.ctypes.data_as(self.m._i64p) for a in arrs])
        s._keep = arrs
        return s


def logits(T, B, C, dt, seed=0):
    g = torch.Generator(device="cuda").manual_seed(seed)
    return (torch.randn(T, B, C, device="cuda", generator=g, dtype=torch.float64) * 3).to(TORCH_DT[dt])


def main():
    ap = argparse.ArgumentParser(description=__doc__.split("\n")[0])
    ap.add_argument("--lib", help="library to trace (default: the in-tree build)")
    args = ap.parse_args()
    api = Api(args.lib)
    lib, st, cs = api.lib, api.stream.cuda_stream, api.copy_stream.cuda_stream
    out = sys.stdout
    keep = []
    flags = ctypes.c_int32()

    def ws_for(T, B, C, W, P):
        n = lib.ctcx_workspace_bytes(T, B, C, W, P)
        w = torch.empty(n, dtype=torch.uint8, device="cuda")
        keep.append(w)
        return w, n

    for path, (T, B, C, W, P, blank) in SHAPES.items():
        seq = torch.full((B,), T, dtype=torch.int32, device="cuda")
        seq[0] = T - 3
        ws, nws = ws_for(T, B, C, W, P)
        sz = api.sizes(P)
        for dt in (F32, F16, BF16, F64):
            x = logits(T, B, C, dt)
            keep.append(x)
            trace("%s dtype=%d decode_view" % (path, dt), lambda x=x, dt=dt: lib.ctcx_decode_view(
                x.data_ptr(), dt, 0, T, B, C, seq.data_ptr(), W, P, 0, blank, -1, ws.data_ptr(), nws, st,
                ctypes.byref(sz), ctypes.byref(flags)), out)
        x32 = logits(T, B, C, F32)
        xs = torch.empty(T, B + 2, C, device="cuda")
        xs[:, 1:B + 1] = x32
        trace("%s f32 decode_view of a batch shard" % path, lambda: lib.ctcx_decode_view(
            xs[:, 1].data_ptr(), F32, (B + 2) * C, T, B, C, seq.data_ptr(), W, P, 1, blank, -1, ws.data_ptr(), nws,
            st, ctypes.byref(sz), ctypes.byref(flags)), out)
        trace("%s f32 decode_f32 + pack_f32" % path, lambda: run_pack(lib, api, x32, seq, T, B, C, W, P, blank, ws,
                                                                     nws, st, keep), out)
        if path != "wide":  # (a scorer table takes the narrow or the generic kernel)
            scores = -torch.rand((C + 1) * C, device="cuda")
            keep.append(scores)
            trace("%s scorer" % path, lambda scores=scores: lib.ctcx_decode_scorer_f32(
                x32.data_ptr(), T, B, C, seq.data_ptr(), W, P, 0, blank, -1, scores.data_ptr(), ws.data_ptr(), nws,
                st, ctypes.byref(sz), ctypes.byref(flags)), out)
        lib.ctcx_debug_set_beam_impl(1)
        for dt in (F32, F16):
            x = logits(T, B, C, dt, seed=1)
            keep.append(x)
            trace("%s dtype=%d forced generic" % (path, dt), lambda x=x, dt=dt: lib.ctcx_decode_view(
                x.data_ptr(), dt, 0, T, B, C, seq.data_ptr(), W, P, 0, blank, -1, ws.data_ptr(), nws, st,
                ctypes.byref(sz), ctypes.byref(flags)), out)
        lib.ctcx_debug_set_beam_impl(0)
        # the deferred route (ctcx_finish) and the two-phase route (copy, event, parse)
        trace("%s deferred + finish" % path, lambda: lib.ctcx_decode_f32(
            x32.data_ptr(), T, B, C, seq.data_ptr(), W, P, 0, blank, -1, ws.data_ptr(), nws, st, None, None) or
            lib.ctcx_finish(ws.data_ptr(), T, B, P, st, ctypes.byref(sz), ctypes.byref(flags)), out)
        host = torch.empty(lib.ctcx_result_bytes(P), dtype=torch.uint8).pin_memory()
        packed = torch.empty(1 << 16, dtype=torch.int64, device="cuda")
        keep += [host, packed]

        def two_phase():
            rc = lib.ctcx_decode_f32(x32.data_ptr(), T, B, C, seq.data_ptr(), W, P, 0, blank, -1, ws.data_ptr(), nws,
                                     st, None, None)
            rc = rc or lib.ctcx_pack_compact(ws.data_ptr(), T, B, P, 4, packed.data_ptr(), packed.numel(), st)
            rc = rc or lib.ctcx_result_copy_async(ws.data_ptr(), T, B, P, host.data_ptr(), host.numel(), st)
            api.stream.synchronize()
            return rc or lib.ctcx_result_parse(host.data_ptr(), T, B, P, ctypes.byref(sz), ctypes.byref(flags))
        trace("%s two-phase + pack_compact" % path, two_phase, out)
        # host input: page-locked and pageable
        hx = x32.cpu()
        staging = torch.empty(lib.ctcx_hostin_staging_bytes(F32, T, B, C) + 8, dtype=torch.uint8, device="cuda")
        hseq = seq.cpu().numpy()
        keep += [staging, hseq]
        if path != "generic":
            for kind, h in (("pinned", hx.pin_memory()), ("pageable", hx.numpy().copy())):
                keep.append(h)
                ptr = h.data_ptr() if kind == "pinned" else h.ctypes.data
                trace("%s f32 decode_hostin %s" % (path, kind), lambda ptr=ptr: lib.ctcx_decode_hostin(
                    ptr, F32, 0, T, B, C, hseq.ctypes.data, W, P, 0, blank, -1, staging.data_ptr(), staging.numel(),
                    ws.data_ptr(), nws, st, cs, ctypes.byref(sz), ctypes.byref(flags)), out)
        # streaming: reset, two chunks, top paths (room for 2T frames: every step runs twice)
        chunk, Ts = T // 2, 2 * T
        clen = torch.full((B,), chunk, dtype=torch.int32, device="cuda")
        sws, nsws = ws_for(Ts, B, C, W, P)
        keep.append(clen)
        trace("%s stream_reset" % path, lambda: lib.ctcx_stream_reset(sws.data_ptr(), nsws, Ts, B, C, W, P, st), out)
        for k in range(2):
            trace("%s stream_step %d" % (path, k), lambda k=k: lib.ctcx_stream_step_f32(
                sws.data_ptr(), Ts, B, C, W, P, x32[k * chunk].data_ptr(), chunk, clen.data_ptr(), blank, st), out)
        trace("%s stream_top_paths" % path, lambda: lib.ctcx_stream_top_paths(
            sws.data_ptr(), Ts, B, C, W, P, 0, -1, st, ctypes.byref(sz), ctypes.byref(flags)), out)

    # the pre-pass hook, both routes
    T, B, C, W, blank = 3, 4, 100, 8, 0
    ks = ctypes.c_int()
    Ks = (min(C - 1, 2 * W + 3) + 7) // 8 * 8
    pl = torch.empty(T * B * Ks, device="cuda")
    cls = torch.empty(T * B * Ks, dtype=torch.int16, device="cuda")
    for dt in (F32, F16, BF16, F64):
        x = logits(T, B, C, dt, seed=2)
        off = torch.empty(T * B, dtype=torch.float64 if dt == F64 else torch.float32, device="cuda")
        keep += [x, off]
        for route in (0, 1):
            trace("debug_prepass route=%d dtype=%d" % (route, dt), lambda x=x, dt=dt, off=off, route=route:
                  lib.ctcx_debug_prepass(route, x.data_ptr(), dt, T, B, C, 0, blank, W, off.data_ptr(), pl.data_ptr(),
                                         cls.data_ptr(), ctypes.byref(ks), st), out)

    # the host-in, host-out convenience entry
    T, B, C, W, P, blank = SHAPES["narrow"]
    hx = logits(T, B, C, F32).cpu().numpy()
    hseq = np.full(B, T, np.int32)
    res = ctypes.POINTER(api.m.CtcxHostResult)()

    def host_call():
        rc = lib.ctcx_decode_host_f32(hx.ctypes.data, T, B, C, hseq.ctypes.data, W, P, 0, blank, -1,
                                      torch.cuda.current_device(), ctypes.byref(res))
        if rc == 0:
            lib.ctcx_free_host(res)
        return rc
    trace("decode_host_f32", host_call, out)


def run_pack(lib, api, x, seq, T, B, C, W, P, blank, ws, nws, st, keep):
    sz = api.sizes(P)
    rc = lib.ctcx_decode_f32(x.data_ptr(), T, B, C, seq.data_ptr(), W, P, 0, blank, -1, ws.data_ptr(), nws, st,
                             ctypes.byref(sz), None)
    if rc:
        return rc
    n_dec, n_ali = sz._keep[0], sz._keep[2]
    outs = []
    for p in range(P):
        outs.append([torch.empty(int(n), dtype=torch.int64, device="cuda")
                     for n in (n_dec[p] * 2, n_dec[p], 2, n_ali[p] * 2, n_ali[p], 2)])
    logp = torch.empty(B, P, device="cuda")
    keep += [outs, logp]
    ptrs = [(ctypes.c_void_p * P)(*[outs[p][g].data_ptr() for p in range(P)]) for g in range(6)]
    return lib.ctcx_pack_f32(ws.data_ptr(), T, B, P, *ptrs, logp.data_ptr(), st)


if __name__ == "__main__":
    main()
