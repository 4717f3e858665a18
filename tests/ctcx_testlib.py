"""Test-side helpers: ctypes bindings to the CPU checkers under oracle/, synthetic input generators
and a restatement of the reference's sparse packing. TEST INFRASTRUCTURE -- the product package never
imports this module nor anything under oracle/.

Reference citations are relative to /root/reference/tensorflow_ctc_ext_beam_search_decoder/.
"""
import ctypes
import os
import subprocess

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
ORACLE_DIR = os.path.join(ROOT, "oracle")
REF_SO = os.path.join(ORACLE_DIR, "_ref", "libctcx_ref.so")
ORACLE_SO = os.path.join(ORACLE_DIR, "libctcx_oracle.so")

_c_int_p = ctypes.POINTER(ctypes.c_int)
_c_float_p = ctypes.POINTER(ctypes.c_float)
_c_double_p = ctypes.POINTER(ctypes.c_double)


class OracleError(Exception):
    """Raised with the reference's Status message (kernels.cc:111-138, decoder.h:237-243)."""


def build_oracles(force=False):
    """Compile oracle/libctcx_oracle.so and (where /root/reference exists) oracle/_ref."""
    if force or not os.path.exists(ORACLE_SO) or os.path.getmtime(ORACLE_SO) < max(
            os.path.getmtime(os.path.join(ORACLE_DIR, f)) for f in ("ctcx_oracle.c", "libm_port_check.c")):
        subprocess.check_call(["make", "-s", "-C", ORACLE_DIR, "oracle"])
    if os.path.isdir("/root/reference/tensorflow_ctc_ext_beam_search_decoder") and (
            force or not os.path.exists(REF_SO)
            or os.path.getmtime(REF_SO) < os.path.getmtime(os.path.join(ORACLE_DIR, "ref_driver.cc"))):
        subprocess.check_call(["make", "-s", "-C", ORACLE_DIR, "ref"])


def have_ref():
    return os.path.exists(REF_SO)


_libs = {}


def _load(path):
    if path not in _libs:
        _libs[path] = ctypes.CDLL(path)
    return _libs[path]


def _ptr(a, typ):
    return a.ctypes.data_as(typ)


def _dense_out(B, P, T, dtype):
    n = max(B * P, 1)
    return (np.zeros(n, np.int32), np.full(n * max(T, 1), -7, np.int32), np.zeros(n, np.int32),
            np.full(n * max(T, 1), -7, np.int32), np.zeros(n, dtype))


class DenseResult:
    """Dense rows per (b, p): decoded labels, alignment, log-prob (float32 or float64)."""

    def __init__(self, B, P, T, dec_len, dec, ali_len, ali, logp):
        self.B, self.P, self.T = B, P, T
        Ts = max(T, 1)
        self.dec_len = dec_len[:B * P].reshape(B, P)
        self.ali_len = ali_len[:B * P].reshape(B, P)
        self.dec = dec[:B * P * Ts].reshape(B, P, Ts)
        self.ali = ali[:B * P * Ts].reshape(B, P, Ts)
        self.logp = logp[:B * P].reshape(B, P)

    def decoded(self, b, p):
        return self.dec[b, p, :self.dec_len[b, p]].tolist()

    def alignment(self, b, p):
        return self.ali[b, p, :self.ali_len[b, p]].tolist()


def _check_inputs(logits, seq_len):
    logits = np.ascontiguousarray(logits)
    if logits.ndim != 3:
        raise OracleError("inputs is not a 3-Tensor")  # kernels.cc:111-113
    seq_len = np.ascontiguousarray(seq_len, dtype=np.int32)
    if seq_len.ndim != 1:
        raise OracleError("sequence_length is not a vector")  # kernels.cc:122-124
    T, B, C = logits.shape
    if T == 0:
        raise OracleError("max_time is 0")  # kernels.cc:118-120
    if seq_len.shape[0] != B:
        raise OracleError("len(sequence_length) != batch_size.  len(sequence_length):  %d batch_size: %d"
                          % (seq_len.shape[0], B))  # kernels.cc:126-130
    return logits, seq_len


def ref_decode(logits, seq_len, beam_width, top_paths, merge_repeated=False, blank_index=0,
               blank_label=-1, b_range=None, penalty=None):
    """The reference's own decoder (compiled from /root/reference into oracle/_ref). penalty: a
    stateless scorer (constant expansion score) plugged into the reference's BaseBeamScorer
    extension point, float32 only."""
    lib = _load(REF_SO)
    logits, seq_len = _check_inputs(logits, seq_len)
    T, B, C = logits.shape
    if penalty is not None:
        logits = logits.astype(np.float32, copy=False)
        b0, b1 = b_range if b_range is not None else (0, B)
        dec_len, dec, ali_len, ali, logp = _dense_out(B, top_paths, T, np.float32)
        err = ctypes.create_string_buffer(256)
        lib.ctcx_ref_decode_penalty_f32.argtypes = [_c_float_p] + [ctypes.c_int] * 3 + [_c_int_p] + \
            [ctypes.c_int] * 7 + [ctypes.c_float] + [_c_int_p] * 4 + [_c_float_p, ctypes.c_char_p, ctypes.c_int]
        rc = lib.ctcx_ref_decode_penalty_f32(
            _ptr(logits, _c_float_p), T, B, C, _ptr(seq_len, _c_int_p), b0, b1, beam_width, top_paths,
            int(bool(merge_repeated)), blank_index, blank_label, float(penalty), _ptr(dec_len, _c_int_p),
            _ptr(dec, _c_int_p), _ptr(ali_len, _c_int_p), _ptr(ali, _c_int_p), _ptr(logp, _c_float_p), err, 256)
        if rc != 0:
            raise OracleError(err.value.decode())
        return DenseResult(B, top_paths, T, dec_len, dec, ali_len, ali, logp)
    if logits.dtype == np.float64:
        fn, fp, dt = lib.ctcx_ref_decode_f64, _c_double_p, np.float64
    else:
        logits = logits.astype(np.float32, copy=False)
        fn, fp, dt = lib.ctcx_ref_decode_f32, _c_float_p, np.float32
    b0, b1 = b_range if b_range is not None else (0, B)
    dec_len, dec, ali_len, ali, logp = _dense_out(B, top_paths, T, dt)
    err = ctypes.create_string_buffer(256)
    rc = fn(_ptr(logits, fp), T, B, C, _ptr(seq_len, _c_int_p), b0, b1, beam_width, top_paths,
            int(bool(merge_repeated)), blank_index, blank_label, _ptr(dec_len, _c_int_p),
            _ptr(dec, _c_int_p), _ptr(ali_len, _c_int_p), _ptr(ali, _c_int_p), _ptr(logp, fp), err, 256)
    if rc != 0:
        raise OracleError(err.value.decode())
    return DenseResult(B, top_paths, T, dec_len, dec, ali_len, ali, logp)


def ref_trace(logits_tc, beam_width, merge_repeated=False, blank_index=0, blank_label=-1):
    """Per-frame beam (best first) of one utterance from the compiled reference: list over t of
    [(logp, prefix, alignment), ...]."""
    lib = _load(REF_SO)
    x = np.ascontiguousarray(logits_tc, dtype=np.float32)
    T, C = x.shape
    W = beam_width
    n = np.zeros(T, np.int32)
    logp = np.zeros(T * W, np.float32)
    dec_len = np.zeros(T * W, np.int32)
    dec = np.zeros(T * W * T, np.int32)
    ali = np.zeros(T * W * T, np.int32)
    lib.ctcx_ref_trace_f32(_ptr(x, _c_float_p), T, C, W, int(bool(merge_repeated)), blank_index,
                           blank_label, _ptr(n, _c_int_p), _ptr(logp, _c_float_p),
                           _ptr(dec_len, _c_int_p), _ptr(dec, _c_int_p), _ptr(ali, _c_int_p))
    out = []
    for t in range(T):
        row = []
        for p in range(n[t]):
            r = t * W + p
            row.append((float(logp[r]), dec[r * T:r * T + dec_len[r]].tolist(),
                        ali[r * T:r * T + t + 1].tolist()))
        out.append(row)
    return out


N_MARGINS = 5  # CTCX_MARGIN_{ACCEPT,BOTTOM,ORDER,ALIGN,FINAL} in oracle/ctcx_oracle.c
MARGIN_NAMES = ("accept", "bottom", "order", "align", "final")


class OracleStats(ctypes.Structure):
    """Mirror of ctcx_oracle_stats in oracle/ctcx_oracle.c."""
    _fields_ = [
        ("frames", ctypes.c_longlong),
        ("turns_passed_gate", ctypes.c_longlong),
        ("child_evals", ctypes.c_longlong),
        ("accepted", ctypes.c_longlong),
        ("wipes", ctypes.c_longlong),
        ("wipes_before_turn", ctypes.c_longlong),
        ("frames_with_effective_wipe", ctypes.c_longlong),
        ("relevant_children", ctypes.c_longlong),
        ("surviving_children", ctypes.c_longlong),
        ("revisit_accepts", ctypes.c_longlong),
        ("max_relevant_children", ctypes.c_longlong),
        ("effective_wipes", ctypes.c_longlong),
        ("revisit_above_former", ctypes.c_longlong),
    ]


def oracle_decode(logits, seq_len, beam_width, top_paths, merge_repeated=False, blank_index=0,
                  blank_label=-1, want_margin=False, want_stats=False, lm=None):
    """This repo's plain-C restatement (oracle/ctcx_oracle.c). Returns DenseResult; with
    want_margin also a float64 [B,5] array with each utterance's minimum decision margins.
    lm: optional [C+1, C] float32 expansion-score table of the scorer extension point."""
    lib = _load(ORACLE_SO)
    logits, seq_len = _check_inputs(logits, seq_len)
    T, B, C = logits.shape
    if lm is not None:
        logits = logits.astype(np.float32, copy=False)
        lm = np.ascontiguousarray(lm, np.float32)
        assert lm.shape == (C + 1, C)
        dec_len, dec, ali_len, ali, logp = _dense_out(B, top_paths, T, np.float32)
        margin = np.full((max(B, 1), N_MARGINS), np.inf, np.float64)
        stats = OracleStats()
        err = ctypes.create_string_buffer(256)
        rc = lib.ctcx_oracle_decode_lm_f32(
            _ptr(logits, _c_float_p), T, B, C, _ptr(seq_len, _c_int_p), beam_width, top_paths,
            int(bool(merge_repeated)), blank_index, blank_label, _ptr(lm, _c_float_p), _ptr(dec_len, _c_int_p),
            _ptr(dec, _c_int_p), _ptr(ali_len, _c_int_p), _ptr(ali, _c_int_p), _ptr(logp, _c_float_p),
            _ptr(margin, _c_double_p), ctypes.byref(stats), err, 256)
        if rc != 0:
            raise OracleError(err.value.decode())
        res = DenseResult(B, top_paths, T, dec_len, dec, ali_len, ali, logp)
        out = [res] + ([margin[:B]] if want_margin else []) + ([stats] if want_stats else [])
        return out[0] if len(out) == 1 else tuple(out)
    if logits.dtype == np.float64:
        fn, fp, dt = lib.ctcx_oracle_decode_f64, _c_double_p, np.float64
    else:
        logits = logits.astype(np.float32, copy=False)
        fn, fp, dt = lib.ctcx_oracle_decode_f32, _c_float_p, np.float32
    dec_len, dec, ali_len, ali, logp = _dense_out(B, top_paths, T, dt)
    margin = np.full((max(B, 1), N_MARGINS), np.inf, np.float64)
    stats = OracleStats()
    err = ctypes.create_string_buffer(256)
    rc = fn(_ptr(logits, fp), T, B, C, _ptr(seq_len, _c_int_p), beam_width, top_paths,
            int(bool(merge_repeated)), blank_index, blank_label, _ptr(dec_len, _c_int_p),
            _ptr(dec, _c_int_p), _ptr(ali_len, _c_int_p), _ptr(ali, _c_int_p), _ptr(logp, fp),
            _ptr(margin, _c_double_p), ctypes.byref(stats), err, 256)
    if rc != 0:
        raise OracleError(err.value.decode())
    res = DenseResult(B, top_paths, T, dec_len, dec, ali_len, ali, logp)
    out = [res]
    if want_margin:
        out.append(margin[:B])
    if want_stats:
        out.append(stats)
    return out[0] if len(out) == 1 else tuple(out)


def pack_sparse(res, P=None):
    """Restates StoreAllDecodedSequences (kernels.cc:163-257): per path p, row-major over b then
    position: indices [N_p,2] = [b, pos], values [N_p], shape [B, max length over batch] -- returned
    in the raw op's output order (ops.cc:17-23): 6 lists of P arrays + log_probability."""
    P = res.P if P is None else P
    B = res.B
    out = ([], [], [], [], [], [])
    for lens, rows, (o_idx, o_val, o_shape) in ((res.dec_len, res.dec, out[0:3]),
                                               (res.ali_len, res.ali, out[3:6])):
        for p in range(P):
            idx, val, mx = [], [], 0
            for b in range(B):
                n = int(lens[b, p])
                mx = max(mx, n)
                val.extend(rows[b, p, :n].tolist())
                idx.extend([b, i] for i in range(n))
            o_idx.append(np.asarray(idx, np.int64).reshape(-1, 2))
            o_val.append(np.asarray(val, np.int64))
            o_shape.append(np.asarray([B, mx], np.int64))
    return out + (res.logp.copy(),)


def pack_sparse_fast(res, P=None):
    """pack_sparse, vectorised (same arrays; for batches of thousands of utterances)."""
    P = res.P if P is None else P
    B = res.B
    out = ([], [], [], [], [], [])
    for lens, rows, (o_idx, o_val, o_shape) in ((res.dec_len, res.dec, out[0:3]),
                                               (res.ali_len, res.ali, out[3:6])):
        for p in range(P):
            n = np.asarray(lens[:, p], np.int64)
            mask = np.arange(rows.shape[2])[None, :] < n[:, None]
            o_idx.append(np.argwhere(mask).astype(np.int64).reshape(-1, 2))
            o_val.append(np.asarray(rows[:, p, :])[mask].astype(np.int64))
            o_shape.append(np.asarray([B, int(n.max()) if B else 0], np.int64))
    return out + (res.logp.copy(),)


def host_threads(cap=64):
    try:
        n = len(os.sched_getaffinity(0))
    except AttributeError:
        n = os.cpu_count() or 1
    return max(1, min(n, cap))


def _sharded(fn, x, sl, P, threads, dtype):
    """Runs fn(b0, b1) -> DenseResult over contiguous utterance blocks on host threads (the C
    checkers release the GIL) and concatenates the blocks."""
    from concurrent.futures import ThreadPoolExecutor
    T, B, _ = x.shape
    n = max(1, min(threads or host_threads(), B))
    bounds = [(B * i // n, B * (i + 1) // n) for i in range(n)]
    with ThreadPoolExecutor(n) as ex:
        parts = list(ex.map(lambda bb: fn(*bb), bounds))
    r = DenseResult.__new__(DenseResult)
    r.B, r.P, r.T = B, P, T
    r.dec_len = np.concatenate([q.dec_len for q in parts], axis=0)
    r.ali_len = np.concatenate([q.ali_len for q in parts], axis=0)
    r.dec = np.concatenate([q.dec for q in parts], axis=0)
    r.ali = np.concatenate([q.ali for q in parts], axis=0)
    r.logp = np.concatenate([q.logp for q in parts], axis=0)
    return r


def oracle_decode_threaded(x, sl, W, P, merge=False, blank=0, blank_label=-1, lm=None, threads=None):
    """oracle_decode over host threads, one contiguous block of utterances per thread."""
    x = np.asarray(x)
    sl = np.asarray(sl, np.int32)
    return _sharded(lambda b0, b1: oracle_decode(np.ascontiguousarray(x[:, b0:b1]), sl[b0:b1], W, P, merge,
                                                 blank, blank_label, lm=lm),
                    x, sl, P, threads, x.dtype)


def ref_decode_threaded(x, sl, W, P, merge=False, blank=0, blank_label=-1, threads=None):
    """The compiled reference over host threads. It keeps ~0.5 GB of trie per in-flight utterance at
    T=500, W=100 (SURVEY.md section 6), so the number of threads is what bounds the memory."""
    x = np.ascontiguousarray(x)
    sl = np.asarray(sl, np.int32)

    def block(b0, b1):
        r = ref_decode(x, sl, W, P, merge, blank, blank_label, b_range=(b0, b1))
        q = DenseResult.__new__(DenseResult)
        q.B, q.P, q.T = b1 - b0, P, r.T
        q.dec_len, q.ali_len = r.dec_len[b0:b1], r.ali_len[b0:b1]
        q.dec, q.ali, q.logp = r.dec[b0:b1], r.ali[b0:b1], r.logp[b0:b1]
        return q
    return _sharded(block, x, sl, P, threads, x.dtype)


def raw_mismatches(raw, want):
    """Utterances whose raw op outputs (7 groups, device or host tensors) differ from a DenseResult:
    compared array-for-array per path against the vectorised restatement of the reference's packing,
    log_probability by its IEEE bits. Returns the sorted list of differing utterance indices."""
    def npy(a):
        return a.detach().cpu().numpy() if hasattr(a, "detach") else np.asarray(a)
    packed = pack_sparse_fast(want)
    B, P = want.B, want.P
    bad = set()
    for base, lens, rows in ((0, want.dec_len, want.dec), (3, want.ali_len, want.ali)):
        for p in range(P):
            idx, val, shape = npy(raw[base][p]), npy(raw[base + 1][p]), npy(raw[base + 2][p])
            if idx.shape == packed[base][p].shape and np.array_equal(idx, packed[base][p]) and \
                    np.array_equal(val, packed[base + 1][p]) and np.array_equal(shape, packed[base + 2][p]):
                continue
            # locate the utterances: compare per-utterance segments
            got = [[] for _ in range(B)]
            for (b, _), v in zip(idx.tolist(), val.tolist()):
                if 0 <= b < B:
                    got[b].append(v)
            for b in range(B):
                if got[b] != rows[b, p, :lens[b, p]].tolist():
                    bad.add(b)
            if not np.array_equal(shape, packed[base + 2][p]):
                bad.add(-1)
    lp = npy(raw[6])
    view = np.uint64 if lp.dtype == np.float64 else np.uint32
    neq = np.argwhere(lp.view(view) != np.asarray(want.logp, lp.dtype).view(view))
    bad.update(int(b) for b, _ in neq)
    return sorted(bad)


# ----------------------------------------------------------------------------------------------
# Synthetic inputs (SURVEY.md section 8d): identical tensors for the CPU checkers and the GPU path.
def make_logits(kind, T, B, C, blank_index, seed, sigma=1.0, spike=8.0):
    rng = np.random.default_rng(seed)
    x = (rng.standard_normal((T, B, C)) * sigma).astype(np.float32)
    if kind == "gauss":
        return x
    if kind == "peaky":
        nonblank = np.array([c for c in range(C) if c != blank_index], np.int64)
        is_spike = rng.random((T, B)) < 0.25
        lab = nonblank[rng.integers(0, C - 1, (T, B))]
        cls = np.where(is_spike, lab, blank_index)
        tt, bb = np.meshgrid(np.arange(T), np.arange(B), indexing="ij")
        x[tt, bb, cls] += np.float32(spike)
        return x
    raise ValueError(kind)


def ragged_lengths(T, B, seed):
    rng = np.random.default_rng(seed + 1000003)
    return rng.integers(T // 2, T + 1, B).astype(np.int32)


PAPER_PROBS = [[0.3, 0.5, 0.2], [0.25, 0.6, 0.15], [0.6, 0.2, 0.2], [0.4, 0.35, 0.25],
               [0.5, 0.4, 0.1], [0.3, 0.3, 0.4], [0.1, 0.2, 0.7], [0.2, 0.3, 0.5]]


def paper_logits(dtype=np.float64):
    """python/ops/ctc_ext_beam_search_decoder_ops_test.py:25-33 (np.log of the table, float64)."""
    return np.log(np.asarray(PAPER_PROBS, np.float64))[:, None, :].astype(dtype)


# ----------------------------------------------------------------------------------------------
# CPU model of the parallel formulation (tests/model/ctcx_model.cc)
MODEL_SRC = os.path.join(ROOT, "tests", "model", "ctcx_model.cc")
MODEL_SO = os.path.join(ROOT, "tests", "model", "libctcx_model.so")
MODEL_STATS = ("frames cands at_risk fp_iters fp_iters_max wiped wiped_with_cands anomalies cands_max "
               "frames_wipe_matters queries radix_bits_sum fp_unwipes wiped_parents frames_at_risk "
               "suspects_dropped").split()


def build_model(force=False):
    if force or not os.path.exists(MODEL_SO) or os.path.getmtime(MODEL_SO) < os.path.getmtime(MODEL_SRC):
        subprocess.check_call(["g++", "-O2", "-std=c++11", "-ffp-contract=off", "-fPIC", "-shared",
                               "-o", MODEL_SO, MODEL_SRC])


def model_decode(logits, seq_len, beam_width, top_paths, merge_repeated=False, blank_index=0,
                 blank_label=-1, want_stats=False):
    build_model()
    lib = _load(MODEL_SO)
    logits, seq_len = _check_inputs(logits, seq_len)
    logits = logits.astype(np.float32, copy=False)
    T, B, C = logits.shape
    dec_len, dec, ali_len, ali, logp = _dense_out(B, top_paths, T, np.float32)
    st = np.zeros(16, np.int64)
    rc = lib.ctcx_model_decode_f32(_ptr(logits, _c_float_p), T, B, C, _ptr(seq_len, _c_int_p),
                                   beam_width, top_paths, int(bool(merge_repeated)), blank_index,
                                   blank_label, _ptr(dec_len, _c_int_p), _ptr(dec, _c_int_p),
                                   _ptr(ali_len, _c_int_p), _ptr(ali, _c_int_p), _ptr(logp, _c_float_p),
                                   st.ctypes.data_as(ctypes.POINTER(ctypes.c_longlong)))
    if rc != 0:
        raise OracleError({2: "max_time is 0", 6: "requested more paths than the beam width.",
                           7: "Less leaves in the beam search than requested."}.get(rc, "error %d" % rc))
    res = DenseResult(B, top_paths, T, dec_len, dec, ali_len, ali, logp)
    return (res, dict(zip(MODEL_STATS, st.tolist()))) if want_stats else res


MODEL_VARIANTS = {"exact": 0, "count_wiped_rows": 1, "four_rounds": 2}


def model_decode_utts(logits, seq_len, beam_width, top_paths, merge_repeated=False, blank_index=0,
                      blank_label=-1, variant="exact", lm=None):
    """model_decode with the statistics of every utterance: (DenseResult, [dict per utterance],
    int32 [B, T] rounds of the revisit-wipe fixed point per frame, 0 where nobody is at risk).
    variant: "exact", or a fixed point with a known mistake -- "count_wiped_rows" (the candidates of
    wiped rows still count) or "four_rounds" (stops after 4 rounds) -- to show that a case exposes it.
    lm: optional [C+1, C] float32 scorer table, as for oracle_decode."""
    build_model()
    lib = _load(MODEL_SO)
    logits, seq_len = _check_inputs(logits, seq_len)
    logits = logits.astype(np.float32, copy=False)
    T, B, C = logits.shape
    if lm is not None:
        lm = np.ascontiguousarray(lm, np.float32)
        assert lm.shape == (C + 1, C)
    dec_len, dec, ali_len, ali, logp = _dense_out(B, top_paths, T, np.float32)
    st = np.zeros((max(B, 1), 16), np.int64)
    iters = np.zeros((max(B, 1), T), np.int32)
    rc = lib.ctcx_model_decode_lm_utts_f32(_ptr(logits, _c_float_p), T, B, C, _ptr(seq_len, _c_int_p),
                                           beam_width, top_paths, int(bool(merge_repeated)), blank_index,
                                           blank_label, None if lm is None else _ptr(lm, _c_float_p),
                                           _ptr(dec_len, _c_int_p), _ptr(dec, _c_int_p),
                                           _ptr(ali_len, _c_int_p), _ptr(ali, _c_int_p), _ptr(logp, _c_float_p),
                                           None, st.ctypes.data_as(ctypes.POINTER(ctypes.c_longlong)),
                                           _ptr(iters, _c_int_p), MODEL_VARIANTS[variant])
    if rc != 0:
        raise OracleError({2: "max_time is 0", 6: "requested more paths than the beam width.",
                           7: "Less leaves in the beam search than requested."}.get(rc, "error %d" % rc))
    res = DenseResult(B, top_paths, T, dec_len, dec, ali_len, ali, logp)
    return res, [dict(zip(MODEL_STATS, row)) for row in st[:B].tolist()], iters[:B]


def same_result(a, b, bitwise=True):
    """Utterance/path pairs where two DenseResults differ (labels, alignments, log-prob bits)."""
    bad = []
    for u in range(a.B):
        for p in range(a.P):
            lp_ok = (np.asarray(a.logp[u, p]).view(np.uint32 if a.logp.dtype == np.float32 else np.uint64)
                     == np.asarray(b.logp[u, p]).view(np.uint32 if b.logp.dtype == np.float32 else np.uint64)) \
                if bitwise and a.logp.dtype == b.logp.dtype else np.isclose(a.logp[u, p], b.logp[u, p], rtol=1e-6, atol=1e-6)
            if a.decoded(u, p) != b.decoded(u, p) or a.alignment(u, p) != b.alignment(u, p) or not lp_ok:
                bad.append((u, p))
    return bad


# ----------------------------------------------------------------------------------------------
# Golden fixtures generated from the reference itself (tests/golden/make_golden.py)
GOLDEN_NPZ = os.path.join(ROOT, "tests", "golden", "ref_cases.npz")
GOLDEN_JSON = os.path.join(ROOT, "tests", "golden", "ref_cases.json")


class Golden:
    def __init__(self):
        import json
        self.arr = np.load(GOLDEN_NPZ)
        self.meta = json.load(open(GOLDEN_JSON))

    def result(self, name):
        g = lambda k: self.arr["%s/%s" % (name, k)]  # noqa: E731
        dec_len, ali_len = g("dec_len"), g("ali_len")
        B, P = dec_len.shape
        T = g("dec").shape[2]
        r = DenseResult.__new__(DenseResult)
        r.B, r.P, r.T = B, P, T
        r.dec_len, r.ali_len, r.dec, r.ali, r.logp = dec_len, ali_len, g("dec"), g("ali"), g("logp")
        return r

    def tie_free(self, name):
        k = "%s/tie_free" % name
        return self.arr[k] if k in self.arr else None

    def random_cases(self):
        """[(name, x, seq_len, W, P, merge, blank_index, blank_label)]"""
        out = []
        for c in self.meta["random"]:
            name, kind, T, B, C, W, P, merge, blank, bl, seed, sigma, ragged, dt = c
            x = make_logits(kind, T, B, C, blank, seed, sigma)
            if dt == "f64":
                x = x.astype(np.float64)
            sl = ragged_lengths(T, B, seed) if ragged else np.full(B, T, np.int32)
            out.append((name, x, sl, W, P, merge, blank, bl))
        return out

    def literal_cases(self):
        out = []
        for name, rows, sl, W, P, merge, blank, bl in self.meta["literal"]:
            x = np.asarray(rows, np.float32)[:, None, :]
            out.append((name, x, np.asarray([sl], np.int32), W, P, merge, blank, bl))
        return out


# ----------------------------------------------------------------------------------------------
# Revisit-wipe cases found by a search on the CPU model (tests/golden/make_wipe_cases.py)
WIPE_NPZ = os.path.join(ROOT, "tests", "golden", "wipe_cases.npz")
WIPE_TABLE_NPZ = os.path.join(ROOT, "tests", "golden", "wipe_table_cases.npz")  # (make_wipe_table_cases.py)


class WipeCase:
    """One utterance of wipe_cases.npz: logits k/16 (float32, [T, 1, C]), decode attributes, and the
    model's statistics (dict over MODEL_STATS) and fixed-point rounds per frame recorded for it. `lm`: the
    case's scorer table ([C + 1, C] float32, k/16 with -inf) for wipe_table_cases.npz, else None."""

    def __init__(self, arr, name):
        k = arr[name + "/k"]
        self.name = name
        self.x = np.where(k == -32768, -np.inf, k.astype(np.float32) / 16).astype(np.float32)[:, None, :]
        self.T, _, self.C = self.x.shape
        self.W, self.blank, merge, self.P, exposes = (int(v) for v in arr[name + "/attrs"])
        self.merge = bool(merge)
        # the mistaken fixed point (a model_decode_utts variant) under which this case decodes differently
        self.exposes = {v: k for k, v in MODEL_VARIANTS.items()}[exposes] if exposes else None
        self.stats = dict(zip(MODEL_STATS, arr[name + "/stats"].tolist()))
        self.iters = arr[name + "/iters"].astype(np.int32)
        self.sl = np.array([self.T], np.int32)
        self.lm = None
        if name + "/lm" in arr.files:
            q = arr[name + "/lm"]
            self.lm = np.where(q == -32768, -np.inf, q.astype(np.float32) / 16).astype(np.float32)


def wipe_cases(path=WIPE_NPZ):
    arr = np.load(path)
    return [WipeCase(arr, str(n)) for n in arr["names"]]


def wipe_table_cases():
    return wipe_cases(WIPE_TABLE_NPZ)
