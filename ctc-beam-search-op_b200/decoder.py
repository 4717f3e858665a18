"""Host side of the drop-in: `ctc_ext_beam_search_decoder` with the reference's signature.

Mirrors (paths relative to /root/reference/tensorflow_ctc_ext_beam_search_decoder/):
  * the op contract                      cc/ops/ctc_ext_beam_search_decoder_ops.cc:9-24
  * the Python surface                   python/ops/ctc_ext_beam_search_decoder_ops.py:10-12
    (the generated raw wrapper: keyword call, result indexable [0..6] -- see
    python/ops/ctc_ext_beam_search_decoder_ops_test.py:67-100)
  * the documented return value          README.md:19-31  `(decoded, alignment, log_probability)`
  * validation order and messages        cc/kernels/ctc_ext_beam_search_decoder_kernels.cc:97-160
                                         cc/util/ctc_ext_beam_search_decoder.h:237-243

All compute happens in the CUDA library behind include/ctcx.h; PyTorch is used only for device
memory and streams. There is no CPU path: without a CUDA device the call raises.
"""
import collections
import ctypes

import numpy as np
import torch

from . import _lib

SparseTensor = collections.namedtuple("SparseTensor", ["indices", "values", "dense_shape"])

# Same field order as the raw op's outputs (ops.cc:17-23); indexable like the generated TF wrapper.
_RawBase = collections.namedtuple(
    "CTCExtBeamSearchDecoder",
    ["decoded_indices", "decoded_values", "decoded_shape", "alignment_indices", "alignment_values",
     "alignment_shape", "log_probability"])


class CTCExtBeamSearchDecoder(_RawBase):
    """The raw op's 7 output groups (indexable [0..6] like the generated TF wrapper). `.flags` carries
    this decode's diagnostic bits (FLAG_ROUNDING_ANOMALY) -- an attribute, not an eighth output.
    `.slots`: the stream slots of the rows of a per-slot read (CTCExtBeamSearchDecoderStream), else None."""
    flags = 0
    d2h_bytes = 0
    slots = None


class DecodeResult(tuple):
    """`(decoded, alignment, log_probability)` (README.md:19-31) plus `.flags` (and `.slots`, see
    CTCExtBeamSearchDecoder) attributes."""
    flags = 0
    slots = None


class CtcxError(ValueError):
    """Base class; `.code` is the C-ABI return code (include/ctcx.h)."""

    def __init__(self, code, message):
        super().__init__(message)
        self.code = code

    def __reduce__(self):  # picklable: errors travel between ranks (sharding.decode_distributed)
        return (type(self), (self.code, str(self)))


class InvalidArgumentError(CtcxError):
    """tf.errors.InvalidArgumentError counterpart."""


class FailedPreconditionError(CtcxError):
    """tf.errors.FailedPreconditionError counterpart."""


class UnsupportedError(CtcxError):
    """Shape outside the limits of this build (not a reference error)."""


_ERR_CLASS = {1: InvalidArgumentError, 2: InvalidArgumentError, 3: InvalidArgumentError,
              4: FailedPreconditionError, 5: FailedPreconditionError, 6: InvalidArgumentError,
              7: InvalidArgumentError, 8: InvalidArgumentError, 9: UnsupportedError}

FLAG_ROUNDING_ANOMALY = 1  # see DESIGN.md "Known deviation"

_DTYPE_CODE = {torch.float32: _lib.F32, torch.float16: _lib.F16, torch.bfloat16: _lib.BF16,
               torch.float64: _lib.F64}
_copy_streams = {}


def set_beam_impl(name):
    """Test hook: None / "fast" = dispatch by shape; "generic" = route every decode of this process to
    the generic beam kernel (the independent second implementation the parity tests compare with)."""
    if name not in (None, "fast", "generic"):
        raise ValueError("unknown beam implementation %r" % (name,))
    _lib.load().ctcx_debug_set_beam_impl(1 if name == "generic" else 0)


def _copy_stream(device):
    """One side stream per device for the host->device feed of host-input decodes."""
    key = (device.type, device.index)
    if key not in _copy_streams:
        _copy_streams[key] = torch.cuda.Stream(device=device)
    return _copy_streams[key]


def _raise(lib, rc, batch_offset=0):
    msg = lib.ctcx_strerror(rc).decode()
    if rc == 5 and batch_offset:  # kernels.cc:134-138 names the utterance: report its index in the WHOLE batch
        b = lib.ctcx_error_batch_index()
        msg = msg.replace("sequence_length(%d)" % b, "sequence_length(%d)" % (b + batch_offset), 1)
    if rc in _ERR_CLASS:
        exc = _ERR_CLASS[rc](rc, msg)
        if rc == 5:
            exc.batch_index = lib.ctcx_error_batch_index() + int(batch_offset)
        raise exc
    raise RuntimeError("ctcx: %s (code %d)" % (msg, rc))


def _as_tensor(a):
    if isinstance(a, torch.Tensor):
        return a, False
    return torch.from_numpy(np.ascontiguousarray(a)), True


def _carve(buf, B, P, counts, f64):
    """Views of one int64 buffer: the 6*P sparse tensors (ops.cc:17-22) followed by log_probability."""
    n_dec, n_ali = counts
    o = 0
    groups = [[], [], [], [], [], []]

    def take(n, shape):
        nonlocal o
        t = buf[o:o + n].view(shape)
        o += n
        return t

    for p in range(P):
        nd, na = int(n_dec[p]), int(n_ali[p])
        groups[0].append(take(2 * nd, (nd, 2)))
        groups[1].append(take(nd, (nd,)))
        groups[2].append(take(2, (2,)))
        groups[3].append(take(2 * na, (na, 2)))
        groups[4].append(take(na, (na,)))
        groups[5].append(take(2, (2,)))
    n_lp = B * P if f64 else (B * P + 1) // 2  # in int64 units
    lp = buf[o:o + n_lp].view(torch.float64 if f64 else torch.float32)[:B * P].view(B, P)
    return groups, lp


def _pack_elems(B, P, counts, f64):
    n_dec, n_ali = counts
    return sum(3 * int(n_dec[p]) + 3 * int(n_ali[p]) + 4 for p in range(P)) + (B * P if f64 else (B * P + 1) // 2)


def _pack(lib, ws, T, B, P, counts, device, stream, f64=False, host_out=False):
    """Allocate the 6*P sparse tensors from the sizes a decode reported and let ctcx_pack_f32 /
    ctcx_pack_f64 fill them (StoreAllDecodedSequences, kernels.cc:163-257). All outputs are views of
    ONE buffer, so results for host callers cross the bus in a single copy into pinned memory (from
    torch's caching host allocator) instead of 6*P+1 pageable ones."""
    n = _pack_elems(B, P, counts, f64)
    buf = torch.empty((n,), dtype=torch.int64, device=device)
    groups, logp = _carve(buf, B, P, counts, f64)
    ptrs = ctypes.c_void_p * P

    def table(ts):
        return ptrs(*[t.data_ptr() for t in ts])

    pack = lib.ctcx_pack_f64 if f64 else lib.ctcx_pack_f32
    rc = pack(ws.data_ptr(), T, B, P, table(groups[0]), table(groups[1]), table(groups[2]),
              table(groups[3]), table(groups[4]), table(groups[5]), logp.data_ptr(), stream)
    if rc != 0:
        _raise(lib, rc)
    if host_out:
        hbuf = torch.empty((n,), dtype=torch.int64, pin_memory=True)
        hbuf.copy_(buf, non_blocking=True)
        torch.cuda.current_stream(device).synchronize()
        buf = hbuf
        groups, logp = _carve(hbuf, B, P, counts, f64)
    return groups, logp, buf


# Results up to this size take the deferred route (decode and pack enqueued back to back into a buffer
# sized from an upper bound, ONE synchronisation at the end); larger ones the two-phase route (sizes
# first, then exactly sized outputs), whose extra host round trip no longer matters at that scale and
# which never holds or copies more than the exact result.
DEFER_MAX_BYTES_DEVICE = 64 << 20
DEFER_MAX_BYTES_HOST = 8 << 20


def _bound_elems(T, B, P, seq, f64):
    """Upper bound on the int64 slots of the compact output layout: a path's decoded sequence is never
    longer than its alignment, an alignment has exactly sequence_length entries."""
    if seq.is_cuda:
        frames = B * T
    else:
        frames = int(seq.to(torch.int64).clamp(0, T).sum())
    return P * (6 * frames + 4) + (B * P if f64 else (B * P + 1) // 2)


def _frame_strided(x):
    """True if x[t, b, c] sits at t * stride + b * C + c, i.e. x is a contiguous tensor or a batch
    shard [:, b0:b1, :] of one -- what the kernels decode in place (ctcx_decode_view)."""
    T, B, C = x.shape
    st = x.stride()
    return (C == 1 or st[2] == 1) and (B == 1 or st[1] == C) and (T == 1 or st[0] >= B * C)


def ctc_ext_beam_search_decoder_raw(inputs, sequence_length, beam_width, top_paths,
                                    merge_repeated=False, blank_index=0, blank_label=-1,
                                    name=None, device=None, expansion_scores=None, batch_offset=0,
                                    outputs="auto", wait=True):
    """The raw op: returns a 7-field namedtuple of (lists of) tensors, exactly the op's outputs.

    inputs            [max_time, batch, num_classes] float32 or float64 (the reference registers both,
                      kernels.cc:269-275; float64 is computed in float64 by the double instantiations
                      of the kernels and log_probability is float64); float16 / bfloat16 are
                      read by the kernels as they are (widened exactly in registers); numpy array or
                      torch tensor on any device. A batch shard `x[:, b0:b1, :]` of a contiguous
                      tensor is decoded in place (device) / copied with a pitched copy (host) -- no
                      repack. Host inputs are copied to the device in time slabs on a side stream
                      while the beam kernel already runs (ctcx_decode_hostin).
    sequence_length   [batch] int32
    beam_width >= 1, top_paths >= 1, merge_repeated=False, blank_index=0, blank_label=-1
    expansion_scores  optional [num_classes + 1, num_classes] float32 table (entries <= 0) for the
                      reference's scorer extension point (util/ctc_beam_scorer.h): extending an entry
                      whose last label is f (row f + 1; row 0 = empty prefix) by label l adds
                      table[f + 1, l] to the score carried over -- a bigram LM / insertion penalty.
                      float32 inputs only; None = the op's default scorer.
    batch_offset      index of utterance 0 in the caller's whole batch (error messages of a shard)
    outputs           "auto": outputs live where the inputs live (numpy in -> numpy out); "device" /
                      "host" force the placement (torch tensors)
    wait              False: return a PendingDecode right after the work has been enqueued on the
                      current stream; its .result() synchronises and returns the outputs
    `.flags` = diagnostic bits; `.packed` = the one int64 buffer all outputs are views of.
    """
    del name
    if int(beam_width) < 1:
        raise ValueError("Attr beam_width has value %d less than minimum 1" % int(beam_width))
    if int(top_paths) < 1:
        raise ValueError("Attr top_paths has value %d less than minimum 1" % int(top_paths))
    lib = _lib.load()
    x_np = not isinstance(inputs, torch.Tensor)
    if x_np:
        xa = np.asarray(inputs)
        if xa.dtype.kind != "f":
            raise TypeError("inputs must be a floating-point array, got %s" % xa.dtype)
        if not xa.flags.writeable:  # torch.from_numpy wants a writable array
            xa = xa.copy()
        x = torch.from_numpy(xa)
    else:
        x = inputs
    seq, _ = _as_tensor(np.asarray(sequence_length, dtype=np.int32)
                        if not isinstance(sequence_length, torch.Tensor) else sequence_length)
    # kernels.cc:111-130, in order
    if x.dim() != 3:
        raise InvalidArgumentError(1, lib.ctcx_strerror(1).decode())
    T, B, C = (int(s) for s in x.shape)
    if T == 0:
        raise InvalidArgumentError(2, lib.ctcx_strerror(2).decode())
    if seq.dim() != 1:
        raise InvalidArgumentError(3, lib.ctcx_strerror(3).decode())
    if int(seq.shape[0]) != B:
        raise FailedPreconditionError(
            4, "len(sequence_length) != batch_size.  len(sequence_length):  %d batch_size: %d"
            % (int(seq.shape[0]), B))
    if not x.dtype.is_floating_point:
        raise TypeError("inputs must be float32 or float64, got %s" % x.dtype)
    if not torch.cuda.is_available():
        raise RuntimeError("ctcx: no CUDA device available and there is no CPU fallback")

    if device is None:
        device = x.device if x.is_cuda else torch.device("cuda", torch.cuda.current_device())
    device = torch.device(device)
    host_in = not x.is_cuda
    if x.dtype not in _DTYPE_CODE or expansion_scores is not None:
        if expansion_scores is not None and x.dtype == torch.float64:
            raise TypeError("expansion_scores is supported for float32 inputs only")
        x = x.to(torch.float32)
    f64 = x.dtype == torch.float64
    if not _frame_strided(x):
        x = x.contiguous()
    tstride = int(x.stride(0)) if T > 1 else B * C
    W, P = int(beam_width), int(top_paths)
    attrs = (W, P, int(bool(merge_repeated)), int(blank_index), int(blank_label))
    with torch.cuda.device(device):
        cur = torch.cuda.current_stream(device)
        stream = cur.cuda_stream
        ws_bytes = lib.ctcx_workspace_bytes(T, B, C, W, P)
        ws = torch.empty(max(ws_bytes, 256), dtype=torch.uint8, device=device)
        arr = ctypes.c_int64 * P
        n_dec, max_dec, n_ali, max_ali = arr(), arr(), arr(), arr()
        sizes = _lib.CtcxSizes(n_dec, max_dec, n_ali, max_ali)
        flags = ctypes.c_int32(0)
        host_out = host_in if outputs == "auto" else (outputs == "host")
        n_bound = _bound_elems(T, B, P, seq, f64) if (B > 0 and expansion_scores is None and P <= W) else 0
        deferred = 0 < 8 * n_bound <= (DEFER_MAX_BYTES_HOST if host_out else DEFER_MAX_BYTES_DEVICE)
        sizes_arg = None if deferred else ctypes.byref(sizes)
        flags_arg = None if deferred else ctypes.byref(flags)
        xd = sd = sh = staging = esd = None  # device / staging copies made below (kept alive while in flight)
        if host_in and expansion_scores is None:
            # host logits: copied in time slabs on a side stream while the beam kernel already runs
            sh = seq.to(dtype=torch.int32).contiguous()
            n_stage = lib.ctcx_hostin_staging_bytes(_DTYPE_CODE[x.dtype], T, B, C)
            staging = torch.empty(max(n_stage, 16), dtype=torch.uint8, device=device)
            side = _copy_stream(device)
            rc = lib.ctcx_decode_hostin(x.data_ptr(), _DTYPE_CODE[x.dtype], tstride, T, B, C, sh.data_ptr(),
                                        *attrs, staging.data_ptr(), n_stage, ws.data_ptr(), ws_bytes, stream,
                                        side.cuda_stream, sizes_arg, flags_arg)
            if rc == 9 and x.dtype in (torch.float16, torch.bfloat16):  # (test hook only, see below)
                x = x.float().contiguous()
                n_stage = lib.ctcx_hostin_staging_bytes(_lib.F32, T, B, C)
                staging = torch.empty(max(n_stage, 16), dtype=torch.uint8, device=device)
                rc = lib.ctcx_decode_hostin(x.data_ptr(), _lib.F32, 0, T, B, C, sh.data_ptr(), *attrs,
                                            staging.data_ptr(), n_stage, ws.data_ptr(), ws_bytes, stream,
                                            side.cuda_stream, sizes_arg, flags_arg)
            staging.record_stream(side)
        else:
            xd = x.to(device=device, non_blocking=True)
            sd = seq.to(device=device, dtype=torch.int32, non_blocking=True).contiguous()
            if expansion_scores is not None:
                es, _ = _as_tensor(expansion_scores)
                if tuple(es.shape) != (C + 1, C):
                    raise InvalidArgumentError(8, "expansion_scores must have shape [num_classes + 1, num_classes]")
                esd = es.to(device=device, dtype=torch.float32).contiguous()
                xd = xd.contiguous()
                rc = lib.ctcx_decode_scorer_f32(xd.data_ptr(), T, B, C, sd.data_ptr(), *attrs, esd.data_ptr(),
                                                ws.data_ptr(), ws_bytes, stream, ctypes.byref(sizes),
                                                ctypes.byref(flags))
            else:
                rc = lib.ctcx_decode_view(xd.data_ptr(), _DTYPE_CODE[xd.dtype], tstride, T, B, C, sd.data_ptr(),
                                          *attrs, ws.data_ptr(), ws_bytes, stream, sizes_arg, flags_arg)
                if rc == 9 and xd.dtype in (torch.float16, torch.bfloat16):
                    # (test hook only: the generic kernel forced onto a fast-path shape has no room to widen
                    # half-precision logits in the workspace)
                    xd = xd.float().contiguous()
                    rc = lib.ctcx_decode_view(xd.data_ptr(), _lib.F32, 0, T, B, C, sd.data_ptr(), *attrs,
                                              ws.data_ptr(), ws_bytes, stream, sizes_arg, flags_arg)
        if rc != 0:
            _raise(lib, rc, int(batch_offset))
        hbuf = None
        if deferred:  # the pack (and the copy of the result to the host) follow the decode without a round trip
            buf = torch.empty((n_bound,), dtype=torch.int64, device=device)
            rc = lib.ctcx_pack_compact(ws.data_ptr(), T, B, P, 8 if f64 else 4, buf.data_ptr(), n_bound, stream)
            if rc != 0:
                _raise(lib, rc)
            if host_out:  # the whole bound crosses the bus (at most DEFER_MAX_BYTES_HOST)
                hbuf = torch.empty((n_bound,), dtype=torch.int64, pin_memory=True)
                hbuf.copy_(buf, non_blocking=True)
            # sizes + status words follow into page-locked memory; an event of this decode's own marks the end,
            # so that reading this result never waits for decodes enqueued after it
            n_res = lib.ctcx_result_bytes(P)
            hres = torch.empty((n_res,), dtype=torch.uint8, pin_memory=True)
            rc = lib.ctcx_result_copy_async(ws.data_ptr(), T, B, P, hres.data_ptr(), n_res, stream)
            if rc != 0:
                _raise(lib, rc)
            done = torch.cuda.Event()
            done.record(cur)
    # what the enqueued work reads stays alive until complete() has synchronised
    keep = [x, seq, ws, xd, sd, sh, staging, esd]

    def complete(_keep=keep):
        with torch.cuda.device(device):
            if deferred:
                done.synchronize()
                rc = lib.ctcx_result_parse(hres.data_ptr(), T, B, P, ctypes.byref(sizes), ctypes.byref(flags))
                if rc != 0:
                    _raise(lib, rc, int(batch_offset))
                packed = (hbuf if host_out else buf)[:_pack_elems(B, P, (n_dec, n_ali), f64)]
                groups, logp = _carve(packed, B, P, (n_dec, n_ali), f64)
            else:
                groups, logp, packed = _pack(lib, ws, T, B, P, (n_dec, n_ali), device, stream, f64, host_out)
        if host_out and x_np and outputs == "auto":
            groups = [[t.numpy() for t in g] for g in groups]
            logp = logp.numpy()
        res = CTCExtBeamSearchDecoder(*groups, logp)
        res.flags = int(flags.value)
        res.packed = packed
        res.max_lengths = ([int(v) for v in max_dec], [int(v) for v in max_ali])  # dense_shape[1] per path, on the host
        # bytes copied device -> host by this call: sizes + status words, and for host outputs the result buffer
        res.d2h_bytes = 4 * P * 8 + 64 + (8 * (n_bound if deferred else int(packed.numel())) if host_out else 0)
        _keep.clear()
        return res

    if wait:
        return complete()
    return PendingDecode(complete, eager=not deferred)


class PendingDecode:
    """Handle of a decode that was enqueued with `wait=False`: the kernels, the pack and (for host
    outputs) the copy of the result are in flight on the caller's CUDA stream; `.result()` synchronises
    once and returns what the blocking call would have returned (or raises what it would have raised).
    Lets a caller enqueue the next batch before reading this one -- the GPU then runs decode after
    decode without waiting for the host. Results too large for the single-synchronisation route
    (DEFER_MAX_BYTES_*) are computed before the handle is returned."""

    def __init__(self, complete, eager=False):
        self._complete = complete
        self._res = None
        self._exc = None
        if eager:
            self.result()

    def __del__(self):
        # a handle dropped unread still has copies into its page-locked buffers in flight: wait for them
        # before the buffers go back to the allocator
        if getattr(self, "_complete", None) is not None:
            try:
                self.result()
            except Exception:
                pass

    def result(self):
        if self._complete is not None:
            complete, self._complete = self._complete, None
            try:
                self._res = complete()
            except Exception as e:  # re-raised on every call
                self._exc = e
        if self._exc is not None:
            raise self._exc
        return self._res


def ctc_ext_beam_search_decoder(inputs, sequence_length, beam_width, top_paths,
                                merge_repeated=False, blank_index=0, blank_label=-1, name=None,
                                device=None, expansion_scores=None):
    """`(decoded, alignment, log_probability)` as documented by the reference (README.md:19-31):
    decoded[j] / alignment[j] are SparseTensor(indices [N,2] rows [batch, position], values [N],
    dense_shape [batch, max length]) for path j; log_probability is [batch, top_paths]."""
    raw = ctc_ext_beam_search_decoder_raw(inputs, sequence_length, beam_width, top_paths,
                                          merge_repeated, blank_index, blank_label, name, device,
                                          expansion_scores)
    decoded = [SparseTensor(i, v, s) for i, v, s in zip(raw[0], raw[1], raw[2])]
    alignment = [SparseTensor(i, v, s) for i, v, s in zip(raw[3], raw[4], raw[5])]
    out = DecodeResult((decoded, alignment, raw[6]))
    out.flags = raw.flags
    return out


def _to_device(a, device):
    """A small host array on the device, through page-locked memory: the copy is only enqueued on the
    current stream (a copy from pageable memory would wait for the work queued before it)."""
    return torch.from_numpy(a).pin_memory().to(device, non_blocking=True)


def _torch_dtype(dtype):
    """torch dtype of a torch or numpy dtype (np.float64, "float64", ...)."""
    if isinstance(dtype, torch.dtype):
        return dtype
    return torch.from_numpy(np.empty(0, dtype=np.dtype(dtype))).dtype


class CTCExtBeamSearchDecoderStream:
    """Streaming form of the decoder: the reference's `Step / TopPaths / Reset`
    (cc/util/ctc_ext_beam_search_decoder.h:39-53) for a whole batch, with the beam kept on the
    device between calls. Feeding the frames of an utterance in any chunking gives bit-identical
    results to one `ctc_ext_beam_search_decoder` call on the concatenation with the same score type
    and table.

        dec = CTCExtBeamSearchDecoderStream(batch_size=B, num_classes=C, beam_width=100, top_paths=1,
                                            max_time=3000, merge_repeated=True, blank_index=C - 1)
        for chunk in chunks:                  # [chunk_time, B, C] logits
            dec.step(chunk)                   # or dec.step(chunk, lengths) for ragged chunks
            decoded, alignment, logp = dec.top_paths()   # any time; does not disturb the state
        dec.reset()

    Each of the B utterance positions (slots) can also start and finish on its own, so that a server can
    keep B live streams in one batch: `reset(slots)` puts the selected slots back at the root (their
    `max_time` budget starts again) and leaves the others untouched, and `top_paths(slots)` reads the
    selected slots only:

        done = [b for b in range(B) if finished[b]]
        pending = dec.top_paths(done, wait=False)   # enqueued; stepping may go on before it is read
        dec.reset(done)                             # the slots take new utterances from the next step
        ...
        decoded, alignment, logp = pending.result() # row i = slot done[i]

    dtype             score type of the stream (torch or numpy dtype): float32 (default) takes float32,
                      float16 and bfloat16 chunks (half chunks are read in place, as the one-shot decode
                      reads them); float64 takes float64 chunks, computes in float64 and returns float64
                      log_probability. Other chunk types raise TypeError.
    expansion_scores  optional scorer table, as for `ctc_ext_beam_search_decoder_raw` ([num_classes + 1,
                      num_classes], entries <= 0; float32 streams only), checked once here.
    """

    def __init__(self, batch_size, num_classes, beam_width, top_paths, max_time, merge_repeated=False,
                 blank_index=0, blank_label=-1, device=None, dtype=torch.float32, expansion_scores=None):
        if int(beam_width) < 1 or int(top_paths) < 1:
            raise ValueError("beam_width and top_paths must be >= 1")
        self.dtype = _torch_dtype(dtype)
        if self.dtype not in (torch.float32, torch.float64):
            raise TypeError("the streaming decoder computes in float32 or float64, not %s" % self.dtype)
        self._f64 = self.dtype == torch.float64
        self._lib = _lib.load()
        self.B, self.C, self.W, self.P, self.T = (int(batch_size), int(num_classes), int(beam_width),
                                                  int(top_paths), int(max_time))
        es = None
        if expansion_scores is not None:
            if self._f64:
                raise TypeError("expansion_scores is supported for float32 inputs only")
            es, _ = _as_tensor(expansion_scores)
            if tuple(es.shape) != (self.C + 1, self.C):
                raise InvalidArgumentError(8, "expansion_scores must have shape [num_classes + 1, num_classes]")
            es = es.to(dtype=torch.float32)
            if not bool((es.cpu() <= 0).all()):  # log-probabilities (NaN fails too)
                raise InvalidArgumentError(8, self._lib.ctcx_strerror(8).decode())
        if not torch.cuda.is_available():
            raise RuntimeError("ctcx: no CUDA device available and there is no CPU fallback")
        self.merge_repeated, self.blank_index, self.blank_label = (bool(merge_repeated), int(blank_index),
                                                                   int(blank_label))
        self.device = torch.device(device) if device is not None else torch.device("cuda")
        if self.device.index is None:  # (an indexed device: CUDA masks are compared with it)
            self.device = torch.device(self.device.type, torch.cuda.current_device())
        self._score_code = _lib.F64 if self._f64 else _lib.F32
        nbytes = self._lib.ctcx_stream_workspace_bytes_v(self._score_code, self.T, self.B, self.C, self.W, self.P)
        if nbytes == 0:
            raise InvalidArgumentError(8, self._lib.ctcx_strerror(8).decode())
        self._nbytes = nbytes
        self._ws = torch.empty(max(nbytes, 256), dtype=torch.uint8, device=self.device)
        self._esd = None if es is None else es.to(device=self.device).contiguous()
        self.reset()

    def _stream(self):
        return torch.cuda.current_stream(self.device).cuda_stream

    def _chunk_dtypes(self):
        return (torch.float64,) if self._f64 else (torch.float32, torch.float16, torch.bfloat16)

    def reset(self, slots=None):
        """Reset() (decoder.h:212-227): back to the empty prefix for every utterance, or, with `slots`, for
        the selected slots only (the others keep their beams). A selection is one of
          * an iterable of slot indices (list, tuple, range, ...),
          * a bool or integer mask of shape [B] (numpy array or CPU tensor; non-zero = selected),
          * a contiguous CUDA int32 [B] mask on the stream's device, used in place: no allocation, copy or
            synchronisation, so `reset(mask)` can be captured into a CUDA graph with `step_device`.
        A reset slot has consumed no frames and its flags are cleared; the stream-wide check of the scorer
        table is not repeated (it was made at construction)."""
        if slots is None:
            with torch.cuda.device(self.device):
                rc = self._lib.ctcx_stream_reset_v(self._ws.data_ptr(), self._nbytes, self._score_code, self.T,
                                                   self.B, self.C, self.W, self.P, self._stream())
            if rc != 0:
                _raise(self._lib, rc)
            return
        mask, idx = self._selection(slots, host_indices=False)
        if idx is not None and len(idx) == 0:
            return
        with torch.cuda.device(self.device):
            rc = self._lib.ctcx_stream_reset_slots(self._ws.data_ptr(), self._nbytes, self._score_code, self.T,
                                                   self.B, self.C, self.W, self.P, mask.data_ptr(), self._stream())
        if rc != 0:
            _raise(self._lib, rc)

    def _selection(self, slots, host_indices=True):
        """(device int32 [B] mask, sorted slot indices as an int64 numpy array) of a selection (see reset);
        the indices of a CUDA mask are None unless host_indices, which then reads the mask back (one
        synchronisation)."""
        B = self.B
        if isinstance(slots, torch.Tensor) and slots.is_cuda:
            if not (slots.dtype == torch.int32 and tuple(slots.shape) == (B,) and slots.is_contiguous() and
                    slots.device == self.device):
                raise InvalidArgumentError(8, "a CUDA slot mask must be a contiguous int32 [%d] tensor on %s"
                                           % (B, self.device))
            return slots, (np.flatnonzero(slots.cpu().numpy()) if host_indices else None)
        if isinstance(slots, (np.ndarray, torch.Tensor)):
            m = slots.numpy() if isinstance(slots, torch.Tensor) else slots
            if m.shape != (B,) or not (m.dtype == np.bool_ or np.issubdtype(m.dtype, np.integer)):
                raise InvalidArgumentError(8, "a slot mask must be a bool or integer array of shape [%d], got %s %s"
                                           % (B, m.dtype, m.shape))
            idx = np.flatnonzero(m)
        else:
            vals = list(slots)
            if not all(isinstance(v, (int, np.integer)) and not isinstance(v, (bool, np.bool_)) and 0 <= v < B
                       for v in vals):
                raise InvalidArgumentError(8, "slot indices must be integers in [0, %d), got %s" % (B, vals))
            idx = np.unique(np.asarray(vals, dtype=np.int64))
        mask = np.zeros(B, np.int32)
        mask[idx] = 1
        return _to_device(mask, self.device), idx.astype(np.int64)

    def _step(self, x, ln):
        """ctcx_stream_step_v on a frame-strided device chunk and device lengths; returns the code."""
        tstride = int(x.stride(0)) if int(x.shape[0]) > 1 else self.B * self.C
        return self._lib.ctcx_stream_step_v(
            self._ws.data_ptr(), self._nbytes, self.T, self.B, self.C, self.W, self.P, x.data_ptr(),
            _DTYPE_CODE[x.dtype], tstride, int(x.shape[0]), ln.data_ptr(), self.blank_index,
            None if self._esd is None else self._esd.data_ptr(), self._stream())

    def step(self, inputs, sequence_length=None):
        """Step() over a chunk: inputs [chunk_time, batch, num_classes]; sequence_length[b] = how many
        leading frames of the chunk utterance b consumes (default: all). A device chunk that is a batch
        shard `x[:, b0:b1, :]` of a contiguous tensor is read in place."""
        x, _ = _as_tensor(inputs)
        if x.dim() != 3:
            raise InvalidArgumentError(1, self._lib.ctcx_strerror(1).decode())
        if self._f64 and x.dtype != torch.float64:
            raise TypeError("a float64 stream takes float64 chunks, got %s" % x.dtype)
        if not self._f64 and x.dtype == torch.float64:
            raise TypeError("the streaming decoder computes in float32; float64 chunks would not be "
                            "bit-identical to a one-shot float64 decode -- cast explicitly, or make the "
                            "stream with dtype=torch.float64")
        Tc, B, C = (int(v) for v in x.shape)
        if B != self.B or C != self.C:
            raise InvalidArgumentError(8, "chunk shape %s does not match the stream (batch %d, classes %d)"
                                       % (tuple(x.shape), self.B, self.C))
        if Tc == 0:
            return
        with torch.cuda.device(self.device):
            dt = x.dtype if x.dtype in self._chunk_dtypes() else torch.float32
            xd = x.to(device=self.device, dtype=dt, non_blocking=True)
            if not _frame_strided(xd):
                xd = xd.contiguous()
            if sequence_length is None:
                ld = torch.full((B,), Tc, dtype=torch.int32, device=self.device)
            else:
                l, _ = _as_tensor(np.asarray(sequence_length, dtype=np.int32)
                                  if not isinstance(sequence_length, torch.Tensor) else sequence_length)
                if l.dim() != 1 or int(l.shape[0]) != B:
                    raise FailedPreconditionError(4, "len(sequence_length) != batch_size.  ")
                if bool((l.to("cpu") > Tc).any()) or bool((l.to("cpu") < 0).any()):
                    raise FailedPreconditionError(5, "sequence_length(b) <= %d" % Tc)
                ld = l.to(device=self.device, dtype=torch.int32).contiguous()
            rc = self._step(xd, ld)
            if rc == 9 and xd.dtype in (torch.float16, torch.bfloat16):
                # a table with half-precision chunks where the kernel has no room to widen them (as in the
                # one-shot decode), or the test hook's generic kernel forced onto a fast-path shape
                xd = xd.float().contiguous()
                rc = self._step(xd, ld)
            # the kernels read xd / ld asynchronously on this stream; keep them alive until then
            xd.record_stream(torch.cuda.current_stream(self.device))
            ld.record_stream(torch.cuda.current_stream(self.device))
        if rc != 0:
            _raise(self._lib, rc)

    def step_device(self, inputs_dev, lengths_dev):
        """Step() on buffers that already live on the device -- a [chunk_time, batch, num_classes] chunk of
        one of the stream's chunk types (contiguous, or a batch shard of a contiguous tensor) and int32
        [batch] lengths -- without any conversion, allocation or synchronisation: the call only enqueues
        kernels on the current stream, so it can be captured into a CUDA graph
        (`with torch.cuda.graph(g): dec.step_device(x_static, len_static)`) and replayed per chunk,
        which removes the launch overhead that dominates small chunks. Half-precision chunks with a
        scorer table raise UnsupportedError where `step()` would widen them."""
        x, ln = inputs_dev, lengths_dev
        if not (x.is_cuda and x.dtype in self._chunk_dtypes() and x.dim() == 3 and _frame_strided(x) and
                int(x.shape[1]) == self.B and int(x.shape[2]) == self.C):
            raise InvalidArgumentError(8, "step_device needs a frame-strided CUDA %s [chunk_time, %d, %d] tensor"
                                       % ("/".join(str(d) for d in self._chunk_dtypes()), self.B, self.C))
        if not (ln.is_cuda and ln.dtype == torch.int32 and ln.is_contiguous() and tuple(ln.shape) == (self.B,)):
            raise InvalidArgumentError(8, "step_device needs a contiguous CUDA int32 [%d] tensor" % self.B)
        rc = self._step(x, ln)
        if rc != 0:
            _raise(self._lib, rc)

    def top_paths_raw(self, slots=None, wait=True):
        """TopPaths() (decoder.h:229-261) of the frames consumed so far, as the raw 7 output groups
        (device tensors; log_probability in the stream's score type). Does not disturb the state.

        slots   None: every utterance. Otherwise a selection (see reset): the reference's format for the
                selected slots only, in ascending slot order -- batch index i is the i-th selected slot,
                dense_shape[0] = n, log_probability [n, top_paths], `.slots` = the slot indices. A CUDA mask
                is read back to learn them (one synchronisation). Over-fed slots, too few leaves and mixed
                score types are reported for selected slots only.
        wait    False: return a PendingDecode once the read is enqueued on the current stream; it reflects
                the steps enqueued before this call, so the next chunk can be stepped (and the slots reset)
                before `.result()` is read."""
        full = slots is None
        if full and wait:
            return self._read(None, None, True)
        mask, idx = self._selection(slots) if not full else (self._all_slots(), None)
        return self._read(mask, idx, wait)

    def _all_slots(self):
        if getattr(self, "_ones", None) is None:
            self._ones = torch.ones((self.B,), dtype=torch.int32, device=self.device)
        return self._ones

    def _read(self, mask, idx, wait):
        """ctcx_stream_top_paths (mask None) or ctcx_stream_top_paths_slots, packed; idx = the selected slots
        whose rows are kept (None: all rows)."""
        lib, T, B, P, f64 = self._lib, self.T, self.B, self.P, self._f64
        n = B if idx is None else len(idx)
        if n == 0:
            res = self._empty_result()
            return res if wait else PendingDecode(lambda: res)
        arr = ctypes.c_int64 * P
        n_dec, max_dec, n_ali, max_ali = arr(), arr(), arr(), arr()
        sizes = _lib.CtcxSizes(n_dec, max_dec, n_ali, max_ali)
        flags = ctypes.c_int32(0)
        ws, stream, attrs = self._ws.data_ptr(), self._stream(), (int(self.merge_repeated), self.blank_label)
        # the one-shot decode's choice of route: the deferred one (one buffer of the upper bound, read later)
        # up to DEFER_MAX_BYTES_DEVICE; beyond it the sizes first, then exactly sized outputs -- done at
        # once, so that the result still reflects the steps enqueued before this call
        n_bound = _bound_elems(T, B, P, torch.full((n,), T, dtype=torch.int32), f64)  # <= T frames per slot
        deferred = not wait and 8 * n_bound <= DEFER_MAX_BYTES_DEVICE

        def now():
            with torch.cuda.device(self.device):
                if mask is None:
                    rc = lib.ctcx_stream_top_paths(ws, T, B, self.C, self.W, P, *attrs, stream, ctypes.byref(sizes),
                                                   ctypes.byref(flags))
                else:
                    rc = lib.ctcx_stream_top_paths_slots(ws, T, B, self.C, self.W, P, *attrs, mask.data_ptr(), stream,
                                                         ctypes.byref(sizes), ctypes.byref(flags))
                if rc != 0:
                    _raise(lib, rc)
                groups, logp, _ = _pack(lib, self._ws, T, B, P, (n_dec, n_ali), self.device, stream, f64)
                return self._rows(groups, logp, idx, int(flags.value))

        if not deferred:
            return now() if wait else PendingDecode(now, eager=True)
        with torch.cuda.device(self.device):
            # deferred, as a deferred one-shot decode: trace, then -- before any later step or reset rewrites
            # the final beam -- compact pack, result block into page-locked memory, an event
            rc = lib.ctcx_stream_top_paths_slots(ws, T, B, self.C, self.W, P, *attrs, mask.data_ptr(), stream,
                                                 None, None)
            if rc != 0:
                _raise(lib, rc)
            buf = torch.empty((n_bound,), dtype=torch.int64, device=self.device)
            rc = lib.ctcx_pack_compact(ws, T, B, P, 8 if f64 else 4, buf.data_ptr(), n_bound, stream)
            if rc != 0:
                _raise(lib, rc)
            n_res = lib.ctcx_result_bytes(P)
            hres = torch.empty((n_res,), dtype=torch.uint8, pin_memory=True)
            rc = lib.ctcx_result_copy_async(ws, T, B, P, hres.data_ptr(), n_res, stream)
            if rc != 0:
                _raise(lib, rc)
            done = torch.cuda.Event()
            done.record(torch.cuda.current_stream(self.device))

        def complete():
            with torch.cuda.device(self.device):
                done.synchronize()
                rc = lib.ctcx_result_parse(hres.data_ptr(), T, B, P, ctypes.byref(sizes), ctypes.byref(flags))
                if rc != 0:
                    _raise(lib, rc)
                groups, logp = _carve(buf[:_pack_elems(B, P, (n_dec, n_ali), f64)], B, P, (n_dec, n_ali), f64)
                return self._rows(groups, logp, idx, int(flags.value))

        return PendingDecode(complete)

    def _rows(self, groups, logp, idx, flags):
        """The raw result of the whole batch -> the rows of the slots idx (None: all), renumbered on the
        device: batch column i = the i-th selected slot."""
        if idx is not None:
            n = len(idx)
            lookup = np.full(self.B, -1, np.int64)
            lookup[idx] = np.arange(n)
            lookup = _to_device(lookup, self.device)
            for p in range(self.P):
                for g in (0, 3):
                    if groups[g][p].shape[0]:
                        groups[g][p][:, 0] = lookup[groups[g][p][:, 0]]
                groups[2][p][0] = n
                groups[5][p][0] = n
            logp = logp[_to_device(idx, self.device)]
        res = CTCExtBeamSearchDecoder(*groups, logp)
        res.flags = flags
        res.slots = idx
        return res

    def _empty_result(self):
        dev, P = self.device, self.P
        e = lambda *shape: torch.zeros(shape, dtype=torch.int64, device=dev)  # noqa: E731
        groups = [[e(0, 2) for _ in range(P)], [e(0) for _ in range(P)], [e(2) for _ in range(P)],
                  [e(0, 2) for _ in range(P)], [e(0) for _ in range(P)], [e(2) for _ in range(P)]]
        res = CTCExtBeamSearchDecoder(*groups, torch.zeros((0, P), dtype=self.dtype, device=dev))
        res.slots = np.zeros(0, np.int64)
        return res

    def top_paths(self, slots=None, wait=True):
        """`(decoded, alignment, log_probability)` of top_paths_raw(slots, wait), `.slots` and `.flags`
        attached; with wait=False a PendingDecode of it."""
        def convert(raw):
            decoded = [SparseTensor(i, v, s) for i, v, s in zip(raw[0], raw[1], raw[2])]
            alignment = [SparseTensor(i, v, s) for i, v, s in zip(raw[3], raw[4], raw[5])]
            out = DecodeResult((decoded, alignment, raw[6]))
            out.flags = raw.flags
            out.slots = raw.slots
            return out

        raw = self.top_paths_raw(slots, wait)
        return convert(raw) if wait else PendingDecode(lambda: convert(raw.result()))


def decode_host_cabi(inputs, sequence_length, beam_width, top_paths, merge_repeated=False,
                     blank_index=0, blank_label=-1, device=0):
    """The host-buffer C-ABI entry (ctcx_decode_host_f32, or ctcx_decode_host_f64 for float64
    inputs) exactly as a TensorFlow CPU OpKernel would call it: numpy in, numpy out, all copies inside
    the call."""
    lib = _lib.load()
    f64 = np.asarray(inputs).dtype == np.float64
    x = np.ascontiguousarray(inputs, dtype=np.float64 if f64 else np.float32)
    if x.ndim != 3:
        raise InvalidArgumentError(1, lib.ctcx_strerror(1).decode())
    seq = np.ascontiguousarray(sequence_length, dtype=np.int32)
    if seq.ndim != 1:
        raise InvalidArgumentError(3, lib.ctcx_strerror(3).decode())
    T, B, C = x.shape
    if seq.shape[0] != B:
        raise FailedPreconditionError(
            4, "len(sequence_length) != batch_size.  len(sequence_length):  %d batch_size: %d"
            % (seq.shape[0], B))
    res = ctypes.POINTER(_lib.CtcxHostResult)()
    entry = lib.ctcx_decode_host_f64 if f64 else lib.ctcx_decode_host_f32
    rc = entry(x.ctypes.data, T, B, C, seq.ctypes.data, int(beam_width), int(top_paths),
               int(bool(merge_repeated)), int(blank_index), int(blank_label), int(device), ctypes.byref(res))
    if rc != 0:
        _raise(lib, rc)
    try:
        r = res.contents
        P = r.top_paths

        def arr(pp, n):
            return np.ctypeslib.as_array(pp, shape=(n,)).copy() if n else np.zeros((0,), np.int64)

        out = [[], [], [], [], [], []]
        for p in range(P):
            nd, na = int(r.n_decoded[p]), int(r.n_alignment[p])
            out[0].append(arr(r.decoded_indices[p], nd * 2).reshape(nd, 2))
            out[1].append(arr(r.decoded_values[p], nd))
            out[2].append(arr(r.decoded_shape[p], 2))
            out[3].append(arr(r.alignment_indices[p], na * 2).reshape(na, 2))
            out[4].append(arr(r.alignment_values[p], na))
            out[5].append(arr(r.alignment_shape[p], 2))
        lp_ptr = r.log_probability_f64 if f64 else r.log_probability
        logp = (np.ctypeslib.as_array(lp_ptr, shape=(B * P,)).copy().reshape(B, P)
                if B * P else np.zeros((B, P), np.float64 if f64 else np.float32))
    finally:
        lib.ctcx_free_host(res)
    return CTCExtBeamSearchDecoder(*out, logp)
