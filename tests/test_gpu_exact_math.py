"""The layer under the bit-exact scores, checked completely or densely on the device.

* Float math (csrc/ctcx_math.cuh): expf, log1pf, logf and the float LogSumExp on every float of the
  domains the decoder uses, against glibc 2.39 called from C (oracle/libm_port_check.c), in chunks of
  2^26 inputs built on the device from their bit patterns.
* Double math: exp and log at every reduction-cell and table sub-interval edge of their domains, plus
  2^27 pseudo-random arguments each; the double LogSumExp on every float difference in [-104, 0].
* The normaliser kernels of the generic path (LogNormRowKernel, LogNormKernel, LogNormKernelF64) and
  the wide path's fused pre-pass (NormTopClassesKernel, every element type and register tier) through
  ctcx_debug_prepass, against a plain host restatement of decoder.h:71-80 with the same libm: the
  normaliser and the per-frame sorted class list, bit for bit.

The device functions restate glibc 2.39 operation for operation, so these tests need that glibc on
the host: on any other version they fail rather than skip.
"""
import ctypes
import math
import os
from concurrent.futures import ThreadPoolExecutor

import numpy as np
import pytest

import ctcx_testlib as L

pytestmark = pytest.mark.gpu

CHUNK = 1 << 26      # inputs per device launch of a sweep
SUB = 1 << 22        # inputs per host comparison task
THREADS = max(1, min(64, len(os.sched_getaffinity(0))))
SHOW = 16            # mismatching inputs listed in a failure message

_fp = ctypes.POINTER(ctypes.c_float)
_dp = ctypes.POINTER(ctypes.c_double)
_u32p = ctypes.POINTER(ctypes.c_uint32)


def _bits32(x):
    return int(np.float32(x).view(np.uint32))


def _bits64(x):
    return int(np.float64(x).view(np.uint64))


@pytest.fixture(scope="module")
def libs():
    """(device library, host libm checker) once the host is known to run the glibc the device
    code restates."""
    import torch
    if not torch.cuda.is_available():
        pytest.skip("no CUDA device")
    ver = os.confstr("CS_GNU_LIBC_VERSION") or ""
    assert ver == "glibc 2.39", (
        "the device math restates glibc 2.39's expf/log1pf/logf/exp/log; this host runs %r, so it "
        "cannot serve as the reference" % ver)
    from ctc_beam_search_op_b200 import _lib
    cpu = ctypes.CDLL(L.ORACLE_SO)
    cpu.ctcx_libm_mismatches_f32.restype = ctypes.c_longlong
    cpu.ctcx_libm_mismatches_f32.argtypes = [ctypes.c_int, ctypes.c_uint32, ctypes.c_longlong, _fp, _u32p,
                                             ctypes.c_int]
    for f in (cpu.ctcx_libm_expf_v, cpu.ctcx_libm_log1pf_v, cpu.ctcx_libm_logf_v):
        f.argtypes = [_fp, _fp, ctypes.c_int]
    for f in (cpu.ctcx_libm_exp_v, cpu.ctcx_libm_log_v):
        f.argtypes = [_dp, _dp, ctypes.c_int]
    return _lib.load(), cpu


class _Tally:
    """Mismatch count and the lowest mismatching inputs of a sweep whose parts finish in any order."""

    def __init__(self, what):
        self.what, self.n, self.bad, self.checked = what, 0, [], 0

    def add(self, n, bad, checked):
        self.n += n
        self.bad.extend(int(b) for b in bad)
        self.checked += checked

    def check(self, fmt):
        bad = sorted(set(self.bad))[:SHOW]
        assert self.n == 0, "%s: %d of %d inputs differ; first: %s" % (
            self.what, self.n, self.checked, ", ".join(fmt(b) for b in bad))


def _hex32(u):
    return "0x%08x" % u


def _hex64(u):
    return "0x%016x" % u


def _x32(u0, n):
    """Device float32 tensor of the floats with bit patterns u0 ... u0+n-1 (not crossing 2^31)."""
    import torch
    s0 = u0 - (1 << 32) if u0 >= (1 << 31) else u0
    assert (s0 < 0 and s0 + n <= 0) or (s0 >= 0 and s0 + n <= (1 << 31))
    return torch.arange(s0, s0 + n, dtype=torch.int64, device="cuda").to(torch.int32).view(torch.float32)


def _dev32(lib, op, x):
    import torch
    y = torch.empty_like(x)
    assert lib.ctcx_debug_math_f32(op, x.data_ptr(), y.data_ptr(), x.numel(), None) == 0
    return y


def _dev64(lib, op, x):
    import torch
    y = torch.empty_like(x)
    assert lib.ctcx_debug_math_f64(op, x.data_ptr(), y.data_ptr(), x.numel(), None) == 0
    return y


def _libm_task(cpu, op, u0, got):
    """Host task: got (float32 results at bit patterns u0 ...) against libm."""
    first = np.zeros(SHOW, np.uint32)
    n = cpu.ctcx_libm_mismatches_f32(op, u0, len(got), got.ctypes.data_as(_fp), first.ctypes.data_as(_u32p), SHOW)
    assert n >= 0
    return n, first[:min(n, SHOW)], len(got)


def _sweep_f32(u_lo, u_hi, device_chunk, host_tasks):
    """Every bit pattern in [u_lo, u_hi]: device_chunk(u0, n) -> host arrays; host_tasks(u0, arrays)
    -> a list of (tally, callable) run on the pool, one per SUB inputs. The device computes the next
    chunk while the host checks the previous one; at most two chunks are held on the host."""
    chunks = []
    with ThreadPoolExecutor(THREADS) as pool:
        for u0 in range(u_lo, u_hi + 1, CHUNK):
            n = min(CHUNK, u_hi + 1 - u0)
            outs = device_chunk(u0, n)
            chunks.append([(tally, pool.submit(fn)) for s in range(0, n, SUB)
                           for tally, fn in host_tasks(u0 + s, [o[s:s + SUB] for o in outs])])
            if len(chunks) > 1:
                for tally, fut in chunks.pop(0):
                    tally.add(*fut.result())
        for tally, fut in (p for c in chunks for p in c):
            tally.add(*fut.result())


def _sweep_libm(lib, cpu, op, u_lo, u_hi, tally):
    def device_chunk(u0, n):
        return [_dev32(lib, op, _x32(u0, n)).cpu().numpy()]
    _sweep_f32(u_lo, u_hi, device_chunk,
               lambda u0, outs: [(tally, lambda u0=u0, g=outs[0]: _libm_task(cpu, op, u0, g))])


def _libm_values(lib, cpu, op, xs):
    """Device op on a few float32 inputs, against libm; returns (count, bad bit patterns, n)."""
    import torch
    xs = np.ascontiguousarray(xs, np.float32)
    got = _dev32(lib, op, torch.from_numpy(xs).cuda()).cpu().numpy()
    n, bad = 0, []
    for u, g in zip(xs.view(np.uint32).tolist(), got):
        k, first, _ = _libm_task(cpu, op, u, np.array([g], np.float32))
        n += k
        bad += first.tolist()
    return n, bad, len(xs)


# ------------------------------------------------------------------------------------------------
# 1. float math, exhaustively
def test_expf_every_float_in_its_domain(libs):
    """ExpfExact == glibc expf on every float in [-200, -0] and -inf; +0 for every float below -200."""
    import torch
    lib, cpu = libs
    t = _Tally("expf")
    _sweep_libm(lib, cpu, 0, _bits32(-0.0), _bits32(-200.0), t)
    t.add(*_libm_values(lib, cpu, 0, [-np.inf]))
    t.check(_hex32)
    # below -200 (underflow to +0, the device's first branch): checked on the device
    lo, hi = _bits32(-200.0) + 1, _bits32(-np.inf)
    nonzero, first = 0, None
    for u0 in range(lo, hi + 1, CHUNK):
        n = min(CHUNK, hi + 1 - u0)
        y = _dev32(lib, 0, _x32(u0, n)).view(torch.int32)
        nz = (y != 0).nonzero()
        if nz.numel():
            nonzero += nz.numel()
            first = first if first is not None else u0 + int(nz[0, 0])
    assert nonzero == 0, "expf below -200: %d results are not +0; first input %s" % (nonzero, _hex32(first))


def test_log1pf_every_float_in_its_domain(libs):
    """Log1pfExact == glibc log1pf on every float in [+0, 1], which includes the |x| < 2^-29 early
    returns and the hu == 0 branch LogSumExp takes whenever two scores are ~14 nats apart."""
    lib, cpu = libs
    t = _Tally("log1pf")
    _sweep_libm(lib, cpu, 1, _bits32(0.0), _bits32(1.0), t)
    t.check(_hex32)


def test_logf_every_float_in_its_domain(libs):
    """LogfExact == glibc logf on every float in [1, 65536): every normaliser sum up to C = 65535."""
    lib, cpu = libs
    t = _Tally("logf")
    _sweep_libm(lib, cpu, 2, _bits32(1.0), _bits32(65536.0) - 1, t)
    t.check(_hex32)


def test_logsumexp_every_float_difference(libs):
    """LogSumExp(x, 0) and LogSumExp(0, x) in float == util/ctc_loss_util.h:33-41 with glibc on every
    float x in [-104, -0]; the double LogSumExp (the T = double path) at x = d and x = -d for the same
    d equals d's float term widened, plus -d. Edges: +0, both -inf shortcuts, x > 0 (the other arm)."""
    import torch
    lib, cpu = libs
    t32, t_sw, t64 = _Tally("float LogSumExp(x, 0)"), _Tally("float LogSumExp(0, x) vs (x, 0)"), \
        _Tally("double LogSumExp(x, 0) at x = d, -d")

    def device_chunk(u0, n):
        x = _x32(u0, n)
        xd = x.double()
        return [_dev32(lib, 3, x).cpu().numpy(), _dev32(lib, 4, x).cpu().numpy(),
                _dev64(lib, 2, xd).cpu().numpy(), _dev64(lib, 2, -xd).cpu().numpy()]

    def swapped(u0, y3, y4):
        bad = np.nonzero(y3.view(np.uint32) != y4.view(np.uint32))[0]
        return len(bad), (u0 + bad[:SHOW]).tolist(), len(y3)

    def f64(u0, y3, pos, neg):
        d = np.arange(u0, u0 + len(y3), dtype=np.uint64).astype(np.uint32).view(np.float32).astype(np.float64)
        term = y3.astype(np.float64)  # validated against libm by the float task of the same inputs
        bad = np.nonzero((pos.view(np.uint64) != term.view(np.uint64)) |
                         (neg.view(np.uint64) != (-d + term).view(np.uint64)))[0]
        return len(bad), (u0 + bad[:SHOW]).tolist(), len(y3)

    def host_tasks(u0, o):
        return [(t32, lambda: _libm_task(cpu, 3, u0, o[0])), (t_sw, lambda: swapped(u0, o[0], o[1])),
                (t64, lambda: f64(u0, o[0], o[2], o[3]))]

    _sweep_f32(_bits32(-0.0), _bits32(-104.0), device_chunk, host_tasks)
    # +0 (x == 0), -inf (the a == -inf and b == -inf shortcuts) and x > 0 (hi = x): denormals, [0.5, 1),
    # [64, 104], large and infinite arguments
    edges = np.concatenate([
        np.array([0.0, -np.inf, np.inf, 1e30, np.finfo(np.float32).max, 200.0, 104.5], np.float32),
        np.arange(1, 1 << 20, dtype=np.uint32).view(np.float32),
        np.arange(_bits32(0.5), _bits32(1.0), dtype=np.uint32).view(np.float32),
        np.arange(_bits32(64.0), _bits32(104.0) + 1, dtype=np.uint32).view(np.float32)])
    for op in (3, 4):
        xs = torch.from_numpy(edges).cuda()
        got = _dev32(lib, op, xs).cpu().numpy()
        first = np.zeros(SHOW, np.uint32)
        # contiguous bit-pattern runs of `edges` go to the C checker one run at a time
        u = edges.view(np.uint32).astype(np.int64)
        cuts = np.nonzero(np.diff(u) != 1)[0] + 1
        for a, b in zip(np.r_[0, cuts], np.r_[cuts, len(u)]):
            n = cpu.ctcx_libm_mismatches_f32(op, int(u[a]), int(b - a), got[a:b].ctypes.data_as(_fp),
                                             first.ctypes.data_as(_u32p), SHOW)
            t32.add(n, first[:min(n, SHOW)].tolist(), int(b - a))
    xd = torch.tensor([0.0, -0.0, -np.inf], dtype=torch.float64).cuda()
    got = _dev64(lib, 2, xd).cpu().numpy()
    ln2f = _libm_v(cpu.ctcx_libm_log1pf_v, np.ones(1, np.float32), _fp).astype(np.float64)[0]  # log1pf(expf(0))
    want = np.array([ln2f, ln2f, 0.0])
    t64.add(int((got.view(np.uint64) != want.view(np.uint64)).sum()), [], 3)
    for t in (t32, t_sw, t64):
        t.check(_hex32)


# ------------------------------------------------------------------------------------------------
# 2. double math, densely
def _splitmix64(seed, start, n):
    """Outputs start+1 ... start+n of splitmix64 seeded with `seed` (oracle/libm_port_check.c)."""
    with np.errstate(over="ignore"):
        z = np.uint64(seed) + np.arange(start + 1, start + n + 1, dtype=np.uint64) * np.uint64(0x9E3779B97F4A7C15)
        z = (z ^ (z >> np.uint64(30))) * np.uint64(0xBF58476D1CE4E5B9)
        z = (z ^ (z >> np.uint64(27))) * np.uint64(0x94D049BB133111EB)
    return z ^ (z >> np.uint64(31))


def _around(centres_bits, ulps=4):
    c = np.asarray(centres_bits, np.uint64)
    with np.errstate(over="ignore"):  # (-k as uint64: the sum wraps to the pattern k below)
        d = np.arange(-ulps, ulps + 1, dtype=np.int64).astype(np.uint64)
        return (c[:, None] + d[None, :]).ravel().view(np.float64)


def _check_f64(lib, cpu, op, chunks, what):
    """Device op 0 (exp) / 1 (log) on every array of `chunks` against glibc exp / log."""
    import torch
    libm = cpu.ctcx_libm_exp_v if op == 0 else cpu.ctcx_libm_log_v
    t = _Tally(what)

    def task(xs, got):
        want = np.empty_like(xs)
        libm(xs.ctypes.data_as(_dp), want.ctypes.data_as(_dp), len(xs))
        if op == 0:
            want[xs <= -512.0] = 0.0  # documented: below 1e-222 the device returns 0
        bad = np.nonzero(want.view(np.uint64) != got.view(np.uint64))[0]
        return len(bad), xs[bad[:SHOW]].view(np.uint64).tolist(), len(xs)

    with ThreadPoolExecutor(THREADS) as pool:
        futs = []
        for xs in chunks:
            xs = np.ascontiguousarray(xs, np.float64)
            got = _dev64(lib, op, torch.from_numpy(xs).cuda()).cpu().numpy()
            futs += [pool.submit(task, xs[s:s + SUB], got[s:s + SUB]) for s in range(0, len(xs), SUB)]
            while len(futs) > 4 * THREADS:
                t.add(*futs.pop(0).result())
        for f in futs:
            t.add(*f.result())
    t.check(_hex64)


def _old_f64_inputs():
    """The inputs of the earlier sampled test, kept."""
    rng = np.random.default_rng(6)
    n = 400000
    xe = np.concatenate([-np.abs(rng.standard_normal(n) * 25), -rng.random(n) * 512, -10.0 ** rng.uniform(-20, 2.7, n),
                         [0.0, -0.0, -1e-300, -1e-17, -511.99, -512.0, -600.0, -745.2, -1e4, -np.inf]])
    xl = np.concatenate([1 + rng.random(n) * 0.07, 1 + rng.random(n) * 70000, 1 + 10.0 ** rng.uniform(-16, 0, n),
                         [1.0, 1.0 + 2 ** -52, 1.0647, 1.065, 2.0, 29.0, 1024.0, 65535.0]])
    xs = np.concatenate([rng.standard_normal(n) * 20, rng.standard_normal(n) * 1e-3, [0.0, 1e-9, -1e-9, 104.0, -104.0]])
    return xe, xl, xs


N_RANDOM_F64 = 1 << 27


def test_exp_f64_cell_edges_and_random(libs):
    """ExpExactD == glibc exp on (-512, 0]: +-4 ulps around every reduction-cell boundary
    (k + 1/2) ln2/128, the abstop edges, 2^27 splitmix64 arguments (half uniform in value, half
    uniform in bit pattern); 0 for x <= -512 and -inf."""
    lib, cpu = libs
    k = np.arange(-94549, 0, dtype=np.float64)
    b = (k + 0.5) * (math.log(2) / 128)
    cells = _around(b[b > -512.0].view(np.uint64))
    cells = cells[(cells > -512.0) & (cells <= 0.0)]
    edges = np.concatenate([_around([_bits64(-2.0 ** -54), _bits64(-512.0), _bits64(-2.0 ** -1022)]),
                            [0.0, -0.0, -np.inf, -5e-324, -1e-300, -2.0 ** -60]])
    edges = edges[edges <= 0.0]
    xe, _, _ = _old_f64_inputs()
    lo_e, hi_e = _bits64(-2.0 ** -60), _bits64(-511.99)

    def random_chunks():
        half = N_RANDOM_F64 // 2
        for s in range(0, half, 1 << 24):
            z = _splitmix64(7, 2 * s, 2 * (1 << 24))
            yield -512.0 * ((z[0::2] >> np.uint64(11)).astype(np.float64) * 2.0 ** -53)
            yield (np.uint64(lo_e) + z[1::2] % np.uint64(hi_e - lo_e)).view(np.float64)

    _check_f64(lib, cpu, 0, [cells, edges, xe] + list(random_chunks()), "double exp")


def test_log_f64_table_edges_and_random(libs):
    """LogExactD == glibc log on [1, 65536): +-4 ulps at the 128 table sub-interval edges of all 16
    binades and at both edges of the near-1 polynomial window, 1 + n 2^-52 for n < 2^16, 2^22
    arguments inside the window and 2^27 uniform in bit pattern."""
    lib, cpu = libs
    off, sub = 0x3fe6000000000000, 1 << 45
    lo_l, hi_l = _bits64(1.0), _bits64(65536.0)
    table = _around([off + m * sub for m in range((lo_l - off) // sub, (hi_l - off) // sub)])
    window = _around([0x3fee000000000000, 0x3fee000000000000 + 0x3090000000000])
    near1 = 1.0 + np.arange(1 << 16, dtype=np.float64) * 2.0 ** -52
    _, xl, _ = _old_f64_inputs()
    hi_n = 0x3fee000000000000 + 0x3090000000000
    z = _splitmix64(8, 0, 1 << 22)
    in_window = (np.uint64(lo_l) + z % np.uint64(hi_n - lo_l)).view(np.float64)

    def random_chunks():
        for s in range(0, N_RANDOM_F64, 1 << 24):
            z = _splitmix64(9, s, 1 << 24)
            yield (np.uint64(lo_l) + z % np.uint64(hi_l - lo_l)).view(np.float64)

    table = table[(table >= 1.0) & (table < 65536.0)]
    assert len(table) == 16 * 128 * 9 - 4  # (the 4 below 1.0 dropped)
    _check_f64(lib, cpu, 1, [table, window, near1, in_window, xl] + list(random_chunks()), "double log")


def test_logsumexp_f64_sampled_arguments(libs):
    """The double LogSumExp(x, 0) on the arguments of the earlier sampled test, against
    max(x, 0) + log1pf(expf(-|x| as float)) from glibc (the exhaustive float differences are in
    test_logsumexp_every_float_difference)."""
    import torch
    lib, cpu = libs
    _, _, xs = _old_f64_inputs()
    d32 = (-np.abs(xs)).astype(np.float32)
    e = np.empty_like(d32)
    cpu.ctcx_libm_expf_v(d32.ctypes.data_as(_fp), e.ctypes.data_as(_fp), len(d32))
    l1 = np.empty_like(d32)
    cpu.ctcx_libm_log1pf_v(e.ctypes.data_as(_fp), l1.ctypes.data_as(_fp), len(d32))
    want = np.maximum(xs, 0.0) + l1.astype(np.float64)
    got = _dev64(lib, 2, torch.from_numpy(np.ascontiguousarray(xs)).cuda()).cpu().numpy()
    np.testing.assert_array_equal(got.view(np.uint64), want.view(np.uint64))


# ------------------------------------------------------------------------------------------------
# 3. the normaliser kernels
DT = {"f32": (0, "float32"), "f16": (1, "float16"), "bf16": (2, "bfloat16"), "f64": (3, "float64")}
ROUTE1_C = [33, 63, 64, 65, 127, 128, 129, 256, 257, 512, 513, 1023, 1024, 1025, 2048]
ROUTE0_C = [2, 29, 32] + ROUTE1_C + [2049, 4097, 65535]
N_FAMILIES = 6


def _rows(rng, R, C, blank, dtype):
    """R rows of C logits cycling through the value families: gaussian; one sharp class (+40: every
    other term underflows against it, the sum is exactly 1); constant (the sum is exactly C); three
    quantised levels (ties straddling the Ke cut); offsets of +-1e4; -inf masked classes with a
    finite blank (every second such row masks every class but the blank)."""
    x = rng.standard_normal((R, C)) * 3
    for r in range(R):
        fam, k = r % N_FAMILIES, r // N_FAMILIES
        if fam == 1:
            x[r] = rng.standard_normal(C)
            x[r, rng.integers(C)] += 40.0
        elif fam == 2:
            x[r] = rng.uniform(-5, 5)
        elif fam == 3:
            x[r] = rng.integers(0, 3, C) * -1.5
        elif fam == 4:
            x[r] += 1e4 if k % 2 == 0 else -1e4
        elif fam == 5:
            mask = rng.random(C) < 0.5 if k % 2 == 0 else np.ones(C, bool)
            mask[blank] = False
            x[r, mask] = -np.inf
    return x.astype(np.float64 if dtype == "float64" else np.float32)


def _libm_v(fn, a, ptr):
    a = np.ascontiguousarray(a)
    out = np.empty_like(a)
    fn(a.ctypes.data_as(ptr), out.ctypes.data_as(ptr), a.size)
    return out


def _ref_off(cpu, xw):
    """decoder.h:71-80: max + log(sum of exp(x_j - max) added one term at a time in class order)."""
    if xw.dtype == np.float64:
        exp, log, ptr = cpu.ctcx_libm_exp_v, cpu.ctcx_libm_log_v, _dp
    else:
        exp, log, ptr = cpu.ctcx_libm_expf_v, cpu.ctcx_libm_logf_v, _fp
    mx = xw.max(axis=1)
    e = _libm_v(exp, xw - mx[:, None], ptr)
    s = np.add.accumulate(e, axis=1)[:, -1]  # sequential, not pairwise
    return mx + _libm_v(log, s, ptr)


def _ref_sorted(xw, off, blank, Ke, Ks):
    """The non-blank classes by (x_l - off desc, class asc) in float32, first Ke, then (-inf, 0xffff)."""
    R, C = xw.shape
    pl = (xw - off[:, None]) + np.float32(0.0)  # (+0: the order does not tell -0 from +0)
    u = pl.view(np.uint32)
    key = np.where(u & np.uint32(0x80000000), ~u, u | np.uint32(0x80000000))
    comp = ((~key).astype(np.uint64) << np.uint64(16)) | np.arange(C, dtype=np.uint64)[None, :]
    comp[:, blank] = np.uint64(0xFFFFFFFFFFFFFFFF)
    cls = (np.sort(comp, axis=1)[:, :Ke] & np.uint64(0xffff)).astype(np.int64)
    srt_pl = np.full((R, Ks), -np.inf, np.float32)
    srt_cls = np.full((R, Ks), 0xffff, np.uint16)
    srt_pl[:, :Ke] = np.take_along_axis(pl, cls, axis=1)
    srt_cls[:, :Ke] = cls
    return srt_pl, srt_cls


def _prepass(lib, route, xt, B_shard, b0, blank, W):
    """Runs the hook on xt[:, b0:b0+B_shard, :] (a strided view when the shard is narrower)."""
    import torch
    T, Bf, C = xt.shape
    dt = {torch.float32: 0, torch.float16: 1, torch.bfloat16: 2, torch.float64: 3}[xt.dtype]
    rows = T * B_shard
    off = torch.empty(rows, dtype=torch.float64 if dt == 3 else torch.float32, device="cuda")
    ks = ctypes.c_int(-1)
    Ks = (min(C - 1, 2 * W + 3) + 7) // 8 * 8 if route == 1 else 0
    pl = torch.empty(max(rows * Ks, 1), dtype=torch.float32, device="cuda")
    cls = torch.empty(max(rows * Ks, 1), dtype=torch.int16, device="cuda")
    base = xt.data_ptr() + b0 * C * xt.element_size()
    rc = lib.ctcx_debug_prepass(route, base, dt, T, B_shard, C, Bf * C, blank, W, off.data_ptr(),
                                pl.data_ptr() if route == 1 else None, cls.data_ptr() if route == 1 else None,
                                ctypes.byref(ks), None)
    assert rc == 0, "ctcx_debug_prepass: %s" % lib.ctcx_strerror(rc).decode()
    assert ks.value == Ks
    torch.cuda.synchronize()
    return (off.cpu().numpy(), pl.cpu().numpy()[:rows * Ks].reshape(rows, Ks),
            cls.cpu().numpy().view(np.uint16)[:rows * Ks].reshape(rows, Ks))


def _check_prepass(lib, cpu, route, x, dtype, blank, W, layouts=("dense", "shard"), what=""):
    """x: [T, B, C] values (float32 or float64) -> both layouts on the device against the host."""
    import torch
    T, B, C = x.shape
    tdt = getattr(torch, dtype)
    xt = torch.from_numpy(x).to(tdt)
    xw = xt.to(torch.float64 if dtype == "float64" else torch.float32).numpy().reshape(T * B, C)  # exact widening
    off = _ref_off(cpu, xw)
    if route == 1:
        Ke = min(C - 1, 2 * W + 3)
        srt = _ref_sorted(xw, off, blank, Ke, (Ke + 7) // 8 * 8)
    for layout in layouts:
        if layout == "dense":
            dev, b0, Bf = xt.cuda(), 0, B
        else:  # a batch shard of a wider tensor whose other utterances are NaN
            Bf, b0 = B + 3, 2
            full = torch.full((T, Bf, C), float("nan"), dtype=tdt)
            full[:, b0:b0 + B] = xt
            dev = full.cuda()
        got = _prepass(lib, route, dev, B, b0, blank, W)
        tag = "%s route %d %s C=%d blank=%d W=%d %s" % (what, route, dtype, C, blank, W, layout)
        ui = np.uint64 if dtype == "float64" else np.uint32
        bad = np.nonzero(got[0].view(ui) != off.view(ui))[0]
        assert not len(bad), "%s: off differs in %d of %d rows, first rows %s" % (tag, len(bad), len(off), bad[:SHOW])
        if route == 1:
            bad = np.nonzero((got[1].view(np.uint32) != srt[0].view(np.uint32)).any(axis=1) |
                             (got[2] != srt[1]).any(axis=1))[0]
            assert not len(bad), "%s: sorted class list differs in %d of %d rows, first rows %s" % (
                tag, len(bad), len(off), bad[:SHOW])


def _blanks(C):
    return sorted({0, C // 2, C - 1})


def _widths(C):
    """W = 1 (Ke = 5 < C-1), and the narrowest W with Ke = C-1 where the wide path takes that shape
    (C <= 129); above, the wide path never sees Ke = C-1, and W = 64 gives a second, larger cut."""
    return [1, (C - 3) // 2] if C <= 129 else [1, 64]


@pytest.mark.parametrize("dtype", ["f32", "f16", "bf16", "f64"])
@pytest.mark.parametrize("C", ROUTE0_C)
def test_generic_normaliser(libs, C, dtype):
    """LaunchLogNorm (LogNormRowKernel for C <= 64, LogNormKernel above, LogNormKernelF64; half inputs
    through the exact upcast) on every value family, dense and as a batch shard."""
    lib, cpu = libs
    rng = np.random.default_rng(C * 7 + DT[dtype][0])
    T, B = 3, 2 * N_FAMILIES
    for blank in _blanks(C):  # (the normaliser ignores the blank; the masked rows keep it finite)
        x = _rows(rng, T * B, C, blank, DT[dtype][1]).reshape(T, B, C)
        _check_prepass(lib, cpu, 0, x, DT[dtype][1], blank, 1)


@pytest.mark.parametrize("dtype", ["f32", "f16", "bf16"])
@pytest.mark.parametrize("C", ROUTE1_C)
def test_wide_prepass(libs, C, dtype):
    """LaunchNormTopClasses (NormTopClassesKernel, NI = 2 ... 64 classes per lane) on every value
    family: the normaliser and the sorted class list, for the blank first, in the middle and last,
    with Ke < C-1 and (where the wide path takes it) Ke = C-1, dense and as a batch shard."""
    lib, cpu = libs
    rng = np.random.default_rng(C * 11 + DT[dtype][0])
    T, B = 3, 2 * N_FAMILIES
    for blank in _blanks(C):
        x = _rows(rng, T * B, C, blank, DT[dtype][1]).reshape(T, B, C)
        for W in _widths(C):
            _check_prepass(lib, cpu, 1, x, DT[dtype][1], blank, W)


@pytest.fixture(scope="module")
def sms(libs):
    import torch
    return int(torch.cuda.get_device_properties(torch.cuda.current_device()).multi_processor_count)


@pytest.mark.parametrize("route,dtype,C,per_thread", [
    (0, "f32", 29, True), (0, "bf16", 64, True),     # LogNormRowKernel: 8 CTAs x 256 rows per SM per pass
    (0, "f32", 1025, False), (0, "f64", 65, False),  # warp per row: 16 CTAs x 8 warps per SM per pass
    (1, "f16", 129, False), (1, "f32", 1025, False)])
def test_normalisers_beyond_one_grid_pass(libs, sms, route, dtype, C, per_thread):
    """More rows than one grid holds, so every grid-stride loop runs a second pass."""
    lib, cpu = libs
    one_pass = sms * (8 * 256 if per_thread else 16 * 8)
    T = 16
    B = -(-(one_pass + one_pass // 16) // T)
    rng = np.random.default_rng(C + route)
    blank = C - 1
    x = _rows(rng, T * B, C, blank, DT[dtype][1]).reshape(T, B, C)
    assert T * B > one_pass
    _check_prepass(lib, cpu, route, x, DT[dtype][1], blank, _widths(C)[-1], layouts=("dense",),
                   what="%d rows" % (T * B))


def test_prepass_refuses_what_its_route_does_not_serve(libs):
    import torch
    lib, _ = libs
    x = torch.zeros(2, 2, 40, device="cuda")
    off = torch.empty(4, device="cuda")
    buf = torch.empty(4 * 512, device="cuda")
    ks = ctypes.c_int()
    args = lambda route, dt, C, blank, W: (route, x.data_ptr(), dt, 2, 2, C, 0, blank, W, off.data_ptr(),
                                           buf.data_ptr(), buf.data_ptr(), ctypes.byref(ks), None)
    assert lib.ctcx_debug_prepass(*args(1, 3, 40, 0, 4)) == 9    # float64 on the wide route
    assert lib.ctcx_debug_prepass(*args(1, 0, 32, 0, 4)) == 9    # C <= 32
    assert lib.ctcx_debug_prepass(*args(1, 0, 40, 0, 300)) == 9  # beam wider than the wide kernel's
    assert lib.ctcx_debug_prepass(*args(0, 0, 40, 40, 4)) == 8   # blank outside [0, C)
    assert lib.ctcx_debug_prepass(*args(2, 0, 40, 0, 4)) == 8    # no such route
    torch.cuda.synchronize()
