#!/usr/bin/env python
"""Benchmark of the CTC extended beam-search decode (BASELINE.json metric: utterance-frames
decoded per second at beam=100).

  python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--kind gauss|peaky]
                  [--workload cfg1|cfg2|cfg3|cfg4|cfg5]   (default cfg2, the shape the metric is quoted on)
                  [--dump-outputs DIR]

One "step" = one decode of one batch of synthetic logits: the LibriSpeech char-CTC shape the metric
is quoted on (BASELINE.json configs[1]): T=500, B=256 per GPU, C=29 (blank=28), beam_width=100,
top_paths=1, merge_repeated=true. Multi-GPU: utterances are independent, so every rank decodes its
own B=256 batch (weak scaling, no collective on the data path); value = frames of all ranks / max
time over ranks.

Own arm: `value` times the op with logits resident in HBM (CUDA events, decode + pack, outputs left
on the device); `e2e` times the public call with pinned HOST logits and HOST results (H2D + decode +
pack + D2H inside the timed region). `roofline` is for the dominant kernel (the beam kernel):
algorithmic bytes = 4*C per frame (the fp32 logits, read once) over its CUDA-event duration, against
the measured HBM peak in MEASURED_PEAKS.json. `cpu_baseline` times the reference's own CPU
implementation (oracle/_ref, compiled from the reference's unmodified headers; falls back to the
plain-C port in oracle/) on the host cores on a bounded sample of the same workload.

Reference arm (--impl reference): the reference CPU op on all host cores, same config and metric.

--dump-outputs DIR: after the timed steps, the raw outputs of the last device-resident step (rank 0)
are written as DIR/<output>[_<path>].npy. The inputs depend only on the arguments, so two builds run
with the same arguments can be compared output for output.
"""
import argparse
import ctypes
import json
import os
import subprocess
import sys
import threading
import time
from concurrent.futures import ThreadPoolExecutor

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))

# BASELINE.json configs[0..4]; the metric is quoted on cfg2, the others are selectable for the
# per-shape table in DESIGN.md (B is per GPU)
WORKLOADS = {
    "cfg1": dict(workload="repo test scale (BASELINE configs[0])", T=50, B=8, C=29, blank_index=28,
                 beam_width=10, top_paths=3, merge_repeated=False, blank_label=-1),
    "cfg2": dict(workload="librispeech-char-ctc (BASELINE configs[1])", T=500, B=256, C=29, blank_index=28,
                 beam_width=100, top_paths=1, merge_repeated=True, blank_label=-1),
    "cfg3": dict(workload="wav2vec2-base char head (BASELINE configs[2])", T=1500, B=64, C=32, blank_index=31,
                 beam_width=64, top_paths=4, merge_repeated=False, blank_label=-1),
    "cfg4": dict(workload="conformer-bpe head (BASELINE configs[3])", T=400, B=128, C=1024, blank_index=1023,
                 beam_width=16, top_paths=1, merge_repeated=False, blank_label=-1),
    "cfg5": dict(workload="throughput sweep (BASELINE configs[4], 1024 utterances per GPU)", T=500, B=1024, C=29,
                 blank_index=28, beam_width=100, top_paths=1, merge_repeated=True, blank_label=-1),
}
CFG = dict(WORKLOADS["cfg2"])
L2_BYTES = 126 * 1024 * 1024
DUMP_LIMIT_BYTES = 64 * 1024 * 1024


def make_batch(kind, seed, T, B, C, blank):
    import ctcx_testlib as L
    return L.make_logits(kind, T, B, C, blank, seed)


def outputs_to_numpy(raw):
    """The raw op's outputs as {file name: array}: one array per output and path (decoded_values_0,
    ...), log_probability as one [B, top_paths] array. Integer outputs become float64, which holds
    every index and label exactly; log-probabilities keep their float type. Above DUMP_LIMIT_BYTES in
    all, every sparse output keeps the same fixed, seeded sample of its entries (indices and values of
    one path stay paired)."""
    arrays = {}
    for name, group in zip(raw._fields, raw):
        for key, t in ([(name, group)] if name == "log_probability" else
                       [("%s_%d" % (name, p), t) for p, t in enumerate(group)]):
            a = t.detach().cpu().numpy()
            arrays[key] = a if a.dtype in (np.float32, np.float64) else a.astype(np.float64)
    sparse = [k for k in arrays if k.startswith(("decoded_indices", "decoded_values", "alignment_indices",
                                                 "alignment_values"))]
    sparse_bytes = sum(arrays[k].nbytes for k in sparse)
    budget = DUMP_LIMIT_BYTES - sum(a.nbytes for a in arrays.values()) + sparse_bytes
    if sparse_bytes > budget:
        for key in sparse:
            n = arrays[key].shape[0]
            keep = np.random.default_rng(0).choice(n, n * budget // sparse_bytes, replace=False)
            arrays[key] = arrays[key][np.sort(keep)]
    return arrays


def write_outputs(arrays, out_dir):
    os.makedirs(out_dir, exist_ok=True)
    for key, a in arrays.items():
        np.save(os.path.join(out_dir, key + ".npy"), a)


# ------------------------------------------------------------------------------------------------
def cpu_reference_run(x, n_utt, threads):
    """Decode the first n_utt utterances of x with the reference CPU implementation on `threads`
    host threads (one utterance per task; the library releases the GIL). Returns (seconds, kind)."""
    import ctcx_testlib as L
    L.build_oracles()
    T, B, C = x.shape
    sl = np.full(B, T, np.int32)
    kind = "reference" if L.have_ref() else "port"

    def one(b):
        if kind == "reference":
            L.ref_decode(x, sl, CFG["beam_width"], CFG["top_paths"], CFG["merge_repeated"],
                         CFG["blank_index"], CFG["blank_label"], b_range=(b, b + 1))
        else:
            L.oracle_decode(x[:, b:b + 1], sl[b:b + 1], CFG["beam_width"], CFG["top_paths"],
                            CFG["merge_repeated"], CFG["blank_index"], CFG["blank_label"])

    t0 = time.perf_counter()
    with ThreadPoolExecutor(max_workers=threads) as ex:
        list(ex.map(one, range(n_utt)))
    return time.perf_counter() - t0, kind


def host_threads():
    """Host threads used for the CPU reference: all cores the process may use, capped at 64 (the
    reference keeps ~0.5 GB of trie per in-flight utterance, SURVEY.md section 6)."""
    try:
        n = len(os.sched_getaffinity(0))
    except AttributeError:
        n = os.cpu_count() or 1
    return max(1, min(n, 64))


class ClockSampler:
    """Samples nvidia-smi clocks / throttle reasons during the timed region."""

    Q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, index):
        self.index, self.proc, self.lines = index, None, []

    def start(self):
        if os.environ.get("CTCX_BENCH_NO_SAMPLER"):
            return
        try:
            self.proc = subprocess.Popen(
                ["nvidia-smi", "-i", str(self.index), "--query-gpu=" + self.Q,
                 "--format=csv,noheader,nounits", "-lms", "20"],
                stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.th = threading.Thread(target=self._read, daemon=True)
            self.th.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.lines.append(line.strip())

    def stop(self):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.15)
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except Exception:
            self.proc.kill()
        sm, mx, reasons = [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for ln in self.lines:
            f = [v.strip() for v in ln.split(",")]
            if len(f) < 7:
                continue
            try:
                sm.append(float(f[0]))
                mx.append(float(f[1]))
            except ValueError:
                continue
            for nm, v in zip(names, f[3:7]):
                if v.lower().startswith("active"):
                    reasons.add(nm)
        return {"sm_mhz": float(np.median(sm)) if sm else None,
                "sm_max_mhz": float(max(mx)) if mx else None, "samples": len(sm),
                "reasons": sorted(reasons)}


# ------------------------------------------------------------------------------------------------
def run_reference_arm(args, rank, world):
    if rank != 0:
        return
    cores = host_threads()
    T, B, C = CFG["T"], CFG["B"], CFG["C"]
    x = make_batch(args.kind, 1, T, B, C, CFG["blank_index"])
    n_utt = min(B, cores)  # one utterance per core per step: a bounded sample of the workload
    for _ in range(args.warmup if args.warmup < 1 else 1):
        cpu_reference_run(x, min(n_utt, cores), cores)
    times = []
    kind = "reference"
    for _ in range(args.steps):
        dt, kind = cpu_reference_run(x, n_utt, cores)
        times.append(dt)
    total = sum(times)
    value = n_utt * T * len(times) / total
    line = {
        "impl": "reference", "metric": "utterance_frames_per_s_beam100", "value": value,
        "unit": "frames/s", "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup,
        "ms_per_step": 1e3 * total / len(times), "higher_is_better": True, "scaling": "weak",
        "vs_baseline": None, "dtype": "f32", "data": "synthetic (%s logits, seed 1)" % args.kind,
        "config": dict(CFG, n_gpus=args.gpus, kind=args.kind,
                       note="CPU reference; each step decodes %d utterances (1 per host thread)" % n_utt),
        "cpu_baseline": {"value": value, "unit": "frames/s", "cores": cores, "kind": kind,
                         "sample": "%d utterances of T=%d per step, %d steps" % (n_utt, T, len(times))},
        "e2e": {"value": value, "unit": "frames/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(line), flush=True)


def run_own_arm(args, rank, world, local_rank, out_fd=1):
    import torch
    import torch.distributed as dist
    import ctc_beam_search_op_b200 as op
    from ctc_beam_search_op_b200 import _lib

    if not torch.cuda.is_available():
        raise RuntimeError("bench.py needs a CUDA device (there is no CPU fallback)")
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    lib = _lib.load()
    # one process per GPU: sit on the cores (and allocate the pinned buffers on the memory) next to it
    near_cpus = None if args.no_numa_bind else op.bind_host_to_device(local_rank)
    T, B, C = CFG["T"], CFG["B"], CFG["C"]
    W, P = CFG["beam_width"], CFG["top_paths"]
    kw = dict(beam_width=W, top_paths=P, merge_repeated=CFG["merge_repeated"],
              blank_index=CFG["blank_index"], blank_label=CFG["blank_label"])

    # inputs rotate over enough distinct batches that consecutive steps never find their logits in
    # L2 (total > 126 MB); every step also streams ~100 MB of back-pointer records through L2.
    bytes_per_batch = T * B * C * 4
    n_rot = L2_BYTES // bytes_per_batch + 2
    base = make_batch(args.kind, 1 + rank, T, B, C, CFG["blank_index"])
    host_batches, dev_batches = [], []
    rng = np.random.default_rng(77 + rank)
    in_dt = {"f32": torch.float32, "f16": torch.float16, "bf16": torch.bfloat16, "f64": torch.float64}[args.dtype]
    bytes_per_batch = T * B * C * {"f32": 4, "f16": 2, "bf16": 2, "f64": 8}[args.dtype]
    if args.scorer:  # the reference's scorer extension point: a random label-bigram table (log-probabilities)
        kw["expansion_scores"] = -np.abs(np.random.default_rng(5).standard_normal((C + 1, C))).astype(np.float32)
    n_rot = L2_BYTES // bytes_per_batch + 2
    for r in range(n_rot):
        xb = base if r == 0 else np.ascontiguousarray(base[:, rng.permutation(B), :])
        hb = torch.from_numpy(xb).to(in_dt).pin_memory()
        host_batches.append(hb)
        dev_batches.append(hb.to(dev))
    seq_host = torch.full((B,), T, dtype=torch.int32).pin_memory()
    seq_dev = seq_host.to(dev)
    frames_per_step = T * B

    def step_device(i):
        return op.ctc_ext_beam_search_decoder_raw(dev_batches[i % n_rot], seq_dev, **kw)

    def step_e2e(i):
        return op.ctc_ext_beam_search_decoder_raw(host_batches[i % n_rot], seq_host, **kw)

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    # clocks / throttle reasons are sampled from before the warm-up to after the e2e region (the
    # timed regions themselves last only ~0.1 s; nvidia-smi needs a moment to start)
    # (one sampler per node is enough evidence and keeps seven more polling processes off the host cores
    # that feed the other ranks)
    sampler = ClockSampler(local_rank)
    if rank == 0:
        sampler.start()
    time.sleep(0.3)

    # ---- warm-up ----
    for i in range(max(args.warmup, 3)):
        step_device(i)
    out = None
    for i in range(max(args.warmup, 3, n_rot)):  # the host path has its own cold costs (side stream, pinned
        out = step_e2e(i)                        # result buffers): once over every rotating batch, holding the
    del out                                      # previous result while the next is produced, as the timed loop does
    barrier()

    # ---- device-resident timing (CUDA events per step on the launching stream) ----
    lib.ctcx_profile_enable(1)
    evs = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True))
           for _ in range(args.steps)]
    kern_ms = np.zeros((args.steps, 5), np.float32)
    buf = (ctypes.c_float * 5)()
    barrier()
    wall0 = time.perf_counter()
    for i, (e0, e1) in enumerate(evs):
        e0.record()
        res = step_device(i)
        e1.record()
        lib.ctcx_profile_get(buf)
        kern_ms[i] = list(buf)
        if i < args.steps - 1:
            res = None  # freed before the next step, as in the warm-up; the last step's result is kept
    barrier()
    wall_dev = time.perf_counter() - wall0
    lib.ctcx_profile_enable(0)
    dev_ms = float(sum(e0.elapsed_time(e1) for e0, e1 in evs))
    dumped = outputs_to_numpy(res) if args.dump_outputs and rank == 0 else None
    del res

    # ---- end-to-end timing: pinned host logits in, host results out ----
    barrier()
    t0 = time.perf_counter()
    d2h = 0
    step_s = []
    for i in range(args.steps):
        ts = time.perf_counter()
        out = step_e2e(i)
        # bytes that crossed the bus device->host for this call (the result buffer as copied -- an upper
        # bound of the exact tensors on the single-synchronisation route -- plus the sizes block)
        d2h = out.d2h_bytes
        step_s.append(time.perf_counter() - ts)
    torch.cuda.synchronize()
    e2e_s = time.perf_counter() - t0
    if os.environ.get("CTCX_BENCH_VERBOSE"):
        sys.stderr.write("e2e per-step ms: %s\n" % " ".join("%.2f" % (1e3 * v) for v in step_s))
    barrier()

    # ---- supplementary: the same steps with ONE decode in flight behind the one being read ----
    # (`wait=False` handles: batch i+1 is enqueued before batch i's result is read, so the GPU never waits
    # for the host between decodes; every result is still read inside the timed region)
    def pipelined(batches, seq):
        pend, last = None, None
        for i in range(max(args.warmup, 3, n_rot)):  # warm-up in the same pattern (two results alive: the page-locked
            nxt = op.ctc_ext_beam_search_decoder_raw(batches[i % n_rot], seq, wait=False, **kw)  # buffers of both exist)
            if pend is not None:
                last = pend.result()
            pend = nxt
        last = pend.result()
        pend = None
        barrier()
        ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        t_start = time.perf_counter()
        ev0.record()
        for i in range(args.steps):
            nxt = op.ctc_ext_beam_search_decoder_raw(batches[i % n_rot], seq, wait=False, **kw)
            if pend is not None:
                last = pend.result()
            pend = nxt
        last = pend.result()
        ev1.record()
        torch.cuda.synchronize()
        wall = time.perf_counter() - t_start
        assert last[4][0].numel() == frames_per_step
        return ev0.elapsed_time(ev1), wall * 1e3

    pipe_dev_ms, _ = pipelined(dev_batches, seq_dev)
    _, pipe_e2e_ms = pipelined(host_batches, seq_host)
    barrier()
    clocks = sampler.stop()

    if world > 1:
        t = torch.tensor([dev_ms, e2e_s * 1e3, pipe_dev_ms, pipe_e2e_ms], dtype=torch.float64, device=dev)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        dev_ms, e2e_ms, pipe_dev_ms, pipe_e2e_ms = (float(v) for v in t)
    else:
        e2e_ms = e2e_s * 1e3
    sharded = None
    if args.workload == "cfg2" and args.dtype == "f32" and not args.scorer and not args.no_sharded:
        del dev_batches, host_batches
        torch.cuda.empty_cache()
        sharded = run_sharded_cfg5(rank, world, local_rank, steps=args.steps, warmup=3)
    if rank != 0:
        return

    total_frames = frames_per_step * args.steps * world
    value = total_frames / (dev_ms * 1e-3)
    e2e_value = total_frames / (e2e_ms * 1e-3)
    peaks_path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(peaks_path):
        peak, peak_src = float(json.load(open(peaks_path))["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
    else:
        peak, peak_src = 6650.0, "fallback (B200_PROFILING.md)"
    beam_ms = float(kern_ms[:, 1].mean())
    algo_bytes = float(bytes_per_batch)  # per beam-kernel launch: the logits, read once
    achieved = algo_bytes / (beam_ms * 1e-3) / 1e9
    traffic = None
    tr_path = os.path.join(ROOT, "profiles", "beam_kernel_traffic.json")
    if os.path.exists(tr_path):
        traffic = json.load(open(tr_path)).get("dram_bytes_per_launch")

    line = {
        "metric": "utterance_frames_per_s_beam100", "value": value, "unit": "frames/s",
        "n_gpus": world, "steps": args.steps, "warmup": max(args.warmup, 3),
        "ms_per_step": dev_ms / args.steps, "higher_is_better": True, "scaling": "weak",
        "vs_baseline": None, "dtype": "f64" if args.dtype == "f64" else "f32",
        "data": "synthetic (%s logits, seed 1+rank)" % args.kind,
        "config": dict(CFG, n_gpus=world, kind=args.kind, global_batch=B * world, input_dtype=args.dtype,
                       scorer="bigram table" if args.scorer else None,
                       host_cores_near_gpu=(len(near_cpus) if near_cpus else None),
                       l2="inputs rotate over %d distinct batches (%.0f MB > 126 MB L2)"
                          % (n_rot, n_rot * bytes_per_batch / 1e6)),
        "clocks": clocks,
        "e2e": {"value": e2e_value, "unit": "frames/s", "h2d_bytes_per_step": bytes_per_batch + B * 4,
                "d2h_bytes_per_step": int(d2h), "ms_per_step": e2e_ms / args.steps},
        # per step: [normaliser + class selection pre-pass (wide vocabularies only)], beam, trace, scan, flags,
        # [output pointer table (single-synchronisation route) | scorer-table check], pack
        "gpu_launches": (5 + (1 if C > 32 else 0) + (1 if args.scorer else 0) + (0 if args.scorer else 1)) * args.steps,
        "kernel_ms": {"lognorm": float(kern_ms[:, 0].mean()), "beam": beam_ms,
                      "trace": float(kern_ms[:, 2].mean()), "scan": float(kern_ms[:, 3].mean()),
                      "wall_ms_per_step": 1e3 * wall_dev / args.steps},
        "roofline": {"bound": "hbm", "achieved": achieved, "peak": peak, "unit": "GB/s",
                     "frac": achieved / peak, "traffic": traffic if args.workload == "cfg2" else None,
                     "kernel": ("BeamKernelT (generic)" if ((args.dtype == "f64" or args.scorer) and C > 32) else
                                "BeamKernelWide" if (32 < C <= 2048) else
                                "BeamKernelV4 (scorer variant)" if args.scorer else
                                "BeamKernelV4 (double)" if args.dtype == "f64" else "BeamKernelV4"),
                     "peak_source": peak_src,
                     "note": "algorithmic bytes = 4*C per frame (logits read once); the kernel is "
                             "bound by the T-long serial recurrence per utterance, not by HBM"},
    }
    line["pipelined"] = {
        "note": "same workload with one decode in flight behind the one being read (wait=False handles); "
                "value / e2e above are one blocking call per step",
        "depth": 2,
        "value": frames_per_step * world * args.steps / (pipe_dev_ms * 1e-3), "ms_per_step": pipe_dev_ms / args.steps,
        "e2e_value": frames_per_step * world * args.steps / (pipe_e2e_ms * 1e-3),
        "e2e_ms_per_step": pipe_e2e_ms / args.steps, "unit": "frames/s"}
    if sharded is not None:
        line["sharded_cfg5"] = sharded
    if not args.no_cpu_baseline and world == 1:  # a reported baseline, measured at N=1 only
        cores = host_threads()
        n_utt = min(B, cores)
        dt, kind = cpu_reference_run(base, n_utt, cores)
        n1 = 8 if T * W >= 20000 else 32
        dt1, _ = cpu_reference_run(base, n1, 1)
        # the op as it really runs is single-threaded (kernels.cc:68-90): that is the primary figure; the
        # batch sharded over all host threads (memory-bound: ~0.5 GB of trie per utterance in flight) beside it
        line["cpu_baseline"] = {"value": n1 * T / dt1, "unit": "frames/s", "cores": 1, "kind": kind,
                                "sample": "%d utterances of this workload on one thread (%.1f s)" % (n1, dt1),
                                "all_host_threads": {"value": n_utt * T / dt, "cores": cores,
                                                     "sample": "%d utterances, one per thread (%.1f s)" % (n_utt, dt)}}
    if dumped is not None:
        write_outputs(dumped, args.dump_outputs)
    sys.stdout.flush()
    os.write(out_fd, (json.dumps(line) + "\n").encode())


def run_sharded_cfg5(rank, world, local_rank, steps, warmup):
    """BASELINE configs[4] as the north star states it: ONE global batch of 8192 utterances (T=500, C=29,
    beam 100), batch-sharded over the ranks through the product's sharding API (decode_distributed: rank r
    decodes block r IN PLACE from a view of the time-major tensor, the sparse outputs are gathered on rank 0
    INSIDE the timed region). Strong scaling: frames/s = 8192 * 500 / max-over-ranks wall time per step.
    Two variants: logits resident on each GPU / in page-locked host memory. Each runs `steps` timed steps
    (--steps): about 80 ms per step for the two together on one B200 (1000 W power limit), so about 4 s at
    the default of 50 steps."""
    import torch
    import torch.distributed as dist
    import ctc_beam_search_op_b200 as op
    dev = torch.device("cuda", local_rank)
    T, B, C, W = 500, 8192, 29, 100
    kw = dict(beam_width=W, top_paths=1, merge_repeated=True, blank_index=28, blank_label=-1)
    g = torch.Generator(device=dev)
    g.manual_seed(4)  # the same global tensor on every rank; each rank only ever reads its own block
    x_dev = torch.randn((T, B, C), generator=g, device=dev, dtype=torch.float32)
    seq_dev = torch.full((B,), T, dtype=torch.int32, device=dev)
    b0, b1 = op.shard_bounds(B, world)[rank]
    # host variant: this rank's block of the global tensor lives in page-locked host memory; the view handed
    # to the API is still [:, b0:b1, :] of a [T, B, C]-shaped tensor (other blocks are never touched)
    # (N = 1: the whole tensor; N > 1: each rank holds its own block, the usual multi-process layout)
    x_host = x_dev.cpu().pin_memory() if world == 1 else None
    x_block = x_dev[:, b0:b1, :].contiguous().cpu().pin_memory() if world > 1 else None
    seq_host = torch.full((B,), T, dtype=torch.int32)
    seq_block = seq_host[b0:b1]

    def decode_dev():
        if world == 1:
            return op.ctc_ext_beam_search_decoder_raw(x_dev, seq_dev, **kw)
        return op.decode_distributed(x_dev, seq_dev, dst=0, **kw)

    def decode_host():
        if world == 1:
            return op.ctc_ext_beam_search_decoder_raw(x_host, seq_host, **kw)
        return op.decode_distributed(x_block, seq_block, dst=0, global_batch=B, **kw)

    out = {}
    for name, fn in (("device_resident", decode_dev), ("host_resident", decode_host)):
        res = None
        for _ in range(max(2, warmup)):
            res = fn()  # (held while the next one is produced, as in the timed loop: same allocation pattern)
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
        t0 = time.perf_counter()
        for _ in range(steps):
            res = fn()
        torch.cuda.synchronize()
        dt = time.perf_counter() - t0
        if world > 1:
            t = torch.tensor([dt], dtype=torch.float64, device=dev)
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
            dt = float(t[0])
            dist.barrier()
        out[name] = {"value": B * T * steps / dt, "unit": "frames/s", "ms_per_step": 1e3 * dt / steps}
        if rank == 0:
            n_ali = int(res[4][0].shape[0])
            assert n_ali == B * T, (n_ali, B * T)  # the merged result covers the whole batch
    out.update(global_batch=B, T=T, C=C, beam_width=W, steps=steps, scaling="strong",
               gather="sparse outputs gathered on rank 0 inside the timed region (NCCL, GPU to GPU, merged on "
                      "the device; host variant: plus one copy of the merged result to the host)" if world > 1
               else "single GPU: nothing to gather")
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=50)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--kind", default="gauss", choices=["gauss", "peaky"])
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-sharded", action="store_true", help="skip the B=8192 strong-scaling leg")
    ap.add_argument("--workload", default="cfg2", choices=sorted(WORKLOADS))
    ap.add_argument("--dtype", default="f32", choices=["f32", "f16", "bf16", "f64"],
                    help="element type of the logits (scores are float32; float64 for f64, the op's T = double)")
    ap.add_argument("--scorer", action="store_true", help="decode with a label-bigram expansion-score table")
    ap.add_argument("--no-numa-bind", action="store_true",
                    help="do not move the process next to its GPU (bind_host_to_device) before allocating host buffers")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="write the raw outputs of the last timed device-resident step as "
                         "DIR/<output>_<path>.npy and DIR/log_probability.npy")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl == "reference":
        ap.error("--dump-outputs applies to --impl ours")
    CFG.clear()
    CFG.update(WORKLOADS[args.workload])
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    if args.impl == "reference":
        run_reference_arm(args, rank, world)
        return
    # stdout must carry exactly one JSON line: NCCL prints its version banner there, so fd 1 points
    # to stderr until the result is ready
    sys.stdout.flush()
    saved_stdout = os.dup(1)
    os.dup2(2, 1)
    if world > 1:
        import torch
        import torch.distributed as dist
        torch.cuda.set_device(local_rank)
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))
        dist.barrier()
    try:
        run_own_arm(args, rank, world, local_rank, saved_stdout)
    finally:
        if world > 1:
            import torch.distributed as dist
            dist.destroy_process_group()


if __name__ == "__main__":
    main()
