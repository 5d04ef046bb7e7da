#!/usr/bin/env python
"""bench.py -- headline benchmark of the B200 hot path (BASELINE.json metric).

One step = one pass of the hot path over one synthetic ComplexF32 stream shard:
    y = conv(x, v)              overlap-save FFT convolution, 4097-tap FIR on 2^26 samples   (BASELINE config 2)
    P = welch_pgram(y[:2^26])   n = nfft = 4096, 50 % overlap, hanning, two-sided            (Welch stage of the metric)
metric = input samples per second through both stages (Gsamples/s), whole job over all ranks.

  python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--log2n 26] [--workload ...] [--dump-outputs DIR]
  N > 1: python -m torch.distributed.run --nnodes=1 --nproc-per-node N --master-addr 127.0.0.1 ... bench.py --gpus N

Multi-GPU (the contract line is weak scaling): every rank owns a 2^26-sample shard of one long stream (plus the nv-1
sample left halo), convolves its own output range with no collective, accumulates the Welch power of its own segments
scaled by the GLOBAL 1/(k r), and the only exchange is one NCCL all-reduce of the 4096-bin power vector per step (async,
overlapped with the next step's convolution).  For N > 1 the same line carries `strong`: ONE 2^26-sample stream
range-sharded over the N GPUs.  `check` validates what the timed pipeline left in its output buffers (outside the timed
region).  --workload selects BASELINE configs[2..4] as bench lines of their own.

`--impl reference` times the reference's CPU path: the unmodified DSP.jl + FFTW through bench_ref/cpu_reference.jl when a
`julia` with DSP.jl is on PATH; otherwise (this image) the CPU oracle port (oracle/, numpy + scipy pocketfft, the stream
cut into block / segment ranges that run on all host threads) of the same two stages, at the full 2^26 size when K + W
steps fit in ~3 minutes, else on a bounded sample.
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

NV = 4097
NSEG, NOVERLAP = 4096, 2048
METRIC = "Gsamples/s filt+welch on 2^26 cplx-F32"


def make_taps():
    """4097-tap complex bandpass (SURVEY.md 8d, C2): Hamming-windowed sinc shifted to 0.3 pi."""
    n = np.arange(NV) - NV // 2
    return (0.2 * np.sinc(0.2 * n) * np.hamming(NV) * np.exp(1j * np.pi * 0.3 * n)).astype(np.complex64)


def hanning64(n):
    x = -0.5 + np.arange(n, dtype=np.float64) / (n - 1)
    return 0.5 * (1 + np.cos(2 * np.pi * x))


class ClockSampler:
    """nvidia-smi sampling DURING the timed region (B200_PROFILING.md clocks line)."""

    def __init__(self, index):
        self.rows = []
        self.proc = None
        self.index = index

    def start(self):
        q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
             "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
             "clocks_event_reasons.sw_power_cap")
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={q}", "--format=csv,noheader,nounits", "-lms", "20",
                                          "-i", str(self.index)], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.thread = threading.Thread(target=self._read, daemon=True)
            self.thread.start()
        except OSError:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append(line.strip())

    def stop(self):
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.15)
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except Exception:
            self.proc.kill()
        sm, smax, reasons = [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for r in self.rows:
            f = [t.strip() for t in r.split(",")]
            if len(f) < 7:
                continue
            try:
                sm.append(float(f[0])); smax.append(float(f[1]))
            except ValueError:
                continue
            for nme, v in zip(names, f[3:7]):
                if v.lower().startswith("active"):
                    reasons.add(nme)
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": max(smax) if smax else None,
                "samples": len(sm), "reasons": sorted(reasons)}


DUMP_SAMPLE, DUMP_EDGE, DUMP_SEED = 1 << 20, 4096, 20260101


def dump_outputs(out_dir, arrays, d):
    """--dump-outputs: write each array the timed path handed back in its last step as <out_dir>/<name>.npy, so that two
    builds run with the same arguments (same seeded inputs) can be compared output for output.  Complex arrays are written
    as float (re, im) pairs along a trailing axis of 2.  An array of more than DUMP_SAMPLE elements is written as a fixed
    sample of its flattened elements -- the first and last DUMP_EDGE plus DUMP_SAMPLE drawn with a fixed seed -- and the
    sampled flat indices go beside it as <name>_index.npy (float64, exact); about 16 MB per sampled array.  With several
    ranks every rank writes its own arrays, suffixed _rank<r>."""
    import torch
    os.makedirs(out_dir, exist_ok=True)
    suffix = f"_rank{d.rank}" if d.world > 1 else ""
    for name, t in arrays.items():
        t = t.detach()
        if t.numel() > DUMP_SAMPLE:
            n = t.numel()
            rng = np.random.default_rng(DUMP_SEED)
            idx = np.unique(np.concatenate([np.arange(DUMP_EDGE), np.arange(n - DUMP_EDGE, n), rng.integers(0, n, DUMP_SAMPLE)]))
            t = t.reshape(-1)[torch.from_numpy(idx).to(t.device)]
            np.save(os.path.join(out_dir, f"{name}{suffix}_index.npy"), idx.astype(np.float64))
        t = t.cpu()
        a = (torch.view_as_real(t) if t.is_complex() else t).numpy()
        assert a.dtype in (np.float32, np.float64), (name, a.dtype)
        np.save(os.path.join(out_dir, f"{name}{suffix}.npy"), a)


def measured_peak_gbs():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    try:
        with open(p) as f:
            return float(json.load(f)["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
    except Exception:
        return 6650.0, "fallback (B200_PROFILING.md 6.65 TB/s)"


# ------------------------------------------------------------------------------------------- CPU baseline (oracle port)

def cpu_reference_step(x, v, win, workers):
    """The reference's CPU path for one step, restated (oracle/): overlap-save conv with the reference's own block
    length (optimalfftfiltlength -> 65536, src/dspbase.jl:268-291, 490-609) + welch_pgram (src/periodograms.jl:746-759),
    Float32 arithmetic.  The reference runs these loops on ONE Julia thread (only FFTW is threaded); to give the CPU arm
    every host core, the stream is cut into `workers` ranges of whole overlap-save blocks / Welch segments that run
    concurrently (numpy and pocketfft release the GIL), each range with single-threaded FFTs -- same blocks, same
    arithmetic, the Welch partial sums added at the end."""
    import scipy.fft as sfft
    from concurrent.futures import ThreadPoolExecutor
    from oracle import dspbase as od
    from oracle import periodograms as op
    n, nv = len(x), len(v)
    nfft = od.optimalfftfiltlength(nv, n)
    L = nfft - nv + 1
    nout = n + nv - 1
    nblk = -(-nout // L)
    parts = max(1, min(workers, nblk // 4))
    y = np.empty(nout, dtype=np.complex64)

    def conv_part(i):
        b0, b1 = nblk * i // parts, nblk * (i + 1) // parts            # blocks [b0, b1): outputs [b0 L, min(b1 L, nout))
        o0, o1 = b0 * L, min(b1 * L, nout)
        lo = max(0, o0 - (nv - 1))
        seg = x[lo: min(n, o1)]
        with sfft.set_workers(1):
            part = od.conv_kern_os(seg, v, nfft, batched=True)          # full convolution of the range; keep its share
        y[o0:o1] = part[o0 - lo: o1 - lo]

    hop = NSEG - NOVERLAP
    k = (n - NSEG) // hop + 1
    wparts = max(1, min(workers, k // 64))
    acc = [None] * wparts

    def welch_part(i):
        k0, k1 = k * i // wparts, k * (i + 1) // wparts                  # segments [k0, k1)
        with sfft.set_workers(1):
            p, _ = op.welch_pgram(y[k0 * hop: (k1 - 1) * hop + NSEG], NSEG, NOVERLAP, onesided=False, nfft=NSEG, window=win)
        acc[i] = p * np.float32(k1 - k0)                                 # undo the range's own 1/k

    with ThreadPoolExecutor(max_workers=workers) as pool:
        list(pool.map(conv_part, range(parts)))
        list(pool.map(welch_part, range(wparts)))
    p = np.sum(acc, axis=0, dtype=np.float64) / k
    return y, p.astype(np.float32)


def time_cpu_baseline(log2_sample, reps, workers, warm_full=0):
    rng = np.random.default_rng(1002)
    n = 1 << log2_sample
    x = ((rng.standard_normal(n, dtype=np.float32) + 1j * rng.standard_normal(n, dtype=np.float32)) * np.float32(2 ** -0.5)).astype(np.complex64)
    v = make_taps()
    win = hanning64(NSEG)
    cpu_reference_step(x[: 1 << 18], v, win, workers)      # warm-up (plan caches, imports)
    for _ in range(warm_full):
        cpu_reference_step(x, v, win, workers)
    ts = []
    for _ in range(reps):
        t0 = time.perf_counter()
        cpu_reference_step(x, v, win, workers)
        ts.append(time.perf_counter() - t0)
    return n, ts


def julia_reference(args):
    """The unmodified reference (DSP.jl + FFTW) through bench_ref/cpu_reference.jl, when a `julia` with DSP.jl installed
    is on PATH (not the case in this image: returns None and the caller falls back to the oracle port)."""
    import shutil
    exe = shutil.which("julia")
    if not exe:
        return None
    try:
        out = subprocess.run([exe, "-t", "auto", os.path.join(ROOT, "bench_ref", "cpu_reference.jl"), str(args.log2n),
                              str(max(1, args.steps)), str(max(1, min(args.warmup, 2)))],
                             capture_output=True, text=True, timeout=1500)
        for ln in reversed(out.stdout.strip().splitlines()):
            if ln.startswith("{"):
                return json.loads(ln)
    except Exception:
        pass
    return None


def run_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    workers = os.cpu_count() or 1
    jl = julia_reference(args)
    if jl is not None:
        val, ms, kind, log2s = float(jl["value"]), float(jl["ms_per_step"]), "reference", args.log2n
        sample = jl.get("sample", "")
        workers = int(jl.get("cores", workers))
        nfft_conv = "optimalfftfiltlength (DSP.jl)"
    else:
        # oracle port.  Sample size: the full 2^log2n workload when K + W steps of it fit in ~3 minutes of host time
        # (probe: one step at 2^22), otherwise the largest power of two that does
        _, probe = time_cpu_baseline(min(args.log2n, 22), 1, workers)
        per_sample = probe[0] / float(1 << min(args.log2n, 22))
        log2s = args.log2n
        while log2s > 20 and per_sample * (1 << log2s) * (args.steps + min(args.warmup, 2)) > 180.0:
            log2s -= 1
        n, ts = time_cpu_baseline(log2s, max(1, args.steps), workers, warm_full=min(args.warmup, 2))
        ms = 1e3 * float(np.mean(ts))
        val = n / (ms * 1e-3) / 1e9
        kind = "port"
        sample = (f"2^{log2s} samples per step; oracle port (numpy + scipy pocketfft, Float32, nfft 65536 as the reference "
                  f"picks), the stream cut into ranges of whole blocks / segments that run on {workers} threads (the reference's "
                  "own loops are single-threaded); Julia/FFTW not installable in this image (bench_ref/cpu_reference.jl runs "
                  "the real DSP.jl where julia exists)")
        nfft_conv = 65536
    full = log2s == args.log2n
    line = {
        "metric": METRIC, "value": val, "unit": "Gsamples/s", "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup,
        "ms_per_step": ms, "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "c64 (ComplexF32)",
        "data": "synthetic", "impl": "reference",
        "config": {"workload": f"overlap-save conv 4097-tap + welch_pgram(4096, 50%, hanning) on 2^{log2s} ComplexF32"
                               + ("" if full else f" (bounded sample of the 2^{args.log2n} workload)"), "nfft_conv": nfft_conv,
                   "samples_per_step": 1 << log2s},
        "cpu_baseline": {"value": val, "unit": "Gsamples/s", "cores": workers, "kind": kind, "sample": sample},
        "e2e": {"value": val, "unit": "Gsamples/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(line))


# ------------------------------------------------------------------------------------------- GPU arm

def kernel_counters():
    """Per-launch hardware counters of the headline kernels, taken from the committed `ncu --set full` captures
    (profiles/kernel_counters.json names the capture each number comes from): executed warp instructions for the FP32-issue
    roofline, DRAM bytes for `roofline.traffic`."""
    try:
        with open(os.path.join(ROOT, "profiles", "kernel_counters.json")) as f:
            return json.load(f)
    except Exception:
        return {}


def bind_to_gpu_numa_node(torch, index):
    """Pin this process to the CPUs of the NUMA node the GPU hangs off, BEFORE any pinned host buffer is allocated: pinned
    pages are placed by first touch, and with N ranks started by torchrun they otherwise land on whatever node the rank
    happened to run on -- the host-pointer end-to-end path then crosses the inter-socket link (round 1: 21.9 ms per step at
    N = 1, 32.8 ms at N = 4/8).  Best effort: returns the node or None."""
    try:
        pr = torch.cuda.get_device_properties(index)
        bdf = "%04x:%02x:%02x.0" % (pr.pci_domain_id, pr.pci_bus_id, pr.pci_device_id)
        with open(f"/sys/bus/pci/devices/{bdf}/numa_node") as f:
            node = int(f.read().strip())
        if node < 0:
            return None
        with open(f"/sys/devices/system/node/node{node}/cpulist") as f:
            cpus = set()
            for part in f.read().strip().split(","):
                a, _, b = part.partition("-")
                cpus.update(range(int(a), int(b or a) + 1))
        os.sched_setaffinity(0, cpus)
        return node
    except Exception:
        return None


class Dist:
    def __init__(self):
        import torch
        self.torch = torch
        self.world = int(os.environ.get("WORLD_SIZE", "1"))
        self.rank = int(os.environ.get("RANK", "0"))
        self.local_rank = int(os.environ.get("LOCAL_RANK", "0"))
        if not torch.cuda.is_available():
            raise SystemExit("bench.py --impl ours needs a CUDA device (no CPU fallback)")
        torch.cuda.set_device(self.local_rank)
        torch.manual_seed(1000 + self.rank)            # same inputs every run, so --dump-outputs can compare two builds
        from dspb200 import _lib
        _lib.check(_lib.lib.dspb200_set_device(self.local_rank))
        self.dev = torch.device("cuda", self.local_rank)
        try:
            self.orig_affinity = os.sched_getaffinity(0)
        except Exception:
            self.orig_affinity = None
        self.numa = bind_to_gpu_numa_node(torch, self.local_rank)
        self.pg = None
        if self.world > 1:
            import torch.distributed as dist
            dist.init_process_group("nccl", device_id=self.dev)
            self.pg = dist

    def sync_all(self):
        self.torch.cuda.synchronize()
        if self.pg is not None:
            self.pg.barrier()
            self.torch.cuda.synchronize()

    def max_over_ranks(self, vals):
        if self.pg is None:
            return [float(v) for v in vals]
        t = self.torch.tensor(list(vals), device=self.dev, dtype=self.torch.float64)
        self.pg.all_reduce(t, op=self.pg.ReduceOp.MAX)
        return [float(v) for v in t.tolist()]

    def close(self):
        if self.pg is not None:
            self.pg.destroy_process_group()


class ConvWelch:
    """The headline step on one rank: the rank owns samples [rank*n, (rank+1)*n) of one n*world-sample ComplexF32 stream
    (plus the nv-1 sample left halo and the Welch overlap its last segments need from the right neighbour's range),
    convolves its own output range -- no collective -- and accumulates the Welch power of the segments that start in its
    range, scaled by the GLOBAL 1/(k r); the only exchange is one sum all-reduce of the 4096-bin power vector.  The
    all-reduce of step i is asynchronous (NCCL's own stream) and is waited for only after step i+1's convolution has been
    enqueued, so it overlaps that kernel instead of sitting between two steps."""

    def __init__(self, d, n, nfft):
        import torch
        from dspb200 import _lib
        self.d, self.n = d, n
        world, rank, dev = d.world, d.rank, d.dev
        self.n_global = n * world
        halo, hop = NV - 1, NSEG - NOVERLAP
        self.hop = hop
        self.k_global = (self.n_global - NSEG) // hop + 1
        self.seg_begin = (rank * n + hop - 1) // hop if rank > 0 else 0       # segments whose start lies in this rank's range
        self.seg_end = min(self.k_global, ((rank + 1) * n + hop - 1) // hop)
        need_hi = (self.seg_end - 1) * hop + NSEG if self.seg_end > self.seg_begin else (rank + 1) * n
        self.hi = max((rank + 1) * n, min(need_hi, self.n_global))
        self.lo = max(0, rank * n - halo)
        # synthetic input, resident in HBM before the timed region; deterministic per-block generation so overlapping
        # halos agree across ranks
        g = torch.Generator(device=dev)
        blk = 1 << 20
        self.x = torch.empty(self.hi - self.lo, dtype=torch.complex64, device=dev)
        for b0 in range((self.lo // blk) * blk, self.hi, blk):
            g.manual_seed(1002 + b0 // blk)
            chunk = torch.view_as_complex(torch.randn(blk, 2, generator=g, device=dev, dtype=torch.float32)) * (2 ** -0.5)
            s0, s1 = max(b0, self.lo), min(b0 + blk, self.hi)
            self.x[s0 - self.lo: s1 - self.lo] = chunk[s0 - b0: s1 - b0]
        self.taps = make_taps()
        self.win = hanning64(NSEG)
        self.norm2 = float(np.sum(self.win * self.win))
        self.r = self.k_global * 1.0 * self.norm2                            # r = k * fs * norm2 (src/periodograms.jl:751)
        self.os_plan = _lib.OsPlan(self.taps, nfft)
        self.spec = _lib.SpecPlan(np.complex64, NSEG, NOVERLAP, NSEG, False, self.win)
        # the conv of the global stream restricted to this rank's own sample range (same-length filter output)
        self.out_lo, self.out_cnt = rank * n, self.hi - rank * n
        self.y = torch.empty(self.out_cnt, dtype=torch.complex64, device=dev)
        self.pw = [torch.zeros(NSEG, dtype=torch.float32, device=dev) for _ in range(2)]
        self.stream = torch.cuda.current_stream()
        self.sp = self.stream.cuda_stream
        self.pending = None
        self.i = 0

    def conv(self):
        self.os_plan.exec_range_dev(self.x.data_ptr(), self.lo, self.x.numel(), self.y.data_ptr(), self.out_lo, self.out_cnt, self.sp)

    def welch(self):
        pw = self.pw[self.i & 1]
        self.spec.welch_range_dev(self.y.data_ptr(), self.out_cnt, self.out_lo, self.seg_begin, self.seg_end, self.r, pw.data_ptr(), self.sp)
        return pw

    def step(self, ev=None):
        if ev:
            ev[0].record(self.stream)
        self.conv()
        if ev:
            ev[1].record(self.stream)
        if self.pending is not None:                   # step i-1's all-reduce: overlapped with this step's convolution
            self.pending.wait()
            self.pending = None
        pw = self.welch()
        if ev:
            ev[2].record(self.stream)
        if self.d.pg is not None:
            self.pending = self.d.pg.all_reduce(pw, async_op=True)
        self.i += 1
        return pw

    def finish(self):
        if self.pending is not None:
            self.pending.wait()
            self.pending = None

    def time(self, steps, warmup):
        import torch
        from dspb200 import _lib
        d = self.d
        for _ in range(max(warmup, 3)):
            self.step()
        self.finish()
        d.sync_all()
        ev = [[torch.cuda.Event(enable_timing=True) for _ in range(3)] for _ in range(steps)]
        l0 = _lib.launch_count()
        e_start, e_stop = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        d.sync_all()
        e_start.record(self.stream)
        for i in range(steps):
            self.last = self.step(ev[i])
        self.finish()
        e_stop.record(self.stream)
        d.sync_all()
        launches = _lib.launch_count() - l0
        total_ms = e_start.elapsed_time(e_stop)
        conv_ms = float(np.mean([ev[i][0].elapsed_time(ev[i][1]) for i in range(steps)]))
        welch_ms = float(np.mean([ev[i][1].elapsed_time(ev[i][2]) for i in range(steps)]))
        total_ms, conv_ms, welch_ms = d.max_over_ranks([total_ms, conv_ms, welch_ms])
        return {"ms_per_step": total_ms / steps, "conv_ms": conv_ms, "welch_ms": welch_ms, "launches": int(launches),
                "value": self.n_global / (total_ms / steps * 1e-3) / 1e9}

    def time_graph(self, steps, warmup):
        """The same step with its kernels replayed from CUDA graphs: two graphs (conv -> Welch into power buffer 0 / 1), the
        all-reduce of step i issued asynchronously after graph i and overlapped with graph i+1.  At small per-GPU sizes
        (strong scaling, N = 8: 2^23 samples per GPU, ~0.1 ms of kernels) the four launches of a step and the Python /
        ctypes time between them are a visible part of it; the graphs remove that.  Returns an error dict when capture is
        not possible."""
        import torch
        d = self.d
        try:
            side = torch.cuda.Stream()
            side.wait_stream(torch.cuda.current_stream())
            graphs = []
            with torch.cuda.stream(side):
                def body(pw, sp):
                    self.os_plan.exec_range_dev(self.x.data_ptr(), self.lo, self.x.numel(), self.y.data_ptr(), self.out_lo, self.out_cnt, sp)
                    self.spec.welch_range_dev(self.y.data_ptr(), self.out_cnt, self.out_lo, self.seg_begin, self.seg_end, self.r, pw.data_ptr(), sp)
                for _ in range(3):
                    body(self.pw[0], side.cuda_stream)
                side.synchronize()
                for i in range(2):
                    g = torch.cuda.CUDAGraph()
                    with torch.cuda.graph(g, stream=side):
                        body(self.pw[i], torch.cuda.current_stream().cuda_stream)
                    graphs.append(g)
            torch.cuda.current_stream().wait_stream(side)
            st = torch.cuda.current_stream()
            pending = [None, None]

            def step(i):
                b = i & 1
                if pending[b] is not None:             # all-reduce of step i-2: long done
                    pending[b].wait()
                    pending[b] = None
                graphs[b].replay()
                if d.pg is not None:
                    pending[b] = d.pg.all_reduce(self.pw[b], async_op=True)
                return self.pw[b]

            def drain():
                for b in range(2):
                    if pending[b] is not None:
                        pending[b].wait()
                        pending[b] = None
            for i in range(max(warmup, 3)):
                step(i)
            drain()
            d.sync_all()
            a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            a.record(st)
            for i in range(steps):
                self.last = step(i)
            drain()
            b.record(st)
            d.sync_all()
            ms = d.max_over_ranks([a.elapsed_time(b) / steps])[0]
            return {"ms_per_step": ms, "value": self.n_global / (ms * 1e-3) / 1e9,
                    "what": "conv + Welch replayed from CUDA graphs, async all-reduce overlapped with the next graph"}
        except Exception as e:                          # capture not supported in this configuration
            return {"error": str(e)[:200]}

    def check(self):
        """Outside the timed region: what the timed pipeline left in `y` / `pw` against independent computations.
        conv: two 2^16-output windows of y (the start of this rank's range -- the shard boundary -- and an interior one)
        against the Float64 oracle run on the matching input slice; PSD: the all-reduced power vector against a
        Float64 torch.fft Welch estimate of the same y (window product, |.|^2, mean over ALL ranks' segments)."""
        import torch
        from oracle import dspbase as od
        d = self.d
        cnt = min(1 << 16, self.out_cnt)
        worst = 0.0
        for a in sorted({self.out_lo, self.out_lo + (self.out_cnt - cnt) // 2 // 2 * 2}):
            x_lo = max(a - (NV - 1), 0)
            xs = self.x[x_lo - self.lo: a + cnt - self.lo].cpu().numpy().astype(np.complex128)
            ref = od.conv_exact(xs, self.taps)[a - x_lo: a - x_lo + cnt]
            got = self.y[a - self.out_lo: a - self.out_lo + cnt].cpu().numpy()
            worst = max(worst, float(np.linalg.norm(got - ref) / np.linalg.norm(ref)))
        acc = torch.zeros(NSEG, dtype=torch.float64, device=d.dev)
        w = torch.from_numpy(self.win).to(d.dev)
        first = self.seg_begin * self.hop - self.out_lo          # local index of this rank's first segment
        nloc = max(0, self.seg_end - self.seg_begin)
        view = self.y[first:].unfold(0, NSEG, self.hop) if nloc > 0 else None
        for b0 in range(0, nloc, 1024):
            z = view[b0: min(b0 + 1024, nloc)].to(torch.complex128) * w
            acc += (torch.fft.fft(z, dim=1).abs() ** 2).sum(dim=0)
        if d.pg is not None:
            d.pg.all_reduce(acc)
        ref = (acc / self.r).cpu().numpy()
        got = self.last.cpu().numpy().astype(np.float64)
        perr = float(np.linalg.norm(got - ref) / np.linalg.norm(ref))
        ok = worst < 1e-6 and perr < 1e-6
        return {"conv_relerr_vs_oracle_f64": worst, "welch_relerr_vs_f64_fft_of_y": perr, "tolerance": 1e-6, "ok": bool(ok),
                "what": "post-timing contents of y (2 windows of 2^16 outputs incl. the shard boundary) and of the all-reduced PSD"}


def e2e_legs(d, cw, args):
    """End to end through the repo's public API (dspb200.conv / dspb200.welch_pgram, the mirror of the reference's
    calls): every step copies the step's input from PINNED host memory to the GPU, filters, estimates the PSD and
    reads the PSD back.  Pipeline form: the filter output stays in HBM between the two calls (DeviceArray), so the
    stream crosses PCIe once.  `e2e_host_calls` is the same step through the two host-pointer C-ABI calls
    (dspb200_os_exec + dspb200_welch_exec), where the filter output comes back to the host and is uploaded again."""
    import torch
    import dspb200
    n, rank = cw.n, d.rank
    xh = torch.empty(n, dtype=torch.complex64).pin_memory()
    xh.copy_(cw.x[(rank * n - cw.lo): (rank * n - cw.lo) + n].cpu())
    yh = torch.empty(n, dtype=torch.complex64).pin_memory()
    ph = torch.empty(NSEG, dtype=torch.float32).pin_memory()
    k_local = (n - NSEG) // cw.hop + 1
    r_local = k_local * cw.norm2
    reps = max(2, min(args.steps, 5))

    def timed(fn):
        fn()
        d.sync_all()
        t0 = time.perf_counter()
        for _ in range(reps):
            fn()
        torch.cuda.synchronize()
        return d.max_over_ranks([(time.perf_counter() - t0) / reps])[0]

    wcfg = dspb200.WelchConfig(n, np.complex64, n=NSEG, noverlap=NOVERLAP, onesided=False, nfft=NSEG, window=cw.win)
    result = {}

    def e2e_step():
        # pinned host pointer in, PSD (host numpy) out: dspb200.filt_welch streams the input through the GPU in chunks,
        # copy of chunk c+1 overlapping the convolution and the Welch accumulation of chunk c
        result["p"] = dspb200.filt_welch(xh.data_ptr(), n, cw.taps, wcfg, nfft=(args.nfft or None)).power

    e2e = None
    if hasattr(dspb200, "filt_welch"):
        dt = timed(e2e_step)
        e2e = {"value": cw.n_global / dt / 1e9, "unit": "Gsamples/s", "ms_per_step": dt * 1e3,
               "h2d_bytes_per_step": int(n * 8), "d2h_bytes_per_step": int(NSEG * 4),
               "note": "public API dspb200.filt_welch(x_host_pinned, taps, WelchConfig): chunked H2D overlapped with conv + Welch "
                       "accumulate per chunk, PSD to host"}
    xd = dspb200.DeviceArray((n,), np.complex64)

    def e2e_serial_step():
        xd.copy_from_host_ptr(xh.data_ptr(), n * 8)                                  # H2D, pinned
        yd = dspb200.conv(xd, cw.taps, algorithm="fft_overlapsave", nfft=(args.nfft or None))
        result["p"] = dspb200.welch_pgram(yd[:n], wcfg).power                        # D2H of the PSD

    dts = timed(e2e_serial_step)
    e2e_serial = {"value": cw.n_global / dts / 1e9, "unit": "Gsamples/s", "ms_per_step": dts * 1e3,
                  "h2d_bytes_per_step": int(n * 8), "d2h_bytes_per_step": int(NSEG * 4),
                  "note": "public API, two calls: to-device copy from pinned host memory -> dspb200.conv -> dspb200.welch_pgram -> PSD to host"}
    if e2e is None:
        e2e = e2e_serial

    def e2e_host_step():
        cw.os_plan.exec_ptr(xh.data_ptr(), n, 1, yh.data_ptr(), n)             # filt-style same-length output
        cw.spec.welch_ptr(yh.data_ptr(), n, r_local, ph.data_ptr())

    dth = timed(e2e_host_step)
    e2e_host = {"value": cw.n_global / dth / 1e9, "unit": "Gsamples/s", "ms_per_step": dth * 1e3,
                "h2d_bytes_per_step": int(2 * n * 8), "d2h_bytes_per_step": int(n * 8 + NSEG * 4),
                "note": "two host-pointer C-ABI calls (dspb200_os_exec + dspb200_welch_exec), pinned buffers, chunked copy/compute overlap"}
    del xd
    return e2e, e2e_serial, e2e_host


def time_on_stream(fn, steps, warmup=3):
    import torch
    st = torch.cuda.current_stream()
    for _ in range(max(warmup, 3)):
        fn()
    torch.cuda.synchronize()
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record(st)
    for _ in range(steps):
        fn()
    b.record(st)
    torch.cuda.synchronize()
    return a.elapsed_time(b) / steps


def run_ours(args):
    import torch
    from dspb200 import _lib
    if args.workload != "conv_welch":
        return run_other_workload(args)
    d = Dist()
    world, rank = d.world, d.rank
    n = 1 << args.log2n                    # samples per rank (weak scaling: the driver's contract line)
    cw = ConvWelch(d, n, args.nfft)

    # clocks / throttle reasons are sampled from the warm-up through the device-timed and end-to-end regions
    clocks = ClockSampler(d.local_rank)
    if rank == 0:
        clocks.start()
    res = cw.time(args.steps, args.warmup)
    if args.dump_outputs:
        dump_outputs(args.dump_outputs, {"conv_out": cw.y, "welch_psd": cw.last}, d)
    chk = cw.check() if not args.no_check else None

    e2e = e2e_serial = e2e_host = None
    if not args.no_e2e:
        e2e, e2e_serial, e2e_host = e2e_legs(d, cw, args)
    clk = clocks.stop() if rank == 0 else None

    # ---- strong scaling: ONE 2^log2n-sample stream range-sharded over the N ranks (BASELINE: ">= 6x at 8 GPUs")
    strong = None
    if world > 1 and not args.no_strong:
        n_s = n // world
        cws = ConvWelch(d, n_s, args.nfft)
        rs = cws.time(args.steps, args.warmup)
        cs = cws.check() if not args.no_check else None
        rg = cws.time_graph(args.steps, args.warmup) if args.graph else None      # opt-in: NCCL inside a captured graph
        cg = cws.check() if (not args.no_check and rg and "value" in rg) else None
        strong = {"scaling": "strong", "samples_total": n, "samples_per_gpu": n_s, "value": rs["value"], "unit": "Gsamples/s",
                  "ms_per_step": rs["ms_per_step"], "stages_ms": {"conv": rs["conv_ms"], "welch": rs["welch_ms"]},
                  "check": cs, "cuda_graph": dict(rg, check=cg) if rg else None,
                  "note": "speed-up = value / the N = 1 run's value (same 2^%d-sample stream); the all-reduce of step i "
                          "overlaps the convolution of step i+1" % args.log2n}
        del cws

    # ---- Welch on a real Float32 stream (BASELINE config 3) -- reported beside the headline, rank 0, N = 1 only
    extra = {}
    hop = NSEG - NOVERLAP
    if world == 1 and not args.no_extra:
        xr = torch.randn(n, device=d.dev, dtype=torch.float32)
        spec_r = _lib.SpecPlan(np.float32, NSEG, NOVERLAP, NSEG, True, cw.win)
        pr = torch.zeros(NSEG // 2 + 1, dtype=torch.float32, device=d.dev)
        k3 = (n - NSEG) // hop + 1
        ms3 = time_on_stream(lambda: spec_r.welch_dev(xr.data_ptr(), n, k3 * cw.norm2, pr.data_ptr(), cw.sp), args.steps)
        extra["welch_f32_config3"] = {"ms": ms3, "gsamples_s": n / (ms3 * 1e-3) / 1e9,
                                      "hbm_gbs_algorithmic": 4.0 * n / (ms3 * 1e-3) / 1e9}

    if rank != 0:
        d.close()
        return

    peak, peak_src = measured_peak_gbs()
    conv_ms, welch_ms = res["conv_ms"], res["welch_ms"]
    conv_bytes = 16.0 * cw.out_cnt                    # 8 B read + 8 B written per ComplexF32 sample (SURVEY.md 8d)
    achieved = conv_bytes / (conv_ms * 1e-3) / 1e9
    welch_bytes = 8.0 * cw.out_cnt
    kc = kernel_counters()
    ck = kc.get("conv_cf32_4097taps_2^26", {}) if (args.log2n == 26 and cw.os_plan.fused and cw.os_plan.nfft == 16384) else {}
    conv_kernel = ck.get("kernel") or ("fused overlap-save kernel, nfft = %d" % cw.os_plan.nfft if cw.os_plan.fused else "cuFFT pipeline")
    sm_mhz = (clk or {}).get("sm_mhz") or 1965.0
    fp32_issue = None
    if ck.get("inst_executed"):
        # issue-slot roofline: one warp instruction per scheduler per cycle, 4 schedulers x 148 SMs
        t_issue_ms = ck["inst_executed"] / (4 * 148 * sm_mhz * 1e6) * 1e3
        fp32_issue = {"warp_instructions_per_launch": ck["inst_executed"], "sm_mhz": sm_mhz, "min_ms_at_full_issue": t_issue_ms,
                      "frac": t_issue_ms / conv_ms, "source": ck.get("source")}
    cpu_workers = os.cpu_count() or 1
    cb = None
    if world == 1 and not args.no_cpu:
        if d.orig_affinity:
            os.sched_setaffinity(0, d.orig_affinity)       # the CPU leg uses every host core again
        ns, ts = time_cpu_baseline(min(args.log2n, 25), 2, cpu_workers, warm_full=1)
        cb = {"value": ns / float(np.mean(ts)) / 1e9, "unit": "Gsamples/s", "cores": cpu_workers, "kind": "port",
              "sample": f"2^{min(args.log2n, 25)} samples x 2 reps (after one untimed) of the same two stages; oracle port (numpy + "
                        f"scipy pocketfft, Float32, nfft 65536 as the reference picks), ranges of whole blocks / segments on "
                        f"{cpu_workers} threads; Julia/FFTW not installable here"}
    line = {
        "metric": METRIC, "value": res["value"], "unit": "Gsamples/s", "n_gpus": world, "steps": args.steps,
        "warmup": max(args.warmup, 3), "ms_per_step": res["ms_per_step"], "higher_is_better": True, "scaling": "weak",
        "vs_baseline": None, "dtype": "c64 (ComplexF32; f32 arithmetic)", "data": "synthetic",
        "config": {"workload": f"conv overlap-save 4097-tap FIR + welch_pgram(n=nfft=4096, 50% overlap, hanning, two-sided) "
                               f"on 2^{args.log2n} ComplexF32 samples per GPU (BASELINE configs[1] + Welch stage)",
                   "samples_per_gpu": n, "nfft_conv": cw.os_plan.nfft, "conv_fused": cw.os_plan.fused,
                   "l2_policy": "inputs (512 MiB per stage) exceed the 126 MB L2; no explicit flush",
                   "parallelism": f"stream range-sharded over {world} GPU(s); async NCCL all-reduce of the 4096-bin Welch power "
                                  "only, overlapped with the next step's convolution"},
        "stages_ms": {"conv": conv_ms, "welch": welch_ms},
        "roofline": {"bound": "hbm", "kernel": conv_kernel,
                     "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak, "peak_source": peak_src,
                     "algorithmic_bytes_per_launch": conv_bytes,
                     # dram__bytes_read.sum + dram__bytes_write.sum of one launch, from the committed `ncu --set full` capture
                     "traffic": ck.get("dram_bytes") if world == 1 else None, "traffic_source": ck.get("source"),
                     "fp32_issue": fp32_issue,
                     "welch_stage": {"achieved": welch_bytes / (welch_ms * 1e-3) / 1e9, "frac": welch_bytes / (welch_ms * 1e-3) / 1e9 / peak,
                                     "algorithmic_bytes_per_launch": welch_bytes}},
        "check": chk, "strong": strong,
        "cpu_baseline": cb, "e2e": e2e, "e2e_two_calls": e2e_serial, "e2e_host_calls": e2e_host,
        "gpu_launches": res["launches"], "clocks": clk, "extra": extra,
    }
    print(json.dumps(line))
    d.close()


# ------------------------------------------------------------------------------------------- other BASELINE configs

def run_other_workload(args):
    """--workload welch_real | spectrogram | resample: BASELINE configs[2], [3], [4] as bench lines of their own
    (same JSON contract; device-resident inputs, CUDA events, max over ranks).
      welch_real   2^log2n Float32 samples per GPU, n = nfft = 4096, 50 %, hanning; segment-range shard + PSD all-reduce
      spectrogram  64 channels x 2^22 Float32, n = nfft = 1024, 75 % overlap; the 64 channels are split over the ranks
                   (strong scaling by construction, no collective)
      resample     3//2 polyphase on 2^log2n ComplexF32 per GPU (Float32 taps): contiguous output ranges, no collective
      filt_columns filt(b, 1, x) with the 257-tap FIR of BASELINE configs[0] on a 2^20 x 64 Float32 matrix (time-domain
                   kernel and the overlap-save fftfilt on the same columns); the 64 columns are split over the ranks
                   (SURVEY.md 8e row 5), no collective"""
    import torch
    from fractions import Fraction
    import dspb200
    from dspb200 import _lib, sharding
    d = Dist()
    world, rank, dev = d.world, d.rank, d.dev
    st = torch.cuda.current_stream()
    sp = st.cuda_stream
    peak, peak_src = measured_peak_gbs()
    clocks = ClockSampler(d.local_rank)
    if rank == 0:
        clocks.start()
    wl = args.workload
    if wl == "spectrogram":
        nchan, length, nn, nov = 64, 1 << 22, 1024, 768
        c0, c1 = sharding.channel_shard(nchan, world, rank)
        x = torch.randn((c1 - c0) * length, device=dev, dtype=torch.float32)
        plan = _lib.SpecPlan(np.float32, nn, nov, nn, True, None)
        k = (length - nn) // (nn - nov) + 1
        out = torch.empty((nn // 2 + 1) * k * (c1 - c0), device=dev, dtype=torch.float32)
        fn = lambda: plan.stft_dev(x.data_ptr(), length, c1 - c0, float(nn), True, out.data_ptr(), sp)   # noqa: E731
        outputs = {"spectrogram_power": out}
        units, unit = nchan * length, "Gsamples/s"
        bytes_local = 4.0 * (c1 - c0) * length + 4.0 * out.numel()
        desc = f"spectrogram 64 ch x 2^22 Float32, n = nfft = 1024, noverlap = 768 (BASELINE configs[3]); channels {c0}..{c1 - 1} on rank 0"
        kernel, scaling, dtype = "stft_w1k_kernel<real> (a warp per 1024-point unit of two packed segments)", "strong", "f32"

        def check():
            # first and last column of this rank's first and last channel against a Float64 FFT of the same samples
            worst, nb_, hop = 0.0, nn // 2 + 1, nn - nov
            for ch in {0, c1 - c0 - 1}:
                for col in (0, k // 2, k - 1):
                    seg = x[ch * length + col * hop: ch * length + col * hop + nn].cpu().numpy().astype(np.float64)
                    pref = np.abs(np.fft.rfft(seg)) ** 2 / nn
                    pref[1:nn // 2] *= 2
                    got = out[(ch * k + col) * nb_: (ch * k + col + 1) * nb_].cpu().numpy()
                    worst = max(worst, float(np.linalg.norm(got - pref) / np.linalg.norm(pref)))
            return worst, 1e-6, "3 columns (first, middle, last) of every rank's first and last channel vs a Float64 FFT"
    elif wl == "filt_columns":
        ncol, length = 64, 1 << 20
        c0, c1 = sharding.channel_shard(ncol, world, rank)
        nn = np.arange(257) - 128
        fir = (0.5 * np.sinc(0.5 * nn) * np.hamming(257)).astype(np.float32)
        x = torch.randn((c1 - c0) * length, device=dev, dtype=torch.float32)
        y = torch.empty_like(x)
        td = args.filt_alg == "td"
        plan = _lib.FirPlan(fir) if td else _lib.OsPlan(fir, 0)
        if td:
            fn = lambda: plan.exec_dev(x.data_ptr(), length, c1 - c0, y.data_ptr(), sp)   # noqa: E731
        else:
            fn = lambda: plan.exec_dev(x.data_ptr(), length, c1 - c0, y.data_ptr(), length, sp)   # noqa: E731
        outputs = {"filt_out": y}
        units, unit = ncol * length, "Gsamples/s"
        bytes_local = 8.0 * (c1 - c0) * length
        desc = (f"filt(b, 1, x) 257-tap FIR on a 2^20 x 64 Float32 matrix (BASELINE configs[0], 64 columns), "
                f"{'time domain (_filt_fir!)' if td else 'overlap-save fftfilt'}; columns {c0}..{c1 - 1} on rank 0")
        kernel = "fir_tile_kernel<float> (FMA-bound: 257 FMAs per sample)" if td else f"os_fused_kernel<float,{plan.nfft},real>"
        scaling, dtype = "strong", "f32"

        def check():
            # head and tail of this rank's last column against the FIR sum in Float64
            col = c1 - c0 - 1
            xh = x[col * length:(col + 1) * length].cpu().numpy().astype(np.float64)
            yh = y[col * length:(col + 1) * length].cpu().numpy()
            full = np.convolve(xh[:4096], fir.astype(np.float64))[:4096]
            tail = np.convolve(xh[-4096 - 256:], fir.astype(np.float64))[256:4096 + 256]
            worst = max(float(np.linalg.norm(yh[:4096] - full) / np.linalg.norm(full)),
                        float(np.linalg.norm(yh[-4096:] - tail) / np.linalg.norm(tail)))
            return worst, (5e-6 if td else 1e-6), ("first and last 4096 outputs of every rank's last column vs the Float64 sum"
                                                    + (" (Float32 fma chain of 257 taps; bit-exactness is pinned by the parity tests)" if td else ""))
    elif wl == "resample":
        # ONE stream of 2^log2n x world samples; rank r computes a contiguous range of the OUTPUT and holds only the input samples
        # that range reads (dspb200_resample_exec_range_dev, global offsets) -- src/Filters/stream_filt.jl:476-515, no collective
        n = 1 << args.log2n
        rate = Fraction(3, 2)
        h = dspb200.resample_filter(rate).astype(np.float32)
        n0, phi0 = dspb200.filters.resample_phase(h.size, rate)
        nx_total, tpp = n * world, -(-h.size // 3)
        nout_total = 3 * nx_total // 2
        sh = sharding.resample_shard(nx_total, nout_total, 3, 2, n0, phi0, tpp, world, rank)
        nx_local = sh.in_end - sh.in_begin
        g = torch.arange(sh.in_begin, sh.in_end, device=dev, dtype=torch.float64)          # a chirp of the GLOBAL sample index:
        ph = (g * g * (0.37 / nx_total)) % 2.0                                             # every rank can generate its own range
        x = torch.polar(torch.ones_like(ph) * 0.5, ph * np.pi).to(torch.complex64).contiguous()
        del g, ph
        plan = _lib.ResamplePlan(np.complex64, h, 3, 2)
        y = torch.empty(sh.out_count, device=dev, dtype=torch.complex64)
        fn = lambda: plan.exec_range_dev(x.data_ptr(), sh.in_begin, nx_local, n0, phi0, y.data_ptr(), sh.j_begin, sh.out_count, sp)   # noqa: E731
        outputs = {"resample_out": y}

        def check():
            # both ends of this rank's output range (the shard boundaries) against the polyphase sum in Float64
            xh = x.cpu().numpy().astype(np.complex128)
            yh = y.cpu().numpy()
            worst = 0.0
            for j0 in (0, sh.out_count // 2, sh.out_count - 256):
                ref = np.zeros(256, np.complex128)
                for jj in range(256):
                    pp = phi0 + (sh.j_begin + j0 + jj) * 2
                    nn_, phi = n0 + pp // 3, pp % 3
                    k = np.arange(phi, h.size, 3)
                    idx = nn_ - np.arange(k.size) - sh.in_begin
                    ok = (idx >= 0) & (idx < nx_local) & (nn_ - np.arange(k.size) < nx_total)
                    ref[jj] = np.sum(h[k][ok].astype(np.float64) * xh[idx[ok]])
                worst = max(worst, float(np.linalg.norm(yh[j0:j0 + 256] - ref) / np.linalg.norm(ref)))
            return worst, 1e-6, "256 outputs at both ends and the middle of every rank's output range vs the polyphase sum in Float64"
        units, unit = nx_total, "Gsamples/s"
        bytes_local = 8.0 * nx_local + 8.0 * sh.out_count
        desc = (f"resample 3//2 of ONE stream of 2^{args.log2n} x {world} ComplexF32 samples, 111 Float32 taps (BASELINE configs[4]); "
                f"rank r holds the input range its contiguous output range reads; outputs {sh.j_begin}..{sh.j_begin + sh.out_count - 1} on rank 0")
        kernel, scaling, dtype = "resample_mp2_kernel<cx<float>,float,cx<float>,3,2,4>", "weak", "c64"
    else:
        n = 1 << args.log2n
        hop = NSEG - NOVERLAP
        win = hanning64(NSEG)
        x = torch.randn(n, device=dev, dtype=torch.float32)
        plan = _lib.SpecPlan(np.float32, NSEG, NOVERLAP, NSEG, True, win)
        k = (n - NSEG) // hop + 1
        pw = torch.zeros(NSEG // 2 + 1, device=dev, dtype=torch.float32)
        r = k * world * float(np.sum(win * win))

        def fn():
            plan.welch_dev(x.data_ptr(), n, r, pw.data_ptr(), sp)
            if d.pg is not None:
                d.pg.all_reduce(pw)
        outputs = {"welch_psd": pw}
        units, unit = n * world, "Gsamples/s"
        bytes_local = 4.0 * n
        desc = f"welch_pgram 2^{args.log2n} Float32 per GPU, n = nfft = 4096, 50 % overlap, hanning (BASELINE configs[2]); PSD all-reduce"
        kernel, scaling, dtype = "welch_fused_kernel<float,4096,real> (3 thread groups per CTA)", "weak", "f32"

        def check():
            # two bin-centred tones: every segment of every rank has the same periodogram, so the all-reduced Welch average
            # must equal the Float64 periodogram of ONE windowed segment (scaling, segment count and the sum over ranks)
            t = torch.arange(n, device=dev, dtype=torch.float64)
            x.copy_((0.7 * torch.cos(t * (2 * np.pi * 300 / NSEG)) + 0.2 * torch.sin(t * (2 * np.pi * 1111 / NSEG))).to(torch.float32))
            fn()
            d.sync_all()
            t1 = np.arange(NSEG, dtype=np.float64)
            seg = (0.7 * np.cos(t1 * (2 * np.pi * 300 / NSEG)) + 0.2 * np.sin(t1 * (2 * np.pi * 1111 / NSEG))) * win
            pref = np.abs(np.fft.rfft(seg)) ** 2 / float(np.sum(win * win))
            pref[1:NSEG // 2] *= 2
            got = pw.cpu().numpy().astype(np.float64)
            return float(np.linalg.norm(got - pref) / np.linalg.norm(pref)), 1e-6, \
                "all-reduced PSD of two bin-centred tones (every segment identical) vs the Float64 periodogram of one segment"
    for _ in range(max(args.warmup, 3)):
        fn()
    d.sync_all()
    l0 = _lib.launch_count()
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record(st)
    for _ in range(args.steps):
        fn()
    b.record(st)
    d.sync_all()
    ms = d.max_over_ranks([a.elapsed_time(b) / args.steps])[0]
    launches = _lib.launch_count() - l0
    clk = clocks.stop() if rank == 0 else None
    if args.dump_outputs:
        dump_outputs(args.dump_outputs, outputs, d)
    chk = None
    if not args.no_check:
        err, tol_, what = check()
        err = d.max_over_ranks([err])[0]
        chk = {"relerr_max_over_ranks": err, "tolerance": tol_, "ok": bool(err <= tol_), "what": what}
    if rank == 0:
        ach = bytes_local / (ms * 1e-3) / 1e9
        print(json.dumps({
            "metric": f"Gsamples/s {wl}", "value": units / (ms * 1e-3) / 1e9, "unit": unit, "n_gpus": world, "steps": args.steps,
            "warmup": max(args.warmup, 3), "ms_per_step": ms, "higher_is_better": True, "scaling": scaling, "vs_baseline": None,
            "dtype": dtype, "data": "synthetic", "config": {"workload": desc, "l2_policy": "inputs exceed the 126 MB L2; no explicit flush"},
            "roofline": {"bound": "hbm", "kernel": kernel, "achieved": ach, "peak": peak, "unit": "GB/s", "frac": ach / peak,
                         "peak_source": peak_src, "algorithmic_bytes_per_launch": bytes_local, "traffic": None},
            "check": chk, "gpu_launches": int(launches), "clocks": clk}))
    d.close()
    if chk is not None and not chk["ok"]:
        sys.exit(3)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--log2n", type=int, default=26)
    ap.add_argument("--nfft", type=int, default=0, help="overlap-save block transform (0 = library choice)")
    ap.add_argument("--workload", default="conv_welch", choices=["conv_welch", "welch_real", "spectrogram", "resample", "filt_columns"])
    ap.add_argument("--filt-alg", default="fft", choices=["fft", "td"], help="filt_columns: overlap-save fftfilt or the time-domain kernel")
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--no-cpu", action="store_true")
    ap.add_argument("--no-extra", action="store_true")
    ap.add_argument("--no-check", action="store_true")
    ap.add_argument("--no-strong", action="store_true")
    ap.add_argument("--graph", action="store_true", help="also time the strong-scaling step replayed from one CUDA graph")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="after the timed steps, write the outputs of the last step as DIR/<name>.npy (see dump_outputs)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "ours":
        ap.error("--dump-outputs writes the outputs of the GPU path (--impl ours)")
    if args.impl == "reference":
        run_reference(args)
    else:
        run_ours(args)


if __name__ == "__main__":
    main()
