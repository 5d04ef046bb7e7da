"""Kernel-only timing of the fused STFT (nfft = 1024, Float32) over a few shapes: channels x length, hop, window.
    python profiles/stft_shapes_probe.py"""
import os
import sys

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import bench  # noqa: E402
from dspb200 import _lib  # noqa: E402

dev = torch.device("cuda", 0)
st = torch.cuda.current_stream()


def timeit(fn, reps=10):
    for _ in range(3):
        fn()
    torch.cuda.synchronize()
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record(st)
    for _ in range(reps):
        fn()
    b.record(st)
    torch.cuda.synchronize()
    return a.elapsed_time(b) / reps


for nchan, log2len, nov, usewin in ((64, 22, 768, False), (64, 22, 768, True), (1, 22, 768, False), (1, 22, 512, False), (1, 22, 512, True),
                                    (4, 22, 512, True), (1, 26, 512, True)):
    length = 1 << log2len
    x = torch.randn(nchan * length, device=dev)
    plan = _lib.SpecPlan(np.float32, 1024, nov, 1024, True, bench.hanning64(1024) if usewin else None)
    k = plan.nsegments(length)
    out = torch.empty(513 * k * nchan, device=dev)
    ms = timeit(lambda: plan.stft_dev(x.data_ptr(), length, nchan, 1024.0, True, out.data_ptr(), 0))
    print(f"nchan={nchan:3d} len=2^{log2len} noverlap={nov} window={usewin}: {ms:.4f} ms  ({nchan * length / ms / 1e6:.1f} Gsamples/s)")
    del x, out
