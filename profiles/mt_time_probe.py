"""Where does the host-array spectrogram spend its time (plan creation / exec / close)?"""
import os
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import dspb200 as dsp  # noqa: E402
from dspb200 import _lib  # noqa: E402
from dspb200.periodograms import compute_window  # noqa: E402

rng = np.random.default_rng(5)
x = rng.standard_normal(1 << 22).astype(np.float32)
win, norm2 = compute_window(dsp.hanning, 1024)
k = (x.size - 1024) // 512 + 1
out = np.zeros((513, k, 1), dtype=np.float32, order="F")
sig = np.asfortranarray(x.reshape(-1, 1))
for rep in range(4):
    t0 = time.perf_counter()
    plan = _lib.SpecPlan(np.float32, 1024, 512, 1024, True, win)
    t1 = time.perf_counter()
    plan.stft(sig, x.size, 1, norm2, True, out)
    t2 = time.perf_counter()
    plan.stft(sig, x.size, 1, norm2, True, out)
    t3 = time.perf_counter()
    plan.close()
    t4 = time.perf_counter()
    print(f"create {1e3 * (t1 - t0):.2f} ms, exec#1 {1e3 * (t2 - t1):.2f}, exec#2 {1e3 * (t3 - t2):.2f}, close {1e3 * (t4 - t3):.2f}")
