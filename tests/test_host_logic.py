"""CPU-only tests of the product's host logic (no kernels run): it must agree with the oracle's restatement of the
reference's scalar helpers, and the C-ABI library must load and export every symbol include/dspb200.h declares."""
import ctypes
import os
import re
import subprocess
from fractions import Fraction

import numpy as np
import pytest

from conftest import ROOT, approx

import dspb200 as dsp
from oracle import dspbase as od
from oracle import filters as of
from oracle import util as ou
from oracle import windows as ow


def test_capi_exports_every_declared_symbol():
    hdr = open(os.path.join(ROOT, "include", "dspb200.h")).read()
    declared = set(re.findall(r"DSPB200_API\s+[\w\s\*]+?\b(dspb200_\w+)\s*\(", hdr))
    assert len(declared) >= 40
    lib = ctypes.CDLL(os.path.join(ROOT, "dsp.jl_b200", "libdspb200.so"))
    for name in sorted(declared):
        assert hasattr(lib, name), f"{name} declared in include/dspb200.h but not exported"
    assert declared == set(dsp._lib.SIGNATURES), "ctypes binding and header disagree"
    assert lib.dspb200_version() == 100
    out = subprocess.run(["nm", "-D", "--defined-only", os.path.join(ROOT, "dsp.jl_b200", "libdspb200.so")],
                         capture_output=True, text=True).stdout
    exported = set(re.findall(r" T (dspb200_\w+)", out))
    assert exported == declared


def test_library_is_sm100a_only():
    out = subprocess.run(["cuobjdump", "--list-elf", os.path.join(ROOT, "dsp.jl_b200", "libdspb200.so")],
                         capture_output=True, text=True)
    if out.returncode != 0:
        pytest.skip("cuobjdump unavailable")
    archs = set(re.findall(r"sm_\d+a?", out.stdout))
    assert archs == {"sm_100a"}, archs


def test_no_cpu_fallback_without_device():
    if dsp.device_count() > 0:
        pytest.skip("a CUDA device is present")
    with pytest.raises(dsp.DSPB200Error):
        dsp.conv(np.ones(300), np.ones(300), algorithm="fft_overlapsave")
    with pytest.raises(dsp.DSPB200Error):
        dsp.welch_pgram(np.arange(64.0), 8, 4, window=None)
    with pytest.raises(dsp.DSPB200Error):
        dsp.filt(np.ones(3), 1.0, np.ones(10))
    with pytest.raises(dsp.DSPB200Error):
        dsp.resample(np.ones(10), Fraction(3, 2))


def test_product_never_imports_oracle():
    pkg = os.path.join(ROOT, "dsp.jl_b200")
    for fn in os.listdir(pkg):
        if fn.endswith(".py"):
            src = open(os.path.join(pkg, fn)).read()
            assert "oracle" not in src, fn


def test_scalar_helpers_match_oracle():
    for n in list(range(1, 300)) + [1000, 1001, 4097, 65537, 10 ** 6 + 3]:
        assert dsp.nextfastfft(n) == ou.nextfastfft(n), n
    assert dsp.nextfastfft((65, 127)) == (70, 128)
    for nb, nx in [(1, 3), (257, 2 ** 20), (4097, 2 ** 26), (67, 2 ** 20), (127, 2 ** 18 - 1), (12, 128), (128, 128)]:
        assert dsp.optimalfftfiltlength(nb, nx) == od.optimalfftfiltlength(nb, nx)
    for n in (1, 2, 8, 128, 4096):
        # independent evaluations of the same closed forms: equal to a few ulp of the window scale
        assert np.allclose(dsp.hanning(n), ow.hanning(n), rtol=0, atol=1e-15)
        assert np.allclose(dsp.hamming(n), ow.hamming(n), rtol=0, atol=1e-15)
        assert np.array_equal(dsp.rect(n), ow.rect(n))
        assert np.allclose(dsp.bartlett(n), ow.bartlett(n), rtol=0, atol=1e-15)
        assert np.allclose(dsp.kaiser(n, 1.8), ow.kaiser(n, 1.8), rtol=1e-12, atol=0)
        assert dsp.hanning(n)[0] == (1.0 if n == 1 else 0.0) and dsp.hanning(n)[-1] == (1.0 if n == 1 else 0.0)
    for dt in (np.float32, np.float64, np.complex64, np.complex128, np.int64, np.int32):
        assert dsp.fftintype(dt) == ou.fftintype(dt)
        assert dsp.fftouttype(dt) == ou.fftouttype(dt)
        assert dsp.fftabs2type(dt) == ou.fftabs2type(dt)
    assert np.array_equal(dsp.rfftfreq(9, 2.0), ou.rfftfreq(9, 2.0)) and np.array_equal(dsp.fftfreq(9, 2.0), ou.fftfreq(9, 2.0))
    assert np.array_equal(dsp.fftfreq(8, 1.0), ou.fftfreq(8, 1.0))


def test_windows_matlab_goldens(goldens):
    assert approx(dsp.hanning(128), goldens["hanning128"])
    assert approx(dsp.hamming(128), goldens["hamming128"])
    assert approx(dsp.bartlett(128), goldens["bartlett128"])
    assert approx(dsp.kaiser(128, 0.4 / np.pi), goldens["kaiser128_0.4"])


def test_resample_host_side(goldens):
    for rate in ("1/2", "2/1", "3/2", "2/3", "5/9", "14/17", "23/1", "1/21"):
        r = Fraction(rate)
        assert np.allclose(dsp.resample_filter(r), of.resample_filter(r), rtol=1e-14, atol=0)
        for hlen in (41, 61, 56, 111, 6):
            sf = of.FIRFilterState(np.zeros(hlen), r)
            sf.setphase(sf.timedelay())
            n0, phi0 = dsp.resample_phase(hlen, r)
            assert (n0, phi0) == (sf.input_deficit - 1, sf.phi_idx - 1), (rate, hlen)
    assert dsp.kaiserord(0.2 / 3) == of.kaiserord(0.2 / 3)
    if dsp.device_count() == 0:                    # with a device the float-rate path runs (test_arbitrary_rate_resample)
        with pytest.raises(dsp.DSPB200Error):      # float rate = arbitrary-rate GPU path: fails loudly without a device
            dsp.resample(np.ones(10), 1.5)


def test_argument_checks_raise_reference_exception_types():
    x = np.arange(8.0)
    with pytest.raises(dsp.ArgumentError):
        dsp.filt(np.zeros(0), 1.0, x)
    with pytest.raises(dsp.ArgumentError):
        dsp.filt(np.ones(2), np.zeros(0), x)
    with pytest.raises(dsp.ArgumentError):
        dsp.filt(np.ones(2), 0.0, x)
    with pytest.raises(dsp.ArgumentError):
        dsp.filt_(np.zeros(3), np.ones(2), 1.0, x)
    with pytest.raises(dsp.ArgumentError):
        dsp.fftfilt_(np.zeros(3), np.ones(2), x)
    with pytest.raises(TypeError):
        dsp.fftfilt(np.ones(2) * 1j, x)
    with pytest.raises(dsp.ArgumentError):
        dsp.conv(np.ones(300), np.ones(300), algorithm="bogus")
    with pytest.raises(dsp.ArgumentError):
        dsp.periodogram(x * 1j, onesided=True)
    with pytest.raises(dsp.DomainError):
        dsp.periodogram(x, nfft=4)
    with pytest.raises(dsp.DomainError):
        dsp.welch_pgram(x, 4, 4, window=None)
    with pytest.raises(dsp.DomainError):
        dsp.welch_pgram(x, 4, 2, nfft=3, window=None)
    with pytest.raises(dsp.DimensionMismatch):
        dsp.welch_pgram(x, 4, 2, window=np.ones(3))
    with pytest.raises(dsp.ArgumentError):
        dsp.stft(x * 1j, 4, 2, onesided=True)
    assert dsp.arraysplit_count(1000, 100, 10) == 11 and dsp.arraysplit_count(3, 4, 1) == 0


def test_host_fft_core_emulation():
    """The shared-memory FFT core (fft_core.cuh) compiled for the host and run pass by pass, vs a double DFT."""
    exe = os.path.join(ROOT, "build", "fft_core_host_check")
    os.makedirs(os.path.dirname(exe), exist_ok=True)
    src = os.path.join(ROOT, "tests", "host", "fft_core_host_check.cu")
    if not os.path.exists(exe) or os.path.getmtime(exe) < max(os.path.getmtime(src), os.path.getmtime(
            os.path.join(ROOT, "dsp.jl_b200", "csrc", "fft_core.cuh"))):
        subprocess.run(["g++", "-std=c++17", "-O2", "-x", "c++", "-w", "-I/usr/local/cuda/include", "-o", exe, src], check=True)
    out = subprocess.run([exe], capture_output=True, text=True)
    assert out.returncode == 0 and "ALL OK" in out.stdout, out.stdout


def test_host_fir_tile_emulation():
    """The register-tiled FIR kernel body (fir_tile.cuh) compiled for the host: every "thread" of a CTA in turn, all four
    element types, tap counts around the chunk / staging-round boundaries, bit for bit against the literal fma chain."""
    exe = os.path.join(ROOT, "build", "fir_tile_host_check")
    os.makedirs(os.path.dirname(exe), exist_ok=True)
    src = os.path.join(ROOT, "tests", "host", "fir_tile_host_check.cu")
    if not os.path.exists(exe) or os.path.getmtime(exe) < max(os.path.getmtime(src), os.path.getmtime(
            os.path.join(ROOT, "dsp.jl_b200", "csrc", "fir_tile.cuh"))):
        subprocess.run(["g++", "-std=c++17", "-O2", "-march=native", "-x", "c++", "-w", "-I/usr/local/cuda/include", "-o", exe, src],
                       check=True)
    out = subprocess.run([exe], capture_output=True, text=True)
    assert out.returncode == 0 and out.stdout.strip().endswith("OK"), out.stdout[-2000:]


def test_inputlength_outputlength_invariants():
    # test/resample.jl:154-182 (FIRDecimator, FIRInterpolator, FIRRational), pure host arithmetic
    import random
    rnd = random.Random(1776)
    for _ in range(1000):
        M = Fraction(rnd.randint(1, 10), rnd.randint(1, 10))
        H = dsp.FIRFilter(np.zeros(rnd.randint(1, 100)) + 1.0, M)
        if M != 1:
            H.setphase(10 * rnd.random())
        yL = rnd.randint(1, 100)
        assert H.outputlength(H.inputlength(yL)) <= yL < H.outputlength(H.inputlength(yL) + 1)
        assert H.outputlength(H.inputlength(yL, True) - 1) < yL <= H.outputlength(H.inputlength(yL, True))
        O = of.FIRFilterState(np.zeros(H.hlen), M)
        O.phi_idx, O.input_deficit = H.phi_idx, H.input_deficit
        assert O.outputlength(37) == H.outputlength(37) and O.inputlength(yL, True) == H.inputlength(yL, True)


def test_dpss_host_matches_oracle_and_matlab(goldens):
    d = dsp.dpss(128, 4)
    assert approx(d, goldens["dpss128_4"])
    o = ow.dpss(128, 4)
    for c in range(7):            # the reference leaves the sign of symmetric tapers to LAPACK; compare up to sign
        assert min(np.abs(d[:, c] - o[:, c]).max(), np.abs(d[:, c] + o[:, c]).max()) < 1e-12
    with pytest.raises(dsp.DomainError):
        dsp.dpss(10, 6)
    # dpsseig (src/windows.jl:739-775): concentration ratios, product vs oracle; the leading tapers are ~1
    e, eo = dsp.dpsseig(d, 4), ow.dpsseig(o, 4)
    assert np.allclose(e, eo, rtol=1e-12) and e[0] > 0.999999 and np.all(np.diff(e) < 0) and 0.5 < e[-1] < 1
    with pytest.raises(dsp.DomainError):
        dsp.dpsseig(d, 64)


def test_arbitrary_rate_design_and_length_bookkeeping():
    # resample_filter(rate::AbstractFloat, Nphi): test/resample.jl:142-151
    ratio, nphi = 3.141592653589793, 32
    h = dsp.resample_filter(ratio, nphi)
    assert np.allclose(h, of.resample_filter_arb(ratio, nphi), rtol=1e-14, atol=1e-17)
    k = np.arange(h.size)
    assert abs(abs(np.sum(h)) - nphi) < 1e-9
    assert abs(abs(np.sum(h * np.exp(-1j * np.pi / nphi * k))) - nphi / 2) < 1e-3 * nphi / 2
    assert np.allclose(dsp.resample_filter(0.37), of.resample_filter_arb(0.37), rtol=1e-14, atol=1e-17)
    # FIRFilter{FIRArbitrary} inputlength / outputlength invariants: test/resample.jl:167-180 (no device work involved)
    rng = np.random.default_rng(42)
    for _ in range(300):
        M = 10 * rng.random() + 1e-3
        H = dsp.FIRFilter(np.zeros(int(rng.integers(1, 101))), float(M))
        O = of.FIRArbitraryState(np.zeros(H.hlen), float(M))
        ph = 10 * rng.random()
        H.setphase(ph)
        O.setphase(ph)
        assert (H.input_deficit, H.phi_accumulator, H.phi_idx) == (O.input_deficit, O.acc, O.phi_idx)
        yL = int(rng.integers(1, 101))
        assert H.inputlength(yL) == O.inputlength(yL) and H.inputlength(yL, True) == O.inputlength(yL, True)
        assert H.outputlength(H.inputlength(yL)) <= yL < H.outputlength(H.inputlength(yL) + 1)
        assert H.outputlength(H.inputlength(yL, True) - 1) < yL <= H.outputlength(H.inputlength(yL, True))
    H = dsp.FIRFilter(None, 2.0)
    H.setphase(H.timedelay())
    assert H.outputlength(H.inputlength(200)) <= 200 < H.outputlength(H.inputlength(200) + 1)
    with pytest.raises(dsp.DomainError):
        dsp.FIRFilter(np.ones(4), -1.0)


def test_arbitrary_rate_exact_counting_matches_literal_accumulator():
    # the product counts the outputs of a FIRArbitrary filt! call in exact rational arithmetic; the reference runs a
    # Float64 accumulator loop (src/Filters/stream_filt.jl:567-625).  Random rates, phases and chunk lengths: same
    # number of outputs, same inputDeficit carry, accumulator within rounding noise.
    from dspb200.filters import _arb_advance
    rng = np.random.default_rng(123)
    worst = 0.0
    for _ in range(150):
        rate = float(10 ** rng.uniform(-1.5, 1.2))
        nphi = int(rng.choice([3, 8, 32]))
        O = of.FIRArbitraryState(np.ones(int(rng.integers(1, 40))), rate, nphi)
        O.setphase(float(10 * rng.random()))
        for _ in range(5):
            xlen = int(rng.integers(0, 60))
            acc, deficit = O.acc, O.input_deficit
            y = O.filt(np.zeros(xlen))
            if xlen < deficit:
                assert len(y) == 0 and O.input_deficit == deficit - xlen and O.acc == acc
                continue
            nout, new_deficit, new_acc = _arb_advance(acc, deficit, nphi / rate, nphi, xlen)
            assert (len(y), O.input_deficit) == (nout, new_deficit)
            worst = max(worst, abs(O.acc - new_acc))
    assert worst < 1e-10


def test_arbitrary_rate_host_state_machine_with_a_numpy_stand_in_for_the_kernel(monkeypatch):
    # The stateful FIRFilter(h, rate::float) wrapper (history / inputDeficit / phiAccumulator carry, [history; x] layout,
    # n0) is exercised on the CPU by replacing the device plan with a numpy model of resample_arb_kernel's contract.
    from fractions import Fraction as Fr
    from dspb200 import _lib

    class FakePlan:
        def __init__(self, dtype_x, h, nphases):
            self.h, self.n = np.asarray(h, dtype=np.float64), int(nphases)
            self.out_dtype = np.result_type(np.dtype(dtype_x), self.h.dtype)
            self.pfb = of.taps2pfb(self.h, self.n)
            self.dpfb = of.taps2pfb(np.concatenate([np.diff(self.h), [0.0]]), self.n)

        def exec(self, xe, nx, n0, acc0, delta, out, nout):
            tpp = self.pfb.shape[0]
            for j in range(nout):
                P = Fr(acc0) + j * Fr(delta)
                q = P // self.n
                r = float(P - q * self.n)
                phi, alpha = int(np.floor(r)), r - np.floor(r)
                first = n0 + int(q) - (tpp - 1)
                win = np.array([xe[i] if 0 <= i < nx else 0.0 for i in range(first, first + tpp)])
                out[j] = np.dot(self.dpfb[:, phi], win) * alpha + np.dot(self.pfb[:, phi], win)

        def close(self):
            pass

    monkeypatch.setattr(_lib, "ResampleArbPlan", FakePlan)
    rng = np.random.default_rng(5)
    for rate in (0.7312, 1.2957, 2.618, 1 / 55.55):
        h = dsp.resample_filter(rate, 32)
        x = rng.standard_normal(300)
        want = of.FIRArbitraryState(h, rate, 32).filt(x)
        assert np.allclose(dsp.filt_multirate(h, x, rate, 32), want, rtol=1e-9, atol=1e-12)
        sf, so, pos, pieces = dsp.FIRFilter(h, rate, 32), of.FIRArbitraryState(h, rate, 32), 0, []
        for step in (1, 1, 3, 64, 0, 100, 5, 126):
            pieces.append(sf.filt(x[pos:pos + step]))
            ref = so.filt(x[pos:pos + step])
            assert pieces[-1].size == ref.size and sf.input_deficit == so.input_deficit and abs(sf.phi_accumulator - so.acc) < 1e-9
            pos += step
        assert pos == x.size and np.allclose(np.concatenate(pieces), want, rtol=1e-9, atol=1e-12)
        y = dsp.resample(x, rate)
        assert y.size == int(np.ceil(x.size * rate)) and np.allclose(y, of.resample_arb_literal(x, rate), rtol=1e-9, atol=1e-12)


def test_extrapolate_signal_pad_equals_length_minus_one():
    # filtfilt with len(x) == len(b): pad_length == n - 1, the tail slice must not collapse (src/Filters/filt.jl:245-259)
    from dspb200.clients import _extrapolate_signal
    for n in (2, 5, 9):
        sig = np.arange(1.0, n + 1.0) ** 2
        for pad in range(0, n):
            ext = _extrapolate_signal(sig, pad)
            assert ext.shape == (n + 2 * pad,)
            assert np.array_equal(ext[pad:pad + n], sig)
            # odd symmetry about both end points (1-based reference loop restated)
            for i in range(1, pad + 1):
                assert ext[pad - i] == 2 * sig[0] - sig[i]
                assert ext[pad + n - 1 + i] == 2 * sig[n - 1] - sig[n - 1 - i]
    m = np.arange(12.0).reshape(6, 2)
    assert _extrapolate_signal(m, 5).shape == (16, 2)


def test_conv_nd_host_dispatch_with_a_numpy_stand_in_for_the_library(monkeypatch):
    """conv(u, v; algorithm) for matrices / rank-3 arrays: the host resolves the algorithm as conv! does
    (src/dspbase.jl:720-751) and hands the library the larger array first with the reference's per-dimension block
    transforms.  The library call is replaced by the oracle's restatements, which also check the contract of the call."""
    from dspb200 import _lib
    from oracle import dspbase as od
    calls = []

    def fake_conv_nd(u, v, nffts, out, overlapsave=False):
        assert u.flags.f_contiguous and v.flags.f_contiguous and out.flags.f_contiguous and u.ndim == v.ndim <= 3
        assert out.shape == tuple(a + b - 1 for a, b in zip(u.shape, v.shape)) and u.dtype == v.dtype == out.dtype
        if nffts is None:
            calls.append("direct")
            out[...] = od.conv_td_nd(u, v)
        elif overlapsave:
            calls.append("os")
            assert u.size >= v.size                                                     # :746-751
            assert list(nffts) == [od.optimalfftfiltlength(nb, nx) for nb, nx in zip(v.shape, u.shape)]      # :736
            out[...] = od.conv_kern_os_nd(u, v, nffts)
        else:
            calls.append("fft")
            assert list(nffts) == [dsp.nextfastfft(n) for n in out.shape]               # :618
            out[...] = od.conv_kern_fft_nd(u, v)

    monkeypatch.setattr(_lib, "conv_nd", fake_conv_nd)
    rng = np.random.default_rng(3)
    u, v = rng.standard_normal((10, 20)), rng.standard_normal((10, 10))
    ref = od.conv_td_nd(u, v)
    for alg, path in (("direct", "direct"), ("fft_simple", "fft"), ("fft_overlapsave", "os"), (":fft_overlapsave", "os"),
                      ("auto", "direct"), ("fast", "direct")):
        del calls[:]
        assert np.allclose(dsp.conv(u, v, algorithm=alg), ref, atol=1e-12) and calls == [path], alg
        assert np.allclose(dsp.conv(v, u, algorithm=alg), ref, atol=1e-12)                # smaller array first
    # :fft picks overlap-save when some block transform is shorter than the output (:737-743), else the single transform pair
    big, small = rng.standard_normal((300, 280)), rng.standard_normal((5, 7))
    for alg in ("fft", "fast", "auto"):
        del calls[:]
        got = dsp.conv(big, small, algorithm=alg)
        assert calls == ["os"] and np.allclose(got, od.conv_kern_fft_nd(big, small), atol=1e-11)
    del calls[:]
    dsp.conv(u, v, algorithm="fft")                                                       # 19 x 29 outputs, nffts (32, 32): one pair
    assert calls == ["fft"]
    # mixed ranks, integers (exact through Float64), a dimension where size(v) > size(u)
    a3, k2 = np.arange(24).reshape(2, 3, 4), np.ones((2, 2), dtype=np.int64)
    for alg in ("direct", "fft_simple", "fft_overlapsave"):
        got = dsp.conv(a3, k2, algorithm=alg)
        assert got.dtype.kind == "i" and np.array_equal(got, od.conv_td_nd(a3, k2))
    x, y = rng.standard_normal((4, 7, 1)), rng.standard_normal((3, 3, 3))
    assert np.allclose(dsp.conv(x, y, algorithm="fft_overlapsave"), od.conv_td_nd(x, y), atol=1e-13)
    with pytest.raises(dsp.ArgumentError):
        dsp.conv(u, v, algorithm="quantum")
