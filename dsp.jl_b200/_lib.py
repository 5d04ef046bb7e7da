"""ctypes binding of libdspb200.so (declared in include/dspb200.h).

The shared library is the product; this module only marshals pointers.  There is no CPU fallback: if the
library is missing the import fails, and without a CUDA device every exec call raises DSPB200Error.
"""
import ctypes as C
import os

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.environ.get("DSPB200_LIB") or os.path.join(_HERE, "libdspb200.so")   # DSPB200_LIB: another build, e.g. to compare two builds output for output

F32, F64, C32, C64 = 0, 1, 2, 3
_NP2DT = {np.dtype(np.float32): F32, np.dtype(np.float64): F64, np.dtype(np.complex64): C32, np.dtype(np.complex128): C64}
_DT2NP = {v: k for k, v in _NP2DT.items()}

OK, EINVALID, ECUDA, ECUFFT, ENOMEM, EUNSUPPORTED = 0, -1, -2, -3, -4, -5


class DSPB200Error(RuntimeError):
    def __init__(self, code, msg):
        super().__init__(f"dspb200 error {code}: {msg}")
        self.code = code


if not os.path.exists(LIB_PATH):
    raise ImportError(
        f"{LIB_PATH} is missing: build it with `python -c 'import __graft_entry__ as g; g.build()'` "
        "(or `make -C dsp.jl_b200/csrc`).  dspb200 has no CPU fallback.")

lib = C.CDLL(LIB_PATH)

_i64, _int, _vp, _dbl, _sz = C.c_int64, C.c_int, C.c_void_p, C.c_double, C.c_size_t
_pp = C.POINTER(C.c_void_p)

# name -> (restype, argtypes); every name must be declared in include/dspb200.h
SIGNATURES = {
    "dspb200_version": (_int, []),
    "dspb200_last_error": (C.c_char_p, []),
    "dspb200_device_count": (_int, [C.POINTER(_int)]),
    "dspb200_set_device": (_int, [_int]),
    "dspb200_device_info": (_int, [C.POINTER(_int), C.POINTER(_int), C.POINTER(_int), C.POINTER(_sz), C.POINTER(_sz)]),
    "dspb200_malloc": (_int, [_pp, _sz]),
    "dspb200_free": (_int, [_vp]),
    "dspb200_host_alloc": (_int, [_pp, _sz]),
    "dspb200_host_free": (_int, [_vp]),
    "dspb200_memcpy_h2d": (_int, [_vp, _vp, _sz, _vp]),
    "dspb200_memcpy_d2h": (_int, [_vp, _vp, _sz, _vp]),
    "dspb200_stream_sync": (_int, [_vp]),
    "dspb200_launch_count": (_i64, []),
    "dspb200_fir_plan_create": (_int, [_pp, _int, _vp, _i64]),
    "dspb200_fir_exec": (_int, [_vp, _vp, _i64, _i64, _vp]),
    "dspb200_fir_exec_dev": (_int, [_vp, _vp, _i64, _i64, _vp, _vp]),
    "dspb200_fir_plan_destroy": (_int, [_vp]),
    "dspb200_os_plan_create": (_int, [_pp, _int, _vp, _i64, _i64]),
    "dspb200_os_plan_nfft": (_int, [_vp, C.POINTER(_i64), C.POINTER(_int)]),
    "dspb200_os_exec": (_int, [_vp, _vp, _i64, _i64, _vp, _i64]),
    "dspb200_os_exec_dev": (_int, [_vp, _vp, _i64, _i64, _vp, _i64, _vp]),
    "dspb200_os_exec_range_dev": (_int, [_vp, _vp, _i64, _i64, _vp, _i64, _i64, _vp]),
    "dspb200_os_plan_destroy": (_int, [_vp]),
    "dspb200_conv_fft_exec": (_int, [_int, _vp, _i64, _vp, _i64, _i64, _vp]),
    "dspb200_conv_direct_exec": (_int, [_int, _vp, _i64, _vp, _i64, _vp]),
    "dspb200_conv_nd_exec": (_int, [_int, _int, _vp, _vp, _vp, _vp, _vp, _vp]),
    "dspb200_conv_nd_exec_dev": (_int, [_int, _int, _vp, _vp, _vp, _vp, _vp, _vp, _vp]),
    "dspb200_conv_nd_os_exec": (_int, [_int, _int, _vp, _vp, _vp, _vp, _vp, _vp]),
    "dspb200_conv_nd_os_exec_dev": (_int, [_int, _int, _vp, _vp, _vp, _vp, _vp, _vp, _vp]),
    "dspb200_conv_nd_os_set_budget": (_int, [C.c_size_t]),
    "dspb200_hilbert_exec": (_int, [_int, _vp, _i64, _i64, _vp]),
    "dspb200_hilbert_exec_dev": (_int, [_int, _vp, _i64, _i64, _vp, _vp]),
    "dspb200_spec_plan_create": (_int, [_pp, _int, _i64, _i64, _i64, _int, _vp]),
    "dspb200_spec_plan_info": (_int, [_vp, C.POINTER(_i64), C.POINTER(_int)]),
    "dspb200_spec_nsegments": (_i64, [_vp, _i64]),
    "dspb200_welch_exec": (_int, [_vp, _vp, _i64, _dbl, _vp]),
    "dspb200_welch_exec_dev": (_int, [_vp, _vp, _i64, _dbl, _vp, _vp]),
    "dspb200_welch_exec_range_dev": (_int, [_vp, _vp, _i64, _i64, _i64, _i64, _dbl, _vp, _vp]),
    "dspb200_welch_begin_dev": (_int, [_vp, _vp]),
    "dspb200_welch_accumulate_dev": (_int, [_vp, _vp, _i64, _i64, _i64, _i64, _vp]),
    "dspb200_welch_finalize_dev": (_int, [_vp, _dbl, _vp, _vp]),
    "dspb200_filt_welch_exec": (_int, [_vp, _vp, _vp, _i64, _dbl, _vp]),
    "dspb200_os_plan_geometry": (_int, [_vp, C.POINTER(_int), C.POINTER(_i64), C.POINTER(_i64)]),
    "dspb200_spec_plan_geometry": (_int, [_vp, C.POINTER(_int), C.POINTER(_i64), C.POINTER(_i64), C.POINTER(_i64)]),
    "dspb200_stft_exec": (_int, [_vp, _vp, _i64, _i64, _dbl, _int, _vp]),
    "dspb200_stft_exec_dev": (_int, [_vp, _vp, _i64, _i64, _dbl, _int, _vp, _vp]),
    "dspb200_arraysplit_exec": (_int, [_vp, _vp, _i64, _vp]),
    "dspb200_periodogram2_exec": (_int, [_int, _vp, _i64, _i64, _i64, _i64, _dbl, _int, _vp]),
    "dspb200_periodogram2_exec_dev": (_int, [_int, _vp, _i64, _i64, _i64, _i64, _dbl, _int, _vp, _vp]),
    "dspb200_mt_plan_create": (_int, [_pp, _int, _i64, _i64, _i64, _int, _vp, _i64]),
    "dspb200_mt_pgram_exec": (_int, [_vp, _vp, _i64, _vp]),
    "dspb200_mt_spectrogram_exec": (_int, [_vp, _vp, _i64, _vp]),
    "dspb200_mt_pgram_exec_dev": (_int, [_vp, _vp, _i64, _vp, _vp]),
    "dspb200_mt_spectrogram_exec_dev": (_int, [_vp, _vp, _i64, _vp, _vp]),
    "dspb200_mt_cross_spectra_exec": (_int, [_vp, _vp, _i64, _int, _i64, _i64, _int, _vp]),
    "dspb200_mt_cross_spectra_exec_dev": (_int, [_vp, _vp, _i64, _int, _i64, _i64, _int, _vp, _vp]),
    "dspb200_spec_plan_destroy": (_int, [_vp]),
    "dspb200_resample_plan_create": (_int, [_pp, _int, _int, _vp, _i64, _i64, _i64]),
    "dspb200_resample_out_dtype": (_int, [_vp, C.POINTER(_int)]),
    "dspb200_resample_exec": (_int, [_vp, _vp, _i64, _i64, _i64, _i64, _vp, _i64]),
    "dspb200_resample_exec_dev": (_int, [_vp, _vp, _i64, _i64, _i64, _i64, _vp, _i64, _vp]),
    "dspb200_resample_exec_range_dev": (_int, [_vp, _vp, _i64, _i64, _i64, _i64, _vp, _i64, _i64, _vp]),
    "dspb200_resample_arb_plan_create": (_int, [_pp, _int, _int, _vp, _i64, _i64]),
    "dspb200_resample_arb_exec": (_int, [_vp, _vp, _i64, _i64, _dbl, _dbl, _vp, _i64]),
    "dspb200_resample_arb_exec_dev": (_int, [_vp, _vp, _i64, _i64, _dbl, _dbl, _vp, _i64, _vp]),
    "dspb200_resample_plan_destroy": (_int, [_vp]),
}
for _name, (_res, _args) in SIGNATURES.items():
    _f = getattr(lib, _name)
    _f.restype = _res
    _f.argtypes = _args


def last_error():
    return lib.dspb200_last_error().decode("utf-8", "replace")


def check(rc):
    if rc != OK:
        raise DSPB200Error(rc, last_error())


def np_dtype_code(dt):
    dt = np.dtype(dt)
    if dt not in _NP2DT:
        raise TypeError(f"unsupported element type {dt}; expected float32/float64/complex64/complex128")
    return _NP2DT[dt]


def code_np_dtype(code):
    return _DT2NP[code]


def ptr(a):
    """Host pointer of a numpy array (kept alive by the caller)."""
    return a.ctypes.data_as(C.c_void_p)


def launch_count():
    return int(lib.dspb200_launch_count())


def device_count():
    n = _int(0)
    rc = lib.dspb200_device_count(C.byref(n))
    return n.value if rc == OK else 0


class _Plan:
    """Owns an opaque plan handle; destroy on GC (the Julia glue attaches a finalizer the same way)."""
    _destroy = None

    def __init__(self):
        self.handle = C.c_void_p(None)

    def close(self):
        if getattr(self, "handle", None) is not None and self.handle.value:
            getattr(lib, self._destroy)(self.handle)
            self.handle = C.c_void_p(None)

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass


class FirPlan(_Plan):
    _destroy = "dspb200_fir_plan_destroy"

    def __init__(self, b):
        super().__init__()
        b = np.ascontiguousarray(b)
        self.dtype = b.dtype
        check(lib.dspb200_fir_plan_create(C.byref(self.handle), np_dtype_code(b.dtype), ptr(b), b.size))

    def exec(self, x, out):
        nx = x.shape[0]
        ncols = x.size // nx if nx else 0
        check(lib.dspb200_fir_exec(self.handle, ptr(x), nx, ncols, ptr(out)))

    def exec_dev(self, x_ptr, nx, ncols, out_ptr, stream=0):
        check(lib.dspb200_fir_exec_dev(self.handle, x_ptr, nx, ncols, out_ptr, stream))


class OsPlan(_Plan):
    _destroy = "dspb200_os_plan_destroy"

    def __init__(self, v, nfft=0):
        super().__init__()
        v = np.ascontiguousarray(v)
        self.dtype = v.dtype
        self.nv = v.size
        check(lib.dspb200_os_plan_create(C.byref(self.handle), np_dtype_code(v.dtype), ptr(v), v.size, int(nfft)))
        n, f = _i64(0), _int(0)
        check(lib.dspb200_os_plan_nfft(self.handle, C.byref(n), C.byref(f)))
        self.nfft, self.fused = n.value, bool(f.value)

    def exec(self, u, out, nu, ncols, nout):
        check(lib.dspb200_os_exec(self.handle, ptr(u), nu, ncols, ptr(out), nout))

    def exec_ptr(self, u_ptr, nu, ncols, out_ptr, nout):
        check(lib.dspb200_os_exec(self.handle, u_ptr, nu, ncols, out_ptr, nout))

    def exec_dev(self, u_ptr, nu, ncols, out_ptr, nout, stream=0):
        check(lib.dspb200_os_exec_dev(self.handle, u_ptr, nu, ncols, out_ptr, nout, stream))

    def exec_range_dev(self, u_ptr, u_begin, nu_local, out_ptr, out_begin, out_count, stream=0):
        check(lib.dspb200_os_exec_range_dev(self.handle, u_ptr, u_begin, nu_local, out_ptr, out_begin, out_count, stream))


class SpecPlan(_Plan):
    _destroy = "dspb200_spec_plan_destroy"

    def __init__(self, dtype, n, noverlap, nfft, onesided, window=None):
        super().__init__()
        self.dtype = np.dtype(dtype)
        w = None if window is None else np.ascontiguousarray(window, dtype=np.float64)
        check(lib.dspb200_spec_plan_create(C.byref(self.handle), np_dtype_code(dtype), int(n), int(noverlap), int(nfft),
                                           1 if onesided else 0, None if w is None else ptr(w)))
        no, f = _i64(0), _int(0)
        check(lib.dspb200_spec_plan_info(self.handle, C.byref(no), C.byref(f)))
        self.nout, self.fused = no.value, bool(f.value)
        self.n, self.noverlap, self.nfft, self.onesided = int(n), int(noverlap), int(nfft), bool(onesided)

    def nsegments(self, length):
        return int(lib.dspb200_spec_nsegments(self.handle, int(length)))

    def welch(self, s, r, out):
        check(lib.dspb200_welch_exec(self.handle, ptr(s), s.size, float(r), ptr(out)))

    def welch_ptr(self, s_ptr, length, r, out_ptr):
        check(lib.dspb200_welch_exec(self.handle, s_ptr, length, float(r), out_ptr))

    def welch_dev(self, s_ptr, length, r, out_ptr, stream=0):
        check(lib.dspb200_welch_exec_dev(self.handle, s_ptr, length, float(r), out_ptr, stream))

    def welch_begin_dev(self, stream=0):
        check(lib.dspb200_welch_begin_dev(self.handle, stream))

    def welch_accumulate_dev(self, s_ptr, length, sample_offset, seg_begin, seg_end, stream=0):
        check(lib.dspb200_welch_accumulate_dev(self.handle, s_ptr, length, sample_offset, seg_begin, seg_end, stream))

    def welch_finalize_dev(self, r, out_ptr, stream=0):
        check(lib.dspb200_welch_finalize_dev(self.handle, float(r), out_ptr, stream))

    def filt_welch_ptr(self, os_plan, x_ptr, n, r, out_ptr):
        check(lib.dspb200_filt_welch_exec(os_plan.handle, self.handle, x_ptr, int(n), float(r), out_ptr))

    def welch_range_dev(self, s_ptr, length, sample_offset, seg_begin, seg_end, r, out_ptr, stream=0):
        check(lib.dspb200_welch_exec_range_dev(self.handle, s_ptr, length, sample_offset, seg_begin, seg_end, float(r),
                                               out_ptr, stream))

    def arraysplit(self, s, out):
        check(lib.dspb200_arraysplit_exec(self.handle, ptr(s), s.size, ptr(out)))

    def stft(self, s, length, nchan, r, psd_only, out):
        check(lib.dspb200_stft_exec(self.handle, ptr(s), length, nchan, float(r), 1 if psd_only else 0, ptr(out)))

    def stft_dev(self, s_ptr, length, nchan, r, psd_only, out_ptr, stream=0):
        check(lib.dspb200_stft_exec_dev(self.handle, s_ptr, length, nchan, float(r), 1 if psd_only else 0, out_ptr, stream))


class MtPlan(SpecPlan):
    """Multitaper plan: `tapers` is an (ntapers, n) float64 matrix already scaled by 1/sqrt(r_t)."""

    def __init__(self, dtype, n, noverlap, nfft, onesided, tapers):
        _Plan.__init__(self)
        self.dtype = np.dtype(dtype)
        t = np.ascontiguousarray(tapers, dtype=np.float64)
        check(lib.dspb200_mt_plan_create(C.byref(self.handle), np_dtype_code(dtype), int(n), int(noverlap), int(nfft),
                                         1 if onesided else 0, ptr(t), t.shape[0]))
        no, f = _i64(0), _int(0)
        check(lib.dspb200_spec_plan_info(self.handle, C.byref(no), C.byref(f)))
        self.nout, self.fused = no.value, bool(f.value)
        self.n, self.noverlap, self.nfft, self.onesided = int(n), int(noverlap), int(nfft), bool(onesided)

    def mt_pgram(self, s, out):
        check(lib.dspb200_mt_pgram_exec(self.handle, ptr(s), s.size, ptr(out)))

    def mt_spectrogram(self, s, out):
        check(lib.dspb200_mt_spectrogram_exec(self.handle, ptr(s), s.size, ptr(out)))

    def mt_pgram_dev(self, s_ptr, length, out_ptr, stream=0):
        check(lib.dspb200_mt_pgram_exec_dev(self.handle, s_ptr, int(length), out_ptr, stream))

    def mt_spectrogram_dev(self, s_ptr, length, out_ptr, stream=0):
        check(lib.dspb200_mt_spectrogram_exec_dev(self.handle, s_ptr, int(length), out_ptr, stream))

    def cross_spectra_dev(self, signal_ptr, nchan, demean, f_lo, nf, coherence, out_ptr, stream=0):
        check(lib.dspb200_mt_cross_spectra_exec_dev(self.handle, signal_ptr, int(nchan), 1 if demean else 0, int(f_lo), int(nf),
                                                    1 if coherence else 0, out_ptr, stream))

    def cross_spectra(self, signal, nchan, demean, f_lo, nf, coherence, out):
        check(lib.dspb200_mt_cross_spectra_exec(self.handle, ptr(signal), int(nchan), 1 if demean else 0, int(f_lo), int(nf),
                                                1 if coherence else 0, ptr(out)))


class ResamplePlan(_Plan):
    _destroy = "dspb200_resample_plan_destroy"

    def __init__(self, dtype_x, h, interp, decim):
        super().__init__()
        h = np.ascontiguousarray(h)
        if h.dtype not in (np.dtype(np.float32), np.dtype(np.float64)):
            raise TypeError("resample taps must be float32 or float64")
        check(lib.dspb200_resample_plan_create(C.byref(self.handle), np_dtype_code(dtype_x), np_dtype_code(h.dtype), ptr(h),
                                               h.size, int(interp), int(decim)))
        d = _int(0)
        check(lib.dspb200_resample_out_dtype(self.handle, C.byref(d)))
        self.out_dtype = code_np_dtype(d.value)

    def exec(self, x, nx, ncols, n0, phi0, out, nout):
        check(lib.dspb200_resample_exec(self.handle, ptr(x), nx, ncols, n0, phi0, ptr(out), nout))

    def exec_dev(self, x_ptr, nx, ncols, n0, phi0, out_ptr, nout, stream=0):
        check(lib.dspb200_resample_exec_dev(self.handle, x_ptr, nx, ncols, n0, phi0, out_ptr, nout, stream))

    def exec_range_dev(self, x_ptr, x_begin, nx_local, n0, phi0, out_ptr, j_begin, nout_local, stream=0):
        check(lib.dspb200_resample_exec_range_dev(self.handle, x_ptr, x_begin, nx_local, n0, phi0, out_ptr, j_begin,
                                                  nout_local, stream))


class ResampleArbPlan(_Plan):
    """FIRArbitrary plan: pfb and derivative bank of `h` split into `nphases` phases."""
    _destroy = "dspb200_resample_plan_destroy"

    def __init__(self, dtype_x, h, nphases):
        super().__init__()
        h = np.ascontiguousarray(h)
        if h.dtype not in (np.dtype(np.float32), np.dtype(np.float64)):
            raise TypeError("resample taps must be float32 or float64")
        check(lib.dspb200_resample_arb_plan_create(C.byref(self.handle), np_dtype_code(dtype_x), np_dtype_code(h.dtype), ptr(h),
                                                   h.size, int(nphases)))
        d = _int(0)
        check(lib.dspb200_resample_out_dtype(self.handle, C.byref(d)))
        self.out_dtype = code_np_dtype(d.value)

    def exec(self, x, nx, n0, acc0, delta, out, nout):
        check(lib.dspb200_resample_arb_exec(self.handle, ptr(x), nx, n0, float(acc0), float(delta), ptr(out), nout))

    def exec_dev(self, x_ptr, nx, n0, acc0, delta, out_ptr, nout, stream=0):
        check(lib.dspb200_resample_arb_exec_dev(self.handle, x_ptr, nx, n0, float(acc0), float(delta), out_ptr, nout, stream))


def conv_fft(u, v, nfft, out):
    check(lib.dspb200_conv_fft_exec(np_dtype_code(u.dtype), ptr(u), u.size, ptr(v), v.size, int(nfft), ptr(out)))


def conv_direct(u, v, out):
    check(lib.dspb200_conv_direct_exec(np_dtype_code(u.dtype), ptr(u), u.size, ptr(v), v.size, ptr(out)))


def conv_nd(u, v, nffts, out, overlapsave=False):
    """u, v, out: Fortran-ordered arrays of equal rank (<= 3) and dtype; nffts: per-dimension FFT sizes (one transform pair
    of that size, or -- overlapsave -- the block transform of the N-D overlap-save blocking) or None (direct)."""
    us = np.asarray(u.shape, dtype=np.int64)
    vs = np.asarray(v.shape, dtype=np.int64)
    nf = None if nffts is None else np.asarray(nffts, dtype=np.int64)
    fn = lib.dspb200_conv_nd_os_exec if overlapsave else lib.dspb200_conv_nd_exec
    check(fn(np_dtype_code(u.dtype), u.ndim, ptr(us), ptr(u), ptr(vs), ptr(v), None if nf is None else ptr(nf), ptr(out)))


def conv_nd_dev(dtype, ushape, u_ptr, vshape, v_ptr, nffts, out_ptr, overlapsave=False, stream=0):
    """Device-pointer form of conv_nd (column-major buffers); returns after the work has completed."""
    us = np.asarray(ushape, dtype=np.int64)
    vs = np.asarray(vshape, dtype=np.int64)
    nf = None if nffts is None else np.asarray(nffts, dtype=np.int64)
    fn = lib.dspb200_conv_nd_os_exec_dev if overlapsave else lib.dspb200_conv_nd_exec_dev
    check(fn(np_dtype_code(np.dtype(dtype)), len(ushape), ptr(us), u_ptr, ptr(vs), v_ptr, None if nf is None else ptr(nf),
             out_ptr, stream))


def conv_nd_os_set_budget(nbytes):
    """Bytes of block buffers one batch of the N-D overlap-save path may use (default 1 GiB)."""
    check(lib.dspb200_conv_nd_os_set_budget(int(nbytes)))


def periodogram2(s, nfft, r, ptype, out):
    """s: Fortran-ordered real matrix; out: Fortran-ordered nfft matrix (ptype 0) or the radial vector."""
    check(lib.dspb200_periodogram2_exec(np_dtype_code(s.dtype), ptr(s), s.shape[0], s.shape[1], int(nfft[0]), int(nfft[1]),
                                        float(r), int(ptype), ptr(out)))


def periodogram2_dev(dtype, s_ptr, shape, nfft, r, ptype, out_ptr, stream=0):
    check(lib.dspb200_periodogram2_exec_dev(np_dtype_code(np.dtype(dtype)), s_ptr, int(shape[0]), int(shape[1]), int(nfft[0]),
                                            int(nfft[1]), float(r), int(ptype), out_ptr, stream))


def hilbert(x, n, ncols, out):
    check(lib.dspb200_hilbert_exec(np_dtype_code(x.dtype), ptr(x), n, ncols, ptr(out)))


def hilbert_dev(dtype, x_ptr, n, ncols, out_ptr, stream=0):
    check(lib.dspb200_hilbert_exec_dev(np_dtype_code(np.dtype(dtype)), x_ptr, n, ncols, out_ptr, stream))
